#!/bin/bash
# Build the WORKING-TREE physics TU with extra nvcc flags into ppo-bipedalwalker_b200/lib/libwalker_b200_<tag>.so, linking the
# other objects of the current build (same-box A/B timing: WB_LIB_PATH=... python scripts/sweep_physics.py ...).
# usage: scripts/build_variant.sh <tag> [nvcc flags, e.g. -DWB_PHASE_PROFILE]
set -e
cd "$(dirname "$0")/.."
tag=$1; shift
unset CC CXX
L=ppo-bipedalwalker_b200/lib
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -ffp-contract=off -ftz=false -prec-div=true -prec-sqrt=true -fmad=false"
nvcc $FLAGS "$@" -c ppo-bipedalwalker_b200/csrc/physics_lanes.cu -o $L/physics_lanes_$tag.o
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $L/libwalker_b200_$tag.so $L/physics_lanes_$tag.o $L/api_env.o $L/physics_scene.o $L/api_scene.o \
  $L/mlp.o $L/mlp_tc.o $L/mlp_generic.o $L/api_policy.o $L/api_population.o -lcudart_static -lpthread -ldl -lrt
echo built $L/libwalker_b200_$tag.so
