#!/bin/bash
# Build the physics TU of another commit into ppo-bipedalwalker_b200/lib/libwalker_b200_<tag>.so (for same-box A/B timing:
# WB_LIB_PATH=... python scripts/sweep_physics.py ...).  usage: scripts/build_ab.sh <commit> <tag>
set -e
cd "$(dirname "$0")/.."
commit=$1; tag=$2
tmp=$(mktemp -d)
git archive "$commit" ppo-bipedalwalker_b200/csrc include | tar -x -C "$tmp"
unset CC CXX
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -ffp-contract=off -ftz=false -prec-div=true -prec-sqrt=true"
objs=""
for f in physics_lanes api_env physics_scene api_scene; do nvcc $FLAGS -fmad=false -c $tmp/ppo-bipedalwalker_b200/csrc/$f.cu -o $tmp/$f.o & done
for f in mlp mlp_tc mlp_generic api_policy api_population; do nvcc $FLAGS -c $tmp/ppo-bipedalwalker_b200/csrc/$f.cu -o $tmp/$f.o & done
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ppo-bipedalwalker_b200/lib/libwalker_b200_$tag.so $tmp/*.o -lcudart_static -lpthread -ldl -lrt
rm -rf "$tmp"
echo built ppo-bipedalwalker_b200/lib/libwalker_b200_$tag.so
