#!/bin/bash
# Build the physics TU of another commit into ppo-bipedalwalker_b200/lib/libwalker_b200_<tag>.so (for same-box A/B timing:
# WB_LIB_PATH=... python scripts/sweep_physics.py ...).  usage: scripts/build_ab.sh <commit> <tag> [nvcc flags]
# The flags go to the four physics sources, e.g. a -DWB_... build switch that commit still has.
set -e
cd "$(dirname "$0")/.."
commit=$1; tag=$2; shift 2
tmp=$(mktemp -d)
git archive "$commit" ppo-bipedalwalker_b200/csrc include | tar -x -C "$tmp"
unset CC CXX
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -ffp-contract=off -ftz=false -prec-div=true -prec-sqrt=true"
pids=""
for f in physics_lanes api_env physics_scene api_scene; do nvcc $FLAGS -fmad=false "$@" -c $tmp/ppo-bipedalwalker_b200/csrc/$f.cu -o $tmp/$f.o & pids="$pids $!"; done
for f in mlp mlp_tc mlp_generic api_policy api_population; do nvcc $FLAGS -c $tmp/ppo-bipedalwalker_b200/csrc/$f.cu -o $tmp/$f.o & pids="$pids $!"; done
fail=0
for p in $pids; do wait $p || fail=1; done
if [ $fail != 0 ]; then rm -rf "$tmp"; echo "build_ab.sh: a compile failed, nothing linked" >&2; exit 1; fi
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ppo-bipedalwalker_b200/lib/libwalker_b200_$tag.so $tmp/*.o -lcudart_static -lpthread -ldl -lrt
rm -rf "$tmp"
echo built ppo-bipedalwalker_b200/lib/libwalker_b200_$tag.so
