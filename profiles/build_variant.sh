#!/bin/bash
# builds an experiment variant of the library: profiles/build_variant.sh NAME -DFLAG ...   ->  build/exp/lib_NAME.so
set -e
name=$1; shift
mkdir -p build/exp
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --fmad=false -Xcompiler -fPIC -shared "$@" \
  -o build/exp/lib_$name.so betazero_b200/csrc/{env,mcts,selfplay,mlp_pair,mlp_pair2,minimax}.cu
echo build/exp/lib_$name.so
