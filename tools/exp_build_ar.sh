#!/bin/bash
# Tuning aid: builds tools/exp/libsrwn_<name>.so with ar_mma.cu compiled with extra flags (e.g. -DSRWN_AR_TIMING).
# Usage: tools/exp_build_ar.sh <name> [nvcc flags...];  run with SRWN_LIB=tools/exp/libsrwn_<name>.so
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/exp
C=sr-wavenet_b200/csrc
name=$1; shift
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC "$@" -c $C/ar_mma.cu -o tools/exp/ar_$name.o
objs=""
for f in api stack_f32 mol ops_generic ar_generate train_f32 train_tc random stft_loss fused encoder; do objs="$objs $C/$f.o"; done
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o tools/exp/libsrwn_$name.so $objs tools/exp/ar_$name.o -lcudart_static -ldl -lrt -lpthread
