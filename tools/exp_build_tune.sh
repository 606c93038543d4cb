#!/bin/bash
# Tuning aid: tools/exp/libsrwn_tune.so = libsrwn.so with train_tc.cu compiled under -DSRWN_TUNING (phase clock stamps).
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/exp
C=sr-wavenet_b200/csrc
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -DSRWN_TUNING $* -c $C/train_tc.cu -o tools/exp/train_tc_tune.o
objs=""
for f in api stack_f32 mol ops_generic ar_generate ar_mma train_f32 stft_loss fused encoder random; do objs="$objs $C/$f.o"; done
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o tools/exp/libsrwn_tune.so $objs tools/exp/train_tc_tune.o -lcudart_static -ldl -lrt -lpthread
