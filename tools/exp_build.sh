#!/bin/bash
# Tuning aid: builds tools/exp/libsrwn_trace.so with fused.cu compiled under -DSRWN_TUNING: the clock64 trace of one
# chunk (tools/trace_fused.py), srwn_debug_read_trace and k_mma_bench (tools/mma_bench.py).  The trace code costs about
# 10 % of the fused kernel's time.  Use with SRWN_LIB=tools/exp/libsrwn_trace.so.
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/exp
C=sr-wavenet_b200/csrc
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -DSRWN_TUNING -c $C/fused.cu -o tools/exp/fused_trace.o
objs=""
for f in api stack_f32 mol ops_generic ar_generate ar_mma train_f32 train_tc stft_loss encoder random; do objs="$objs $C/$f.o"; done
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o tools/exp/libsrwn_trace.so $objs tools/exp/fused_trace.o -lcudart_static -ldl -lrt -lpthread
