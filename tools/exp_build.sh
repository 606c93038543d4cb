#!/bin/bash
# Tuning aid: builds tools/exp/libsrwn_<name>.so, libsrwn.so with one source compiled with extra nvcc flags, e.g.
#   tools/exp_build.sh fused.cu trace -DSRWN_TUNING       the fused kernel's clock64 trace (tools/trace_fused.py)
#   tools/exp_build.sh train_tc.cu tune -DSRWN_TUNING     phase clock stamps of the training kernels (tools/tc_trace.py)
#   tools/exp_build.sh ar_mma.cu timing -DSRWN_AR_TIMING  per-layer clocks of the tensor-core generation kernel
# The other objects of __graft_entry__.SOURCES are linked as the build left them (python __graft_entry__.py first).
# Run with SRWN_LIB=tools/exp/libsrwn_<name>.so.
set -e
cd "$(dirname "$0")/.."
[ $# -ge 2 ] || { echo "usage: tools/exp_build.sh <source.cu> <name> [nvcc flags...]" >&2; exit 2; }
src=$1; name=$2; shift 2
C=sr-wavenet_b200/csrc
read -r -a sources <<< "$(python3 -c 'import __graft_entry__ as g; print(" ".join(g.SOURCES))')"
read -r -a flags <<< "$(python3 -c 'import __graft_entry__ as g; print(" ".join(f for f in g.NVCC_FLAGS if not f.startswith("--use_fast_math")))')"
[[ " ${sources[*]} " == *" $src "* ]] || { echo "$src is not in __graft_entry__.SOURCES" >&2; exit 2; }
mkdir -p tools/exp
objs=()
for f in "${sources[@]}"; do
  if [ "$f" = "$src" ]; then
    objs+=("tools/exp/${f%.cu}_$name.o")
    nvcc "${flags[@]}" "$@" -c "$C/$f" -o "${objs[-1]}"
  else
    [ -f "$C/${f%.cu}.o" ] || { echo "missing $C/${f%.cu}.o: run python __graft_entry__.py first" >&2; exit 2; }
    objs+=("$C/${f%.cu}.o")
  fi
done
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o "tools/exp/libsrwn_$name.so" "${objs[@]}" -lcudart_static -ldl -lrt -lpthread
