#!/bin/bash
# Builds <out> (default profiles/_build/librcn_cuda_phases.so): the product objects of the tree at <src> (default: this one,
# built first with build()) with smallnet.cu recompiled under -DRCN_SN_PHASES (kernel A stamps clock64() at its phase
# boundaries).  Profiling aid only; select it with RCN_CUDA_LIB=<path>.
# (The launch timeline is part of the product library now: rcn_cuda_timeline_enable / _read.)
#   profiles/build_phases.sh [src tree] [out .so]
set -e
cd "$(dirname "$0")/.."
SRC=$(cd "${1:-.}" && pwd)
OUT=${2:-profiles/_build/librcn_cuda_phases.so}
C=$SRC/mercer_research_b200/csrc
mkdir -p "$(dirname "$OUT")"
OBJ="${OUT%.so}_smallnet.o"
nvcc -O3 -std=c++17 -lineinfo --expt-relaxed-constexpr -Xcompiler -fPIC -gencode arch=compute_100a,code=sm_100a \
     -DRCN_SN_PHASES -c $C/smallnet.cu -o "$OBJ"
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT" \
     $C/model.o $C/features.o $C/dense.o "$OBJ" $C/conv.o $C/extops.o $C/dp.o $C/ozaki.o $C/cnn.o $C/optim.o -lcudart
