#!/bin/bash
# Round-2 candidate builds of the mapper kernel (second structure, unc_k2v2.cuh) for tools/gpu_variants.py:
# CTA shapes (CTAs per SM x warps per CTA).
set -e
cd "$(dirname "$0")/../uncalled_b200"
F="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -fmad=false -std=c++17 -Xcompiler -fPIC --shared -diag-suppress 550"
rm -rf variants variants_pt; mkdir -p variants variants_pt
SRC="csrc/unc_abi.cu csrc/unc_index_build.cpp csrc/unc_fast5.cpp -lz"
build() { nvcc $F "${@:2}" -o "variants/$1.so" $SRC; }
build v2_w12c2 -DK2_WARPS=12 -DK2_MIN_CTAS=2 &
build v2_w14c2 -DK2_WARPS=14 -DK2_MIN_CTAS=2 &
build v2_w16c2 -DK2_WARPS=16 -DK2_MIN_CTAS=2 &
wait
nvcc $F -DUNC_PHASE_TIMING -DK2_WARPS=14 -DK2_MIN_CTAS=2 -o variants_pt/v2_w14c2.so $SRC
ls -la variants variants_pt
