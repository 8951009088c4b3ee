#!/bin/bash
# Build libbayescard_b200.so in-tree for sm_100a (the .so is git-ignored but travels with gpurun).
set -euo pipefail
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=../libbayescard_b200.so
SRCS="bc_api.cu bc_convert.cu k1_generic.cu k2_batched.cu k2_umma.cu k3_fused.cu spec_jit.cu spec_codegen.cc bc_marginal.cu bc_sqlc.cc bc_joblight.cc bc_fit.cu bc_structure.cu bc_modelfile.cc"
$NVCC -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xptxas -v ${BC_EXTRA_NVCC:-} \
      -Xcompiler -fPIC,-O2,-Wall,-fvisibility=hidden -shared -cudart static \
      -x cu $SRCS -o $OUT -ldl -lpthread 2> build.log || { cat build.log; exit 1; }
grep -E "error|warning: v|Used [0-9]+ registers|spill" build.log | grep -v "0 bytes spill" | head -40 || true
echo "built $OUT"
