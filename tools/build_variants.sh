#!/usr/bin/env bash
# Builds libbbq_b200.so as of an earlier commit for same-box A/B runs (tools/ab_libs.sh): REF=<commit> tools/build_variants.sh
# Output: build/variants/ref_<commit>.so (build/ is ignored by git).
set -e
cd "$(dirname "$0")/.."
: "${REF:?set REF=<commit> to build the library as of that commit}"
mkdir -p build/variants
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo --fmad=false -std=c++17 -Xcompiler -fPIC -shared"
src=$(mktemp -d)
trap 'rm -rf "$src"' EXIT
git archive "$REF" better-binary-quantization_b200/csrc include | tar -x -C "$src"
$NVCC $FLAGS -o build/variants/ref_${REF:0:7}.so "$src"/better-binary-quantization_b200/csrc/bbq_api.cu
ls -la build/variants/
