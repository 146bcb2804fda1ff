#!/bin/bash
# Build a variant of the library next to the default one for A/B timing (scripts/dev_variant_bench.sh picks it up through
# BOCF_LIB_PATH):   scripts/dev_build_variant.sh rr128 posterior.cu -maxrregcount=128   ->  bocf_b200/csrc/libbocf_rr128.so
# The other objects are the default build's (run `python __graft_entry__.py` first).  Variant .so files are git-ignored.
set -e
name=$1; src=$2; shift 2
cd "$(dirname "$0")/../bocf_b200/csrc"
obj=/tmp/bocf_variant_${name}.o
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC --expt-relaxed-constexpr "$@" -c "$src" -o "$obj"
objs=""
for f in acq api chol kg lml posterior split_gemm; do
  if [ "$f.cu" == "$src" ]; then objs="$objs $obj"; else objs="$objs $f.o"; fi
done
nvcc -shared -o libbocf_${name}.so $objs -gencode arch=compute_100a,code=sm_100a -cudart static
echo "built bocf_b200/csrc/libbocf_${name}.so ($*)"
