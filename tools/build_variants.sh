#!/bin/bash
# Build A/B variants of compile-time knobs next to the default library: tools/build_variants.sh name "-DFLAG=.." ...
# -> headtrackr_b200/variants/libht_<name>.so (select with HT_LIB=<path>); git-ignored, travels to the GPU box.
set -e
cd "$(dirname "$0")/../headtrackr_b200/csrc"
mkdir -p ../variants
while [ $# -ge 2 ]; do
  name=$1; flags=$2; shift 2
  /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a $flags -O3 -std=c++17 -lineinfo -fmad=false \
    -Xcompiler -fPIC,-O2,-Wall -Xptxas -v -shared -o ../variants/libht_$name.so ht_api.cu 2> ../variants/build_$name.log
  grep -E "k_trackILi2EEE|k_cascadeILb1" -A3 ../variants/build_$name.log | grep -E "Used|spill" | head -4
  echo "built $name"
done
