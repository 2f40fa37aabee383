#!/bin/bash
# Builds kernel variants of libsnag_b200.so for A/B power/throughput measurements (load one with SNAG_B200_LIB=snag_b200/_variants/lib_<name>.so).
set -e
cd "$(dirname "$0")/.."
mkdir -p snag_b200/_variants
build() {  # name, extra flags
  name=$1; shift
  objs=""
  for f in abi bw_kernels sim_kernels icl_fused icl_fwd_sym l1_sweep; do
    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC --expt-relaxed-constexpr "$@" \
      -c snag_b200/csrc/$f.cu -o snag_b200/_variants/${name}_$f.o &
    objs="$objs snag_b200/_variants/${name}_$f.o"
  done
  wait
  nvcc -shared -o snag_b200/_variants/lib_$name.so $objs -gencode arch=compute_100a,code=sm_100a
  rm -f $objs
}
if [ $# -eq 0 ]; then
  build base
  build wg4 -DSNAG_EPI_WG=4
else
  # usage: build_variants.sh name1 "flags1" name2 "flags2" ...
  while [ $# -gt 0 ]; do build $1 $2; shift 2; done
fi
ls -la snag_b200/_variants/
