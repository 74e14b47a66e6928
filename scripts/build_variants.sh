#!/bin/bash
# Build tuning variants of libmbcol.so into csrc/variants/ for A/B timing on the GPU box.
# usage: scripts/build_variants.sh name "-DFLAG=..." [name "-D..."]...
set -e
cd "$(dirname "$0")/../minibase-columnar-database_b200/csrc"
mkdir -p variants
while [ $# -ge 2 ]; do
  name=$1; flags=$2; shift 2
  d=variants/$name; mkdir -p $d
  for f in mbc_api mbc_scan mbc_synth mbc_bitmap mbc_join mbc_ingest mbc_sort mbc_shard mbc_group mbc_topk; do
    /usr/local/cuda/bin/nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC --expt-relaxed-constexpr $flags -c $f.cu -o $d/$f.o &
  done
  wait
  /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o variants/libmbcol_$name.so $d/*.o -lcudart
done
ls variants/*.so
