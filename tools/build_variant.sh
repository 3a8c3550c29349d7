#!/bin/bash
# tools/build_variant.sh NAME "-DFLAG ..." [SOURCES] : recompile SOURCES (default score_pair.cu; several as one quoted,
# space-separated list) with extra flags, link with the stock objects into hgrnet_b200/lib/var_NAME.so (select it with
# HGR_LIB=...).  Kernel experiments and diagnostics builds only, e.g. the placement log of tools/placement.py:
#   tools/build_variant.sh placement -DHGR_PLACEMENT "score_pair.cu aggregate_norm.cu topk_merge.cu"
set -e
name=$1; flags=$2; srcs=${3:-score_pair.cu}
L=hgrnet_b200/lib
objs=$(ls $L/*.o | grep -v "/var_")
var_objs=""
for src in $srcs; do
  stem=${src%.cu}
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr $flags -I include -c hgrnet_b200/csrc/$src -o $L/var_${name}_$stem.o
  objs=$(echo "$objs" | grep -v "/$stem.o$")
  var_objs="$var_objs $L/var_${name}_$stem.o"
done
nvcc -gencode arch=compute_100a,code=sm_100a -shared -cudart static -o $L/var_$name.so $objs $var_objs
rm $var_objs
echo built $L/var_$name.so
