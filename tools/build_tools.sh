#!/bin/bash
# Builds the debug / micro-benchmark binaries under tools/bin (sm_100a only; they travel to the GPU box with gpurun).
# VARIANTS="name:flags ..." overrides the sor_bench variants.
set -e
cd "$(dirname "$0")"
NV="nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -I../include -I../slowflow_b200/csrc"
mkdir -p bin
: ${VARIANTS:="r8bar:-DSF_SOR_R=8|-DSF_SOR_NW=8|-DSF_SOR_SYNC=0 r4bar:-DSF_SOR_R=4|-DSF_SOR_NW=16|-DSF_SOR_SYNC=0 r8flag:-DSF_SOR_R=8|-DSF_SOR_NW=8|-DSF_SOR_SYNC=1 r4flag:-DSF_SOR_R=4|-DSF_SOR_NW=16|-DSF_SOR_SYNC=1"}
for v in $VARIANTS; do
  name=${v%%:*}; flags=$(echo "${v#*:}" | tr '|' ' ')
  $NV $flags -DSF_SOR_CLOCKS -o bin/sor_bench_$name sor_bench.cu -lcuda &
  $NV $flags -o bin/sor_plain_$name sor_bench.cu -lcuda &
done
wait
[ -n "$SOR_ONLY" ] && exit 0
$NV -o bin/ffma_bench ffma_bench.cu
$NV -o bin/prep_bench prep_bench.cu
$NV -o bin/tma_bw tma_bw.cu -lcuda
