#!/bin/bash
# A/B of environment toggles inside ONE gpurun call (same box, same clocks): each configuration runs the 1-GPU device-timed bench
# twice, interleaved, so box-to-box variance (+-3 %) does not hide a 1-2 % effect.
#   bash scripts/ab_bench.sh "MLXB200_OVERLAP_SHARED=1" "MLXB200_OVERLAP_SHARED=0" ...
mkdir -p gpurun_out
for rep in 1 2; do
  for cfg in "$@"; do
    line=$(env $cfg timeout 300 python bench.py --no-baseline --no-e2e --steps 40 --warmup 5 2>&1 | grep "rank 0\] decode")
    echo "[$rep] $cfg :: $line" | tee -a gpurun_out/ab_bench.txt
  done
done
