#!/bin/bash
mkdir -p gpurun_out
export DFT_OPTS="use_graph=0"
for k in search_rows match_cta poisson_warm potential_energy density_update; do
  timeout 300 ncu --set full --clock-control none --import-source on -k regex:$k -s 12 -c 1 -f -o gpurun_out/prof_r2_$k python scripts/prof_c3.py > gpurun_out/prof_r2_$k.log 2>&1
  tail -2 gpurun_out/prof_r2_$k.log
done
