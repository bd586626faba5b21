#!/bin/bash
# Round-2 GPU pass: bench line, ncu launch list of the bench command, full ncu captures of the hot kernels
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/smi.txt; nproc >> gpurun_out/smi.txt
timeout 1200 python bench.py > gpurun_out/bench_r2c.json 2> gpurun_out/bench_r2c.err; tail -c 1500 gpurun_out/bench_r2c.json; tail -3 gpurun_out/bench_r2c.err
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 6000 --csv --log-file gpurun_out/launches_r2.csv python bench.py --steps 1 --warmup 0 --no-rn --no-batch --no-micro --no-cpu-baseline --no-parity > gpurun_out/launches_r2.log 2>&1
for k in search_rows match_cta poisson_warm potential_energy density_update; do
  timeout 300 ncu --set full --clock-control none --import-source on -k regex:$k -s 12 -c 1 -f -o gpurun_out/prof_r2_$k DFT_OPTS="use_graph=0" python scripts/prof_c3.py > gpurun_out/prof_r2_$k.log 2>&1
done
ls -la gpurun_out | tail -12
