#!/bin/bash
# GPU call: sanitizer probe of the graph loop, tail-regime timings, per-step timings of the C3 sweep
mkdir -p gpurun_out
for m in g hg gg; do
  echo "== memcheck $m"; timeout 300 compute-sanitizer --tool memcheck --print-limit 3 python scripts/sanitize_r2d.py $m 2>&1 | grep -v "^=========     Host Frame" | tail -25
done
echo "== tail3 host loop (profile)"; python scripts/gpu_tail3.py
echo "== C3 per-step"; DFTATOM_DEBUG_STEPS=1 python scripts/gpu_steps_c3.py 2> gpurun_out/steps_c3.txt; tail -3 gpurun_out/steps_c3.txt
