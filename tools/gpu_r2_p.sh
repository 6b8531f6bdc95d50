#!/bin/bash
# round 2, GPU call P (1 GPU): compute-sanitizer on the TMA-streamed statistics and the placement kernels
mkdir -p gpurun_out
cd "$(dirname "$0")/.."
for tool in memcheck racecheck synccheck; do
  timeout 600 compute-sanitizer --tool $tool --log-file gpurun_out/p_$tool.log python tools/sanitizer_stats.py > gpurun_out/p_$tool.out 2>&1
  echo "$tool: $(tail -1 gpurun_out/p_$tool.out) | $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY|hazard' gpurun_out/p_$tool.log | tail -2 | tr '\n' ' ')"
done
