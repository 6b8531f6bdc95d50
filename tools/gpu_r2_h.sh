#!/bin/bash
# round 2, GPU call H (1 GPU): counting CTA size experiment (GATB_COUNT_THREADS)
mkdir -p gpurun_out
cd "$(dirname "$0")/.."
run() {
  name=$1; shift
  env "$@" timeout 600 python bench.py --steps 6 --warmup 2 --no-cpu-baseline --no-e2e > gpurun_out/h_bench_$name.json 2> gpurun_out/h_bench_$name.err
  python - <<PY
import json
try:
    d=json.load(open("gpurun_out/h_bench_$name.json")); r=d["roofline"]
    print("$name: value %.0f ms/step %.2f count %.3f place %.3f parity %s" % (d["value"], d["ms_per_step"], r["kernel_ms"], r["other_kernels"]["place_kernel_ms"], d["parity_check"]))
except Exception as e:
    print("$name failed", e); print(open("gpurun_out/h_bench_$name.err").read()[-800:])
PY
}
run base GATB_X=0
run threads512 GATB_COUNT_THREADS=512
