#!/bin/bash
# A/B of k_scan's switches on the bench workload (device-resident stream, kernels only).  usage: tools/ab_scan.sh <tag>
tag=${1:-ab}
mkdir -p gpurun_out
run() { # name, env...
    name=$1; shift
    env "$@" python bench.py --no-e2e --no-cpu-baseline --steps 20 --warmup 3 $EXTRA > gpurun_out/${tag}_${name}.json 2> gpurun_out/${tag}_${name}.log
    python - "$name" gpurun_out/${tag}_${name}.json <<'PY'
import json, sys
try:
    d = json.loads(open(sys.argv[2]).read().strip().splitlines()[-1])
    r = d["roofline"]
    print("%-14s ms/step %.3f  k_scan %.3f ms  frac %.3f  launches %d  counters %s" % (sys.argv[1], d["ms_per_step"], r["kernel_ms_per_step"], r["frac"], d["gpu_launches"], d["counters"]))
except Exception as e:
    print(sys.argv[1], "FAILED", e)
PY
}
run all ITX_SCAN_FLAGS=15
run none ITX_SCAN_FLAGS=0
run prefetch ITX_SCAN_FLAGS=1
run domsize ITX_SCAN_FLAGS=2
run window ITX_SCAN_FLAGS=4
run window_ahead ITX_SCAN_FLAGS=12
EXTRA="--mode 2 --reads 25000000" run all_pe ITX_SCAN_FLAGS=15
