#!/bin/bash
# quick iteration: GPU tests, bench c2 + c4 without the CPU baseline leg
mkdir -p gpurun_out
TAG=${1:-q}
timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -6
for wl in c2 c4; do
  timeout 600 python bench.py --workload $wl --steps 10 --warmup 3 --no-cpu-baseline > gpurun_out/bench_${wl}_${TAG}.json 2> gpurun_out/bench_${wl}_${TAG}.err
  tail -c 300 gpurun_out/bench_${wl}_${TAG}.err
  python - <<PY
import json
d=json.loads(open("gpurun_out/bench_${wl}_${TAG}.json").read().strip().splitlines()[-1])
print("${wl}", round(d["value"],1), "struct/s", round(d["ms_per_step"],3), "ms | e2e", round(d["e2e"]["value"],1), round(d["e2e"]["ms_per_step"],2), "ms", d["e2e"].get("breakdown"), "| roofline", d["roofline"]["frac"], d["roofline"]["us_per_launch"])
for k,v in list(d["kernel_shares"].items())[:9]: print("   ",k,v)
PY
done
