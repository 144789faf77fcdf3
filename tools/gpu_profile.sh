#!/bin/bash
# Runs on the GPU box (via gpurun): GPU tests, benches, ncu launch lists, full captures of the top kernels.
set -u
mkdir -p gpurun_out
TAG=${1:-r02}
timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -4 | tee gpurun_out/pytest_gpu_${TAG}.log
for wl in c2 c4 c3; do
  timeout 900 python bench.py --workload $wl --steps 10 --warmup 3 > gpurun_out/bench_${wl}_${TAG}.json 2> gpurun_out/bench_${wl}_${TAG}.err
  tail -c 300 gpurun_out/bench_${wl}_${TAG}.err
done
timeout 600 python bench.py --impl reference --steps 2 --warmup 1 > gpurun_out/bench_ref_c2_${TAG}.json 2>> gpurun_out/bench_ref.err
# launch lists (cold-cache, serialised: compare shares)
for wl in c2 c4; do
  timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv \
    --log-file gpurun_out/launches_${wl}_${TAG}.csv python bench.py --workload $wl --steps 1 --warmup 1 --no-cpu-baseline \
    > gpurun_out/ncu_launch_${wl}.log 2>&1
done
# full captures (one short command each)
timeout 600 ncu --set full --clock-control none --import-source on -k regex:segment_sum -s 3 -c 2 \
  -o gpurun_out/prof_scatter_${TAG} -f python bench.py --workload c4 --scatter-only > gpurun_out/ncu_scatter.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:segment_sum -s 3 -c 2 \
  -o gpurun_out/prof_scatter_c2_${TAG} -f python bench.py --workload c2 --scatter-only > gpurun_out/ncu_scatter_c2.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:gated_ -s 14 -c 6 \
  -o gpurun_out/prof_gated_${TAG} -f python bench.py --workload c4 --steps 1 --warmup 1 --no-cpu-baseline > gpurun_out/ncu_gated.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:linear_tc -s 30 -c 4 \
  -o gpurun_out/prof_linear_${TAG} -f python bench.py --workload c4 --steps 1 --warmup 1 --no-cpu-baseline > gpurun_out/ncu_linear.log 2>&1
ls -la gpurun_out | tail -30
