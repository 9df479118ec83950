#!/bin/bash
# One GPU session of round 2: parity tests (incl. the at-size pins), smoke, bench lines of all three workloads, CPU arm,
# ncu launch list + full capture of the per-sample kernel.   usage: tools/gpu_r02.sh <tag> [skip-tests] [skip-ncu]
TAG=${1:-r02}
mkdir -p gpurun_out
set -x
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv
make -C oracle port >/dev/null
if [ "$2" != "skip-tests" ]; then
  timeout 1800 python -m pytest tests -m gpu -x -q 2>&1 | tail -15 | tee gpurun_out/pytest_${TAG}.txt
  timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3
fi
python -c "import lpcnet_b200, json; print(json.dumps(lpcnet_b200.measure_smem_peak(0)))" | tee gpurun_out/smem_peak_${TAG}.json
timeout 600 python bench.py --gpus 1 --steps 10 --warmup 3 > gpurun_out/bench_${TAG}.json 2> gpurun_out/bench_${TAG}.err; tail -c 4500 gpurun_out/bench_${TAG}.json; tail -5 gpurun_out/bench_${TAG}.err
timeout 600 python bench.py --impl reference --gpus 1 --steps 3 --warmup 1 > gpurun_out/bench_ref_${TAG}.json 2>/dev/null; tail -c 1500 gpurun_out/bench_ref_${TAG}.json
for W in config2_float config5_decode; do
  timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --frames 100 --workload $W > gpurun_out/bench_${W}_${TAG}.json 2>gpurun_out/bench_${W}_${TAG}.err
  tail -3 gpurun_out/bench_${W}_${TAG}.err
  python - <<PY
import json
d=json.loads(open("gpurun_out/bench_${W}_${TAG}.json").read().strip().splitlines()[-1])
print("$W", {k:d[k] for k in ("value","ms_per_step")}, "e2e", d["e2e"]["value"], "roofline frac", d["roofline"]["frac"], "cpu", d.get("cpu_baseline",{}).get("value"), d.get("cpu_baseline",{}).get("one_core_value"))
PY
done
timeout 600 python tools/probe_bench.py 14 256 1024 4096 4736 2>&1 | tail -6 | tee gpurun_out/probe_${TAG}.txt
if [ "$3" != "skip-ncu" ]; then
# every launch with its device time (cold-cache, serialised: compare shares)
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 80 --csv --log-file gpurun_out/launches_${TAG}.csv \
    python bench.py --gpus 1 --steps 2 --warmup 3 --no-cpu-baseline > gpurun_out/ncu_launch_${TAG}.log 2>&1
tail -3 gpurun_out/ncu_launch_${TAG}.log
# the per-sample kernel, full set, source view
timeout 1500 ncu --set full --clock-control none --import-source on -k regex:lpcnet_sample -s 4 -c 1 -o gpurun_out/prof_${TAG} -f \
    python bench.py --gpus 1 --steps 1 --warmup 3 --frames 3 --no-cpu-baseline > gpurun_out/ncu_full_${TAG}.log 2>&1
tail -3 gpurun_out/ncu_full_${TAG}.log
fi
ls -la gpurun_out
