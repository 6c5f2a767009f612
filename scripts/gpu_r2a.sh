#!/bin/bash
# Round 2, GPU call A: strict GPU suite (incl. bench-scale parity vs the reference binary and downstream acceptance),
# vendor onesweep yardstick, bench with the opt-in switch, launch list + section-level ncu of the non-sort kernels at
# bench size.
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.max.sm,clocks.max.mem,power.limit --format=csv > gpurun_out/gpu_info.txt 2>&1
lscpu | egrep 'Model name|^CPU\(s\)|NUMA node\(s\)' >> gpurun_out/gpu_info.txt
echo "== pytest -m gpu"
timeout 1200 python -m pytest tests -m gpu -q --timeout 900 -rxXf > gpurun_out/pytest_gpu.log 2>&1; echo "pytest rc=$?"; tail -30 gpurun_out/pytest_gpu.log
echo "== cub yardstick"
timeout 120 scripts/diag/cub_yardstick.bin 1230000000 2>&1 | tee gpurun_out/cub_yardstick.jsonl
summ() { python - "$1" <<PY
import json, sys
try:
    j = json.load(open(sys.argv[1])); r = j["roofline"]
    print(sys.argv[1], "ms/step %.1f  value %.3g  e2e %.3g (%.1f ms)  pass %.2f ms frac %.3f  stages %s  e2e-stages %s" % (
        j["ms_per_step"], j["value"], j["e2e"]["value"] or 0, j["e2e"]["ms_per_step"] or 0, r["avg_launch_ms"], r["frac"],
        {k: round(v, 1) for k, v in j["stage_ms"].items()}, {k: round(v, 1) for k, v in j["e2e"]["stages"].items() if isinstance(v, float)}))
except Exception as e:
    print(sys.argv[1], "unreadable:", e)
PY
}
echo "== bench: default (with cpu baseline)"
timeout 400 python bench.py --steps 3 --warmup 3 > gpurun_out/bench_default.json 2> gpurun_out/bench_default.err; summ gpurun_out/bench_default.json
echo "== bench: MHB_H2D_CHUNKS=4"
MHB_H2D_CHUNKS=4 timeout 300 python bench.py --steps 3 --warmup 3 --no-cpu-baseline > gpurun_out/bench_chunks.json 2> gpurun_out/bench_chunks.err; summ gpurun_out/bench_chunks.json
echo "== ncu launch list at bench size"
timeout 500 ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file gpurun_out/launches_r2a_10M.csv \
   python bench.py --steps 1 --warmup 1 --no-cpu-baseline --e2e-steps 0 > gpurun_out/ncu_list.log 2>&1; echo rc=$?
echo "== ncu sections of the non-sort kernels at bench size"
timeout 600 ncu --section SpeedOfLight --section MemoryWorkloadAnalysis --section WarpStateStats --section Occupancy --section LaunchStats --section SchedulerStats --section ComputeWorkloadAnalysis \
   --clock-control none -k 'regex:k_count_lanes|k_count_write|k_s2s_judge|k_s2s_gather|k_s2s_write|k_count_extract|k_mark_mercy|k_s2s_extract' -c 9 --csv --page raw --log-file gpurun_out/r2a_nonsort_raw.csv \
   python bench.py --steps 1 --warmup 1 --no-cpu-baseline --e2e-steps 0 > gpurun_out/ncu_nonsort.log 2>&1; echo rc=$?
du -sh gpurun_out
