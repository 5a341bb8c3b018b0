#!/bin/bash
# One GPU box, one pass: the evidence files of a round (copied from gpurun_out/<tag>/ into profiles/ afterwards).
#   gpurun --timeout 2400 -- 'bash tools/final_profile.sh r02'
# Every ncu command runs only after the same program has exited 0 without ncu.
TAG=${1:-r02}
OUT=gpurun_out/$TAG
mkdir -p $OUT
rm -f gpurun_out/parity_counts.jsonl
timeout 900 python -m pytest tests -m gpu -q -s > $OUT/pytest_gpu.log 2>&1; echo "pytest rc=$?" | tee -a $OUT/pytest_gpu.log
cp gpurun_out/parity_counts.jsonl $OUT/ 2>/dev/null
timeout 600 python bench.py --steps 20 --warmup 5 > $OUT/bench_n1.json 2> $OUT/bench_n1.err; echo "bench rc=$?"
timeout 120 python tools/profile_step.py cfg2 2 > $OUT/plain_cfg2.log 2>&1 && \
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/launches_cfg2.csv python tools/profile_step.py cfg2 2 > $OUT/ncu_l2.log 2>&1
timeout 120 python bench.py --steps 2 --warmup 3 --no-extras --no-cpu-baseline > $OUT/plain_bench.log 2>&1 && \
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $OUT/launches_bench.csv python bench.py --steps 2 --warmup 3 --no-extras --no-cpu-baseline > $OUT/ncu_lb.log 2>&1
timeout 400 ncu --set full --clock-control none --import-source on -k regex:"maxmean_tc|dq_pipe|dv_group_sort|dv_gather_grouped|nce_head|nce_partial|dT_kernel|finalize_clip" -c 8 -o $OUT/prof_cfg2 -f python tools/profile_step.py cfg2 1 > $OUT/ncu_full2.log 2>&1
timeout 120 python tools/profile_step.py cfg3 2 > $OUT/plain_cfg3.log 2>&1 && \
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/launches_cfg3.csv python tools/profile_step.py cfg3 2 > $OUT/ncu_l3.log 2>&1
timeout 400 ncu --set full --clock-control none -k regex:"maxmean_tc|dq_pipe|dv_gather_grouped" -c 3 -o $OUT/prof_cfg3 -f python tools/profile_step.py cfg3 1 > $OUT/ncu_full3.log 2>&1
timeout 200 python tools/timeline.py cfg2 6 > $OUT/timeline_cfg2.txt 2>&1
timeout 200 python tools/timeline.py cfg3 6 > $OUT/timeline_cfg3.txt 2>&1
timeout 200 python tools/timeline.py cfg2 4 full > $OUT/timeline_cfg2_full_loss.txt 2>&1
timeout 200 python tools/step_trace.py 100 > $OUT/step_trace.txt 2>&1
timeout 200 python tools/power_probe.py > $OUT/power_probe.txt 2>&1
ls -la $OUT
