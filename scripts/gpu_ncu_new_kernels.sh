#!/bin/bash
# Round 2: ncu evidence for the kernels added in the second half (one GPU; numbers printed under ncu are never bench values).
mkdir -p gpurun_out
echo "=== launch list of the bench command ==="
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/r2b_launches.csv python bench.py --steps 2 --warmup 1 --no-e2e --no-cpu-baseline --no-configs --no-torch-eager --no-sustained > gpurun_out/r2b_launches.log 2>&1
echo "rc=$?"
echo "=== full capture: per-video weight gradient (64 videos, C = 1024) ==="
TRAIN_STEP_ONLY=fused_training timeout 900 ncu --set full --clock-control none --import-source on -k regex:gemm_wgrad_video -s 8 -c 1 -f -o gpurun_out/r2b_prof_wgrad_video python scripts/gpu_train_step.py 64 > gpurun_out/r2b_prof_wgrad_video.log 2>&1
echo "rc=$?"
ls -la gpurun_out/*.ncu-rep
