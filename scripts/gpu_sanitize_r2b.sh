#!/bin/bash
# compute-sanitizer over the kernels added in the second half of round 2: per-video weight gradient, displaced pooling (3dconv).
mkdir -p gpurun_out
SEL='(wgrad_video and 3-64-256-128) or (wgrad_video and 2-128-136-200) or (pool3d_displaced and 5-7-2-3-24) or (pool3d_displaced and 4-6-2-2-8) or (conv3d_projector_training and 24-32) or (variants_match_reference and conv3d_tiny)'
for TOOL in memcheck synccheck; do
  echo "=== $TOOL ==="
  timeout 900 compute-sanitizer --tool $TOOL --error-exitcode 99 python -m pytest tests/test_gpu_parity.py -m gpu -x -q -k "$SEL" > gpurun_out/sanitize_r2b_$TOOL.log 2>&1
  echo "rc=$?"; grep -E "ERROR SUMMARY|passed|failed" gpurun_out/sanitize_r2b_$TOOL.log | tail -3
done
