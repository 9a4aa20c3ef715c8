#!/bin/bash
# Full GPU parity pass, one process per test file so that a trapped kernel cannot poison the others.
# usage (from the repo root, under gpurun): bash tools/gpu_check.sh [files...]
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,driver_version,memory.total --format=csv > gpurun_out/smi.txt 2>&1
FILES=${@:-"tests/test_gpu_fp32.py tests/test_gpu_tc_accum.py tests/test_gpu_tc_accum_fullsize.py tests/test_gpu_quantify.py tests/test_gpu_rolling_ball.py tests/test_gpu_resize.py tests/test_gpu_overlay.py tests/test_gpu_density.py tests/test_gpu_properties.py tests/test_gpu_conv.py tests/test_gpu_exact.py tests/test_gpu_forward.py tests/test_gpu_fullsize.py tests/test_gpu_envelope.py tests/test_gpu_rolling_ball_banded.py tests/test_gpu_cli.py tests/test_gpu_csv.py tests/test_gpu_png.py tests/test_gpu_stress.py"}
rc=0
for f in $FILES; do
  n=$(basename $f .py)
  echo "=== $f"
  timeout 900 python -m pytest $f -q -rP -m gpu --tb=short --maxfail=8 > gpurun_out/$n.log 2>&1
  r=$?
  tail -n 25 gpurun_out/$n.log
  if [ $r -ne 0 ]; then rc=1; fi
  if [ "$n" = "test_gpu_conv" ] && [ $r -ne 0 ]; then
    echo "=== conv_debug"
    timeout 300 python tools/conv_debug.py > gpurun_out/conv_debug.log 2>&1
    tail -n 60 gpurun_out/conv_debug.log
  fi
done
exit $rc
