#!/bin/bash
# Run every -m gpu test module in its own process (a faulting kernel poisons its CUDA context, not the others')
# and leave one log per module under gpurun_out/.   usage: tools/run_gpu_tests.sh [per-module timeout seconds]
T=${1:-600}
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > gpurun_out/gpu.txt 2>&1
rc_all=0
for f in tests/test_gpu_gemm.py tests/test_gpu_elementwise.py tests/test_gpu_attention.py tests/test_gpu_dit.py tests/test_gpu_sampler.py tests/test_gpu_vae.py tests/test_gpu_vae_encode.py tests/test_gpu_primsdf.py tests/test_gpu_pipeline.py tests/test_gpu_raymarch.py tests/test_gpu_ref_fp16.py tests/test_gpu_zz_extra.py; do
  n=$(basename $f .py)
  timeout $T python -m pytest $f -q -m gpu --timeout 300 --no-header -p no:cacheprovider -s > gpurun_out/$n.log 2>&1
  rc=$?
  echo "$n rc=$rc : $(tail -n 1 gpurun_out/$n.log)"
  [ $rc -ne 0 ] && rc_all=1
done
exit $rc_all
