#!/bin/bash
# Runs every GPU test file in its own process (a device-side trap poisons the CUDA context of the process that
# hit it) with a hard timeout, logging into gpurun_out/.  Usage: tools/run_gpu_suite.sh [pytest args]
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/gpu.txt 2>&1
rc=0
for f in tests/test_gpu_kernels.py tests/test_gpu_gemm_contract.py tests/test_gpu_engine_shapes.py tests/test_gpu_stage1.py \
         tests/test_gpu_e2e.py tests/test_gpu_pipeline.py tests/test_gpu_vep_batch.py tests/test_gpu_bpe_shapes.py \
         tests/test_gpu_ism.py tests/test_gpu_modules.py tests/test_gpu_forward_abi.py tests/test_gpu_ad_risk.py \
         tests/test_gpu_cre_attention.py tests/test_gpu_cohort.py tests/test_gpu_knockout.py \
         tests/test_gpu_deletion.py tests/test_gpu_variant_sets.py tests/test_gpu_cohort_variant_sets.py \
         tests/test_gpu_variant_attribution.py; do
  n=$(basename $f .py)
  timeout 900 python -m pytest $f -q -m gpu -s "$@" > gpurun_out/$n.log 2>&1
  r=$?
  echo "== $n exit $r"; tail -n 40 gpurun_out/$n.log
  [ $r -ne 0 ] && rc=$r
done
exit $rc
