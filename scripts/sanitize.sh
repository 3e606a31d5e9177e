#!/bin/bash
# compute-sanitizer over the round-2 kernels (3xTF32 projection / weight-gradient GEMMs, fused step, the compact-batch
# widening): memcheck and racecheck, small shapes.  GPU box, one GPU.
set -u
tag=${1:-r5}
SEL='test_x3_projection_forward_is_fp32_grade or test_x3_projection_backward_is_fp32_grade or test_fused_step_equals_autograd_path_and_torch_adam or test_prefetcher_widens_the_compact_wire_format_bit_exactly'
for tool in memcheck racecheck; do
  timeout 1500 compute-sanitizer --tool $tool --print-limit 20 python -m pytest tests/test_gpu_tc.py tests/test_gpu_heads.py \
    tests/test_gpu_model.py tests/test_gpu_arena.py -q -m gpu -k "$SEL" -p no:cacheprovider \
    > gpurun_out/${tag}_${tool}.log 2>&1
  echo "== $tool rc=$?"; grep -E "ERROR SUMMARY|passed|failed|error" gpurun_out/${tag}_${tool}.log | tail -5
done
