#!/usr/bin/env bash
# Run each GPU op test in its own process (a device trap poisons the CUDA context).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > gpurun_out/gpu.txt 2>&1
: > gpurun_out/ops.log
for t in test_gemm_bias test_gemm_residual_alpha_rowvec_fp32 test_gemm_out_slice test_gemm_geglu test_conv3x3 \
         test_group_norm test_group_norm_sft test_layer_norm test_attention \
         test_attention_fused_qkv_and_peaky test_layout_strided_upsample_concat_misc test_sampler_kernels; do
  echo "=== $t" >> gpurun_out/ops.log
  timeout 300 python -m pytest tests/test_ops_gpu.py -q -m gpu -k "$t and not ${t}_" --tb=short -p no:cacheprovider 2>&1 | tail -40 >> gpurun_out/ops.log
done
grep -E "^===|passed|failed|error" gpurun_out/ops.log
