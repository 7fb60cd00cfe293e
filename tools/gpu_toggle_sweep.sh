#!/bin/bash
# parity suites of the encoder under every scheduling / kernel-selection switch (each switch alone)
mkdir -p gpurun_out
: > gpurun_out/r6q_toggle_sweep.log
for kv in "CFB_GEMM_2CTA=0" "CFB_GEMM_2CTA=1" "CFB_ATTN_PERSIST=0" "CFB_ATTN_PERSIST=1" "CFB_FUSED_TAIL=0" "CFB_FUSED_TAIL=2" "CFB_PACKED_GROUPS=1" "CFB_PACKED_GROUPS=2" "CFB_PACKED_GROUPS=4"; do
  r=$(env $kv timeout 600 python -m pytest tests/test_gpu_encoder.py tests/test_gpu_packed.py tests/test_gpu_canary.py -x -q 2>&1 | tail -1)
  echo "$kv: $r" | tee -a gpurun_out/r6q_toggle_sweep.log
done
