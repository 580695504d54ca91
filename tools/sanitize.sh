# compute-sanitizer memcheck over representative parity tests (small shapes): fused GEMM + LayerNorm (single and grouped problems,
# in-place residual sources), env-batched plan, block entry, device ring, zero-shot draws, checkpoint geometry, golden planners
mkdir -p gpurun_out
timeout 1500 compute-sanitizer --tool memcheck --error-exitcode 7 --print-limit 20 python -m pytest tests/test_gpu_parity.py -x -q -m gpu \
  -k "residual_layernorm_fused and (256 or 300 or 4000) or env_batched_plan_rows and bf16 or reference_format_checkpoints and bf16 or candidate_draws and bf16 or planners_match_reference_golden and bf16 or single_candidate or select_survives" \
  > gpurun_out/san_parity.txt 2>&1; echo "rc=$?" >> gpurun_out/san_parity.txt
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 7 --print-limit 20 python -m pytest tests/test_gpu_kernels.py -x -q -m gpu \
  -k "block_forward and bf16 or k1_ or k4_ or k5_ or k8_" > gpurun_out/san_kernels.txt 2>&1; echo "rc=$?" >> gpurun_out/san_kernels.txt
timeout 600 compute-sanitizer --tool memcheck --error-exitcode 7 --print-limit 20 python -m pytest tests/test_rollout.py tests/test_valloss.py -x -q -m gpu -k "device_resident or eval_mtm_loss_matches" \
  > gpurun_out/san_rollout.txt 2>&1; echo "rc=$?" >> gpurun_out/san_rollout.txt
grep -E "ERROR SUMMARY|passed|failed|rc=|Invalid|out of bounds" gpurun_out/san_parity.txt gpurun_out/san_kernels.txt gpurun_out/san_rollout.txt | head -30
