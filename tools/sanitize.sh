# compute-sanitizer memcheck over representative parity tests (small shapes): fused GEMM + LayerNorm (single and grouped problems,
# in-place residual sources), env-batched plan, block entry, device ring, zero-shot draws, checkpoint geometry, golden planners,
# and the gather-form attention cases up to 1024 batch rows (their guard rows catch stray writes; only memcheck catches stray reads)
# usage: bash tools/sanitize.sh LOG_DIR   (one log per group of tests, LOG_DIR/san_*.txt)
OUT=${1:?usage: bash tools/sanitize.sh LOG_DIR}
mkdir -p "$OUT"
timeout 1500 compute-sanitizer --tool memcheck --error-exitcode 7 --print-limit 20 python -m pytest tests/test_gpu_parity.py -x -q -m gpu \
  -k "residual_layernorm_fused and (256 or 300 or 4000) or env_batched_plan_rows and bf16 or reference_format_checkpoints and bf16 or candidate_draws and bf16 or planners_match_reference_golden and bf16 or single_candidate or select_survives" \
  > "$OUT/san_parity.txt" 2>&1; echo "rc=$?" >> "$OUT/san_parity.txt"
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 7 --print-limit 20 python -m pytest tests/test_gpu_kernels.py -x -q -m gpu \
  -k "block_forward and bf16 or k1_ or k4_ or k5_ or k8_" > "$OUT/san_kernels.txt" 2>&1; echo "rc=$?" >> "$OUT/san_kernels.txt"
timeout 600 compute-sanitizer --tool memcheck --error-exitcode 7 --print-limit 20 python -m pytest tests/test_rollout.py tests/test_valloss.py -x -q -m gpu -k "device_resident or eval_mtm_loss_matches" \
  > "$OUT/san_rollout.txt" 2>&1; echo "rc=$?" >> "$OUT/san_rollout.txt"
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 7 --print-limit 20 python -m pytest tests/test_gpu_attention.py -x -q -m gpu \
  -k "not B8192 and not B8195" > "$OUT/san_attention.txt" 2>&1; echo "rc=$?" >> "$OUT/san_attention.txt"
grep -E "ERROR SUMMARY|passed|failed|rc=|Invalid|out of bounds" "$OUT"/san_*.txt | head -40
