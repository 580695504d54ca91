/*
 * m3pc.h -- C-ABI of the B200-native (sm_100a) M^3PC test-time-planning hot path.
 *
 * The reference (wkh923/m3pc) is pure Python/PyTorch and has NO FFI; this header is the boundary a
 * maintainer would bind from Python (ctypes / cffi / a torch extension shim, see INTEGRATION.md).
 * Every entry point cites the reference interface it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - plain pointers + sizes + a CUDA stream (passed as void*, i.e. cudaStream_t); no torch types.
 *   - every function returns 0 on success, <0 on error (never throws across the ABI);
 *     m3pc_last_error() returns a thread-local message for the last failing call.
 *   - the caller allocates and owns all I/O buffers ("device" = device pointer, "host" = host pointer);
 *     the library owns only what hangs off the handle (packed weights, workspaces).
 *   - all work is enqueued on the caller's stream; no internal host synchronisation except in
 *     m3pc_create / m3pc_finalize_params / m3pc_destroy.
 *   - one handle per (process, device); calls on one handle must be externally serialised.
 *   - there is no CPU fallback: without a sm_100 device every compute call fails with M3PC_ERR_CUDA.
 *
 * Activation layout inside the library is token-major: row = token * B + b (B = batch of candidates or
 * environments).  It is never exposed: all I/O tensors below use the reference's (B, T, d) layout.
 */
#ifndef M3PC_H_
#define M3PC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define M3PC_OK 0
#define M3PC_ERR_INVALID (-1) /* bad argument / unsupported configuration */
#define M3PC_ERR_CUDA (-2)    /* CUDA runtime / driver error, or no sm_100 device */
#define M3PC_ERR_STATE (-3)   /* call order violated (e.g. forward before finalize_params) */
#define M3PC_ERR_NOMEM (-4)

#define M3PC_PREC_BF16 0 /* bf16 operands on tcgen05 tensor cores, fp32 accumulate, fp32 residual stream */
#define M3PC_PREC_FP32 1 /* fp32 operands and accumulate on CUDA cores (reference-grade, 1e-5) */
/* fp32 operands, activations and residual stream as M3PC_PREC_FP32; the contractions on tcgen05 tensor cores (kind::tf32) with
 * each operand split into a tf32 high part and an fp32 remainder, three MMAs per product, fp32 accumulate: fp32-grade accuracy */
#define M3PC_PREC_TF32X3 2

/* modality order everywhere: the reference's dict order, finetune_omtm/learner.py:361-366 */
#define M3PC_STATES 0
#define M3PC_ACTIONS 1
#define M3PC_REWARDS 2
#define M3PC_RETURNS 3

#define M3PC_MAX_T 16    /* traj_length limit (tokens = 4*T <= 64) */
#define M3PC_MAX_ACT 32  /* action dim limit */
#define M3PC_MAX_OBS 128 /* observation dim limit */

/* plan_guidance values, finetune_omtm/learner.py:388-412 */
#define M3PC_GUIDE_RTG 0          /* rtg_guiding            learner.py:271-327 */
#define M3PC_GUIDE_CRITIC 1       /* critic_lambda_guiding  learner.py:211-268 */
#define M3PC_GUIDE_NOISE_CRITIC 2 /* noise_adding_lambda    learner.py:142-208 */
#define M3PC_GUIDE_SAMPLING 3     /* plan=False: mtm_sampling learner.py:103-115 */

typedef struct m3pc_engine* m3pc_handle_t;

/* Replaces omtmConfig + data_shapes + traj_length (omtm/models/mtm_model.py:200-221, 324-437). */
typedef struct {
  int32_t n_embd;      /* multiple of 128; head_dim must be 128 */
  int32_t n_head;      /* n_embd / 128 */
  int32_t n_enc_layer;
  int32_t n_dec_layer;
  int32_t traj_length; /* T <= M3PC_MAX_T */
  int32_t obs_dim;
  int32_t act_dim;
  int32_t precision;     /* M3PC_PREC_* */
  int32_t max_batch;     /* largest B (candidates or envs) a call will pass */
  int32_t chunk;         /* B rows per kernel sequence (L2 blocking); 0 = library default */
  int32_t critic_hidden; /* TwinQ hidden width (256 in the reference); 0 = no critic */
  int32_t reserved[5];
} m3pc_config_t;

const char* m3pc_last_error(void);
const char* m3pc_version(void);

/* Learner.__init__ model construction (finetune_omtm/learner.py:30-36). */
int m3pc_create(m3pc_handle_t* out, const m3pc_config_t* cfg);
int m3pc_destroy(m3pc_handle_t h);

/*
 * omtm.load_state_dict (learner.py:33-35), TwinQ weights (finetune_omtm/model.py:146-160) and tokenizer
 * statistics (omtm/tokenizers/continuous.py:32-62), by NAME:
 *   - every key of the reference's omtm.state_dict(), verbatim ("encoder.layers.0.linear1.weight", ...);
 *   - "critic.q1.net.0.weight" ... "critic.q2.net.4.bias", "critic.obs_mean", "critic.obs_std";
 *   - "tokenizer.<modality>.mean" / ".std" for states, rewards, returns (actions are not normalised).
 * `data` is a HOST pointer to `count` fp32 values in the tensor's row-major order.
 */
int m3pc_set_param(m3pc_handle_t h, const char* name, const float* data, size_t count);
/* Packs weights for the device (bf16 K-major copies, fused constants). Must follow the last m3pc_set_param.
 * The handle keeps the host copies, so a later m3pc_set_param of ANY subset of the names followed by another
 * m3pc_finalize_params re-packs with the new values (the reference mutates parameters in place on every optimiser step,
 * finetune_omtm/learner.py:506-538).  Both calls drop every CUDA graph the handle has captured: a graph freezes the
 * parameter addresses and the scalar statistics it was captured with. */
int m3pc_finalize_params(m3pc_handle_t h);

/* Selects between RESULT-EQUIVALENT launch sequences of the handle (parity tests compare them; none changes what is
 * computed).  Unknown names fail with M3PC_ERR_INVALID.  Names and defaults:
 *   "graphs" 1                 capture m3pc_plan into a CUDA graph and replay it (0: launch every kernel eagerly)
 *   "fused_b1" 1               one cooperative kernel for a B = 1 forward (0: one launch per op)
 *   "fused_ln_min_rows" 1024   smallest GEMM (rows) the fused residual GEMM + LayerNorm kernel is used for (>= 129; below, the
 *                              GEMM is followed by a LayerNorm kernel)
 *   "restrict_deep_decoder" 1  decoders with > 1 layer: last layer on the consumed rows only (0: every row)
 *   "gemm_ln_unit_rows" 0      rows per CTA-pair unit of the fused residual GEMM + LayerNorm kernel: 128 = two accumulators in
 *                              tensor memory (the epilogue of a unit overlaps the MMAs of the next), 256 = one accumulator with
 *                              1/3 less operand traffic per FLOP, 0 = chosen per launch from K and the row count
 *                              (process-wide; bit-identical results)
 * The release library reads no environment variable. */
int m3pc_set_option(m3pc_handle_t h, const char* name, int32_t value);

/*
 * omtm.forward(trajectories, masks)  (mtm_model.py:593-607), P = 1 token per time step.
 *   tok_*   device fp32, tokenised inputs (B,T,d) (what TokenizerManager.encode returns, squeezed)
 *   masks   HOST, 4*T bytes of {0,1}, modality-major (states, actions, rewards, returns)
 *   out_*   device fp32 (B,T,d) raw head outputs (before TokenizerManager.decode); any may be NULL.
 *           out_act_mu / out_act_std are the parameters of the reference's SquashedNormal
 *           (mtm_model.py:313-321): mean = tanh(mu), sample = tanh(mu + std*eps).
 */
int m3pc_forward(m3pc_handle_t h, int32_t batch, const float* tok_states, const float* tok_actions,
                 const float* tok_rewards, const float* tok_returns, const uint8_t* masks, float* out_states,
                 float* out_act_mu, float* out_act_std, float* out_rewards, float* out_returns, void* stream);

/* Per-shard record for the multi-GPU combine (SURVEY.md section 8e). Floats, in this order:
 *   [0] m = max_n J_n   [1] Z = sum exp(tau (J_n - m))   [2] best J   [3] best global idx (as float bits of int32)
 *   [4] best sample key p_n/q_n (relative to local m)   [5] its global idx (int32 bits)   [6] n_cand
 *   [7] reserved   [8 .. 8+A) U = sum exp(tau (J_n - m)) * a0_n   [8+A .. 8+2A) a0 of best key   */
#define M3PC_PARTIAL_FLOATS (8 + 2 * M3PC_MAX_ACT)

/* Learner.rtg_guiding / critic_lambda_guiding / noise_adding_lambda / mtm_sampling on one window
 * (finetune_omtm/learner.py:103-327), after Learner.action_sample built the window (learner.py:342-385). */
typedef struct {
  int32_t guidance;     /* M3PC_GUIDE_* */
  int32_t horizon;      /* h: the planner conditions on tokens < T-h and plans tokens >= T-h */
  int32_t n_cand;       /* candidates evaluated by THIS call (cfg.action_samples, or this rank's shard) */
  int32_t cand_offset;  /* global id of local candidate 0 (noise / index bookkeeping under sharding) */
  float discount;       /* cfg.discount */
  float temperature;    /* cfg.temperature */
  float lmbda;          /* cfg.lmbda (rtg_guiding: the reference hard-codes 0.6, learner.py:272,405-407) */
  int32_t n_env;        /* 0 or 1: one window (the reference's call).  E > 1: E lock-step environments planned in ONE launch
                           sequence (pass 1 at B = E, pass 2 at B = E*n_cand; SURVEY.md section 8f rank 1): every win_* pointer
                           gains a leading E axis, eps is (E*n_cand,h,A), expq (E*n_cand), out_*_action (E,A),
                           dbg_expect_return (E*n_cand), dbg_candidates (E*n_cand,h,A), dbg_indices (E,2) with indices local
                           to the environment; out_partials must be NULL.  Needs E*n_cand <= cfg.max_batch.  Row e of the
                           result equals the single-window call on window e with the same injected noise. */
  const float* win_states;      /* device (T,obs) RAW window (zero padded), learner.py:348-366 */
  const float* win_actions;     /* device (T,act) RAW */
  const float* win_rewards;     /* device (T) RAW */
  const float* win_returns_tok; /* device (T) TOKENISED returns: the host evaluates (rtg-mean)/std in
                                   float64 and rounds to fp32 exactly as the reference does (learner.py:368-385,
                                   continuous.py:74-79) */
  const float* eps;   /* device: injected N(0,1) noise, (n_cand,h,A) for guidance 0/1/2, (A) for 3; NULL = Philox */
  const float* expq;  /* device (n_cand): injected Exp(1) draws of torch.multinomial; NULL = Philox */
  uint64_t seed;      /* Philox key when eps/expq are NULL; counter = global candidate id */
  float* out_eval_action;   /* device (A)  learner.py:323  (mtm_sampling: tanh(mu)) */
  float* out_sample_action; /* device (A)  learner.py:324-325 */
  float* out_partials;      /* device (M3PC_PARTIAL_FLOATS) or NULL */
  float* dbg_expect_return; /* device (n_cand) or NULL: J_n before the max subtraction */
  float* dbg_candidates;    /* device (n_cand,h,A) or NULL */
  int32_t* dbg_indices;     /* device (2) or NULL: [argmax_n J_n, sampled idx] (global ids) */
  int32_t exchange;         /* 1 (n_env <= 1, after m3pc_exchange_connect): this call plans ONE SHARD of the candidates; its selection
                               kernel stores the shard record into every rank's exchange buffer over peer memory (NVLink), waits for
                               the records of all ranks and merges them, so out_eval_action / out_sample_action / dbg_indices hold
                               the GLOBAL result on every rank -- no collective launch, nothing outside the captured CUDA graph.
                               Every rank of the group must issue the same sequence of exchange plans. */
  int32_t reserved0;
  const int32_t* env_horizons; /* HOST (max(n_env, 1)) or NULL: one horizon per environment, each in [1, traj_length]
                                  (learner.py:342-345 clamps the horizon of an environment in its first T - h steps).  `horizon`
                                  must equal the largest entry, which fixes the layouts: eps and dbg_candidates stay
                                  (E*n_cand, horizon, A) and environment e uses the first env_horizons[e] steps of its rows.  All
                                  entries equal: exactly the call with NULL.  Otherwise the environments are split into horizon
                                  classes and each class is planned as the uniform call on its windows at n_env = E_c (bit for bit),
                                  all in one launch sequence (one CUDA graph per horizon pattern).  Philox is keyed by the caller's
                                  environment index, so an environment's draws do not depend on the other environments of the call.
                                  Needs n_env <= 256; cannot be combined with exchange, out_partials or cand_offset. */
  void* reserved1[2];
} m3pc_plan_args_t;

int m3pc_plan(m3pc_handle_t h, const m3pc_plan_args_t* args, void* stream);

/* Peer exchange of the per-shard records (SURVEY.md section 8e: "only per-shard best scores/indices are combined ... over
 * NVLink").  The reference is single-GPU (finetune.py:154); this is the one exchange step candidate sharding adds.
 *   m3pc_exchange_local    allocates this handle's exchange buffer (once) and returns a CUDA IPC handle for it
 *                          (M3PC_IPC_HANDLE_BYTES bytes, for peers in other processes) and/or its device pointer (peers in the
 *                          same process); either output may be NULL.
 *   m3pc_exchange_connect  wires the group: `ipc_handles` = world handles concatenated in rank order (e.g. gathered with
 *                          torch.distributed.all_gather_object) -- opened with cudaIpcOpenMemHandle, which enables peer
 *                          access -- OR `device_ptrs` = world device pointers valid on this device; the other must be NULL.
 *                          Resets the epoch sequence: all ranks (re)connect together.  world <= 32.
 *   m3pc_exchange_status   epochs completed, and the epoch of a wait that timed out (0 = none; a rank whose peer never
 *                          launched its plan gives up after 2 s and returns NaN actions instead of hanging the GPU). */
#define M3PC_IPC_HANDLE_BYTES 64
int m3pc_exchange_local(m3pc_handle_t h, uint8_t* out_ipc_handle, void** out_device_ptr);
int m3pc_exchange_connect(m3pc_handle_t h, int32_t rank, int32_t world, const uint8_t* ipc_handles, void* const* device_ptrs);
int m3pc_exchange_status(m3pc_handle_t h, uint64_t* out_epoch, uint64_t* out_failed_epoch);

/* Combine `n_shards` records (device, n_shards*M3PC_PARTIAL_FLOATS, e.g. the output of an NCCL all-gather)
 * into the global eval / sample action: log-sum-exp merge of the per-shard softmax partials. */
int m3pc_merge_partials(m3pc_handle_t h, const float* partials, int32_t n_shards, float temperature,
                        float* out_eval_action, float* out_sample_action, int32_t* out_indices, void* stream);

/* Zero-shot backward planners on E lock-step environments (zeroshot_omtm/learner.py:60-261); m3pc_backward_plan_env below plans
 * environments at different points of their episodes.
 *   mode 0 = action_id_sample (one pass, gid mask); 1 = action_piid_sample (pi mask -> fill states -> fid mask).
 *   win_* as in m3pc_plan_args_t but with a leading E axis: (E,T,obs) etc.; eps (E,A) or NULL (mean only).
 *   out_eval_action / out_sample_action: device (E,A). */
int m3pc_backward_plan(m3pc_handle_t h, int32_t mode, int32_t n_env, int32_t horizon, const float* win_states,
                       const float* win_actions, const float* win_rewards, const float* win_returns_tok,
                       const float* eps, float* out_eval_action, float* out_sample_action, float* dbg_states_filled,
                       void* stream);

/* m3pc_backward_plan with C action draws per environment (BASELINE.json config 4: "256 parallel envs x 512 candidates").
 * The reference draws ONE action per call, ``action_dist.sample()`` at step T-h of the last pass
 * (zeroshot_omtm/learner.py:136-147, :248-259); C calls on the same history draw C i.i.d. actions from the same
 * distribution.  Here the (one or two) forward passes run once per environment and all C draws come from their action
 * head:   out_sample_actions[e, c, :] = tanh(mu_e + std_e * eps[e, c, :]),   out_eval_action[e, :] = tanh(mu_e).
 *   eps   device (E, C, A) injected N(0,1) noise, or NULL: Philox keyed by (seed, environment, draw)
 *   out_sample_actions device (E, C, A);  n_draws = 1 with the same eps is exactly m3pc_backward_plan. */
int m3pc_backward_plan_draws(m3pc_handle_t h, int32_t mode, int32_t n_env, int32_t horizon, int32_t n_draws, const float* win_states,
                             const float* win_actions, const float* win_rewards, const float* win_returns_tok, const float* eps,
                             uint64_t seed, float* out_eval_action, float* out_sample_actions, void* stream);

/* m3pc_backward_plan_draws with one planning horizon per environment (learner.py:342-345 clamps the horizon of an environment in
 * its first T - h steps), the semantics of m3pc_plan_args_t.env_horizons:
 *   env_horizons  HOST (n_env), each in [1, traj_length]; n_env <= 256 (and <= cfg.max_batch).  M3PC_ERR_INVALID otherwise, before
 *                 any launch.
 *   eps           device (E, C, A) injected N(0,1) noise or NULL (Philox keyed by (seed, environment, draw)); out_sample_actions
 *                 device (E, C, A), (E, A) for C = 1; out_eval_action device (E, A).
 * All entries equal: exactly m3pc_backward_plan_draws at that horizon.  Otherwise the environments are split into horizon classes:
 * one launch gathers their windows, then each class runs the uniform sequence at n_env = E_c on its windows, so each class computes
 * bit for bit what the uniform call on its windows (and its eps rows) computes.  Outputs land in the caller's rows and Philox is keyed
 * by the caller's environment index, so an environment's draws do not depend on the other environments of the call.  The
 * end-of-waypoints clamp (p + h > 1000) changes window contents only and needs no class of its own. */
int m3pc_backward_plan_env(m3pc_handle_t h, int32_t mode, int32_t n_env, const int32_t* env_horizons, int32_t n_draws, const float* win_states,
                           const float* win_actions, const float* win_rewards, const float* win_returns_tok, const float* eps, uint64_t seed,
                           float* out_eval_action, float* out_sample_actions, void* stream);

/* Device-resident episode histories of n_env environment slots (SURVEY.md section 8f rank 1): what the reference keeps as
 * `current_trajectory` numpy arrays (replay_buffer.py:192-205, learner.py:663-675) and re-slices on the host every step
 * (learner.py:346-366).  Each step uploads n*(obs+act+1) floats instead of n windows.
 *   ring: device fp32 (n_env, ring_len, obs+act+1); row t of a slot = [observation | action | reward] of step t of its episode.
 *   Every slot has its own clock, so episodes may end at different steps and a slot may start the next episode at once.
 *   `slots` is a HOST list of n_slots slot indices (any length: it travels in kernel parameters, 256 per launch); per-slot inputs
 *   and outputs are in list order.  `t` / `path_length` are DEVICE (n_env) int32 tables indexed by slot.
 *   m3pc_ring_reset          zeroes the whole history of the listed slots: a new episode (rollout.new_trajectory).  Without it the
 *                            actions / rewards of the previous episode would show up in the windows of the next.
 *   m3pc_ring_append_slots   listed slot k = slots[k] writes obs row k at step t[slot] and (when non-NULL) prev_action row k /
 *                            prev_reward[k] at step t[slot] - 1; a slot with t outside [0, ring_len) writes nothing.
 *   m3pc_ring_write_obs      writes only the observation columns of rows [first_row, first_row + n_rows) of each listed slot from
 *                            obs_rows (device (n_slots, n_rows, obs)): the waypoint table of a zero-shot episode
 *                            (zeroshot_omtm/learner.py:75-79), stored once after m3pc_ring_reset.  The appends that follow overwrite
 *                            rows 0 .. path_length with the observations of the episode, so windows with future_obs see what the
 *                            host builder sees on a history whose observations array holds the waypoints.
 *   m3pc_ring_windows_slots  window k of the (n_slots, T, .) planner windows is slot s = slots[k] at step p = path_length[s] with
 *                            horizon h = horizons[k] (HOST list, in [1, T]), exactly as learner.py:346-366 builds it: the states,
 *                            actions and rewards of steps p-T+h .. p (the last T-h+1 steps, zero where before step 0), zero padded
 *                            to T.  With future_obs the states window instead holds the T stored steps from p-T+h on, the future
 *                            waypoints included (zeroshot_omtm/learner.py:77-79, :97-106); when p+h > 1000 only the first
 *                            max(T-(p+h-1000), T-h+1) of them, the rest zero.  Every step of the return window is rtg_tok[k]
 *                            (device (n_slots)), the tokenised return-to-go the host computes as for m3pc_plan_args_t.win_returns_tok. */
int m3pc_ring_reset(float* ring, int32_t n_env, int32_t ring_len, int32_t obs_dim, int32_t act_dim, const int32_t* slots, int32_t n_slots,
                    void* stream);
int m3pc_ring_append_slots(float* ring, int32_t n_env, int32_t ring_len, int32_t obs_dim, int32_t act_dim, const int32_t* t, const int32_t* slots,
                           int32_t n_slots, const float* obs, const float* prev_action, const float* prev_reward, void* stream);
int m3pc_ring_write_obs(float* ring, int32_t n_env, int32_t ring_len, int32_t obs_dim, int32_t act_dim, const int32_t* slots, int32_t n_slots,
                        int32_t first_row, int32_t n_rows, const float* obs_rows, void* stream);
int m3pc_ring_windows_slots(const float* ring, int32_t n_env, int32_t ring_len, int32_t obs_dim, int32_t act_dim, const int32_t* path_length,
                            const int32_t* slots, const int32_t* horizons, int32_t n_slots, int32_t traj_length, int32_t future_obs,
                            const float* rtg_tok, float* win_states, float* win_actions, float* win_rewards, float* win_returns_tok,
                            void* stream);

/* ---- kernel-level entry points (unit parity tests and profiling; same kernels the calls above launch) ---- */

/* C[M,N] = epilogue(A[M,K] * W[N,K]^T): flags bit0 = GELU(erf), bit1 = C += residual (fp32 in place, C is fp32),
 * bit2 = ReLU. bias (N) fp32 or NULL.  bf16 variant: A, W are bf16 (device), C is bf16 unless bit1 (then fp32). */
int m3pc_gemm_bf16(const void* A, const void* W, const float* bias, void* C, int32_t M, int32_t N, int32_t K,
                   int32_t flags, void* stream);
int m3pc_gemm_fp32(const float* A, const float* W, const float* bias, float* C, int32_t M, int32_t N, int32_t K,
                   int32_t flags, void* stream);
/* m3pc_gemm_fp32's contract on the tensor cores with the 3xTF32 split (the GEMM of M3PC_PREC_TF32X3): problems of at most 128
 * rows, with N not a multiple of 256 or with K not a multiple of 4 run on the CUDA-core fp32 kernel.  A, W, C and bias (when
 * not NULL) must be 16-byte aligned; M3PC_ERR_INVALID otherwise. */
int m3pc_gemm_tf32x3(const float* A, const float* W, const float* bias, float* C, int32_t M, int32_t N, int32_t K,
                     int32_t flags, void* stream);
/* n independent bf16 GEMMs (arrays of n operands / shapes / flags as in m3pc_gemm_bf16; bias may be NULL or hold NULLs)
 * in as few launches as possible: up to 4 problems whose N are multiples of 256 share one launch of the CTA-pair
 * tensor-core kernel -- how the engine issues the decoder-embedding runs, the decoder K/V + Q projections, the
 * per-modality output heads (mtm_model.py:646-661, :428-433) and the two critics (finetune_omtm/model.py:146-171). */
int m3pc_gemm_bf16_grouped(int32_t n, const void* const* A, const void* const* W, const float* const* bias,
                           void* const* C, const int32_t* M, const int32_t* N, const int32_t* K, const int32_t* flags,
                           void* stream);
/* Fused residual GEMM + LayerNorm (N = 512): X[M,512] (fp32, in place) += A[M,K] W[512,K]^T + bias, or, with `table`,
 * X = table[row / rows_per_group] + A W^T + bias; Y[M,512] (bf16) = LayerNorm(X; gamma, beta), eps 1e-5.  A, W bf16. */
int m3pc_gemm_ln_bf16(const void* A, const void* W, const float* bias, float* X, void* Y, const float* gamma, const float* beta,
                      const float* table, int32_t rows_per_group, int32_t M, int32_t K, void* stream);

/* Epilogue flags of m3pc_gemm_bf16_problems (the first three are those of m3pc_gemm_bf16). */
#define M3PC_EPI_GELU 1      /* GELU(erf) */
#define M3PC_EPI_RESIDUAL 2  /* C (fp32) += result, in place */
#define M3PC_EPI_RELU 4      /* ReLU, after GELU when both are set */
#define M3PC_EPI_ROWTABLE 8  /* add table[(row / rows_per_group) * N + col] before the activations */
#define M3PC_EPI_OUT_F32 16  /* C is fp32 without a residual */
/* One bf16 GEMM C[M,N] = act(A[M,K] W[N,K]^T + bias + table[row / rows_per_group]) (+ C with M3PC_EPI_RESIDUAL).  A, W, C device,
 * 16-byte aligned; bias (N) fp32 or NULL; table (ceil(M / rows_per_group), N) fp32, given exactly when M3PC_EPI_ROWTABLE is set.
 * bias and table must be 16-byte aligned (the epilogues read them with vector loads); rows_per_group >= 1; K % 64 == 0,
 * N % 128 == 0.  M3PC_EPI_ROWTABLE and M3PC_EPI_RESIDUAL exclude each other. */
typedef struct {
  const void* A;
  const void* W;
  const float* bias;
  const float* table;
  void* C;
  int32_t M, N, K;
  int32_t rows_per_group;
  int32_t flags;
} m3pc_gemm_problem_t;
/* The n >= 1 problems of the HOST array p, issued as the engine issues its grouped GEMMs: 4 at a time, a group of problems whose N
 * are multiples of 256 as one launch of the CTA-pair kernel when one of them has more than 128 rows, every other problem on its own.
 * Every argument is checked before any CUDA call; M3PC_ERR_INVALID otherwise.  out_kernel: NULL, or HOST int32[4n] that receives
 * {kind, a, b, launch} per problem: kind 0 = the skinny CUDA-core kernel (M <= 32); 1 = the single-CTA tensor-core kernel with
 * a = tile width BN and b = cluster size; 2 = the CTA-pair kernel with a = 1 when its pairs stride over the units (else 0) and
 * b = the problems sharing that launch; launch = index of the kernel launch within this call. */
int m3pc_gemm_bf16_problems(const m3pc_gemm_problem_t* p, int32_t n, int32_t* out_kernel, void* stream);
/* One job of m3pc_gemm_ln_bf16_grouped: X[M,512] = residual + A[M,K] W[512,K]^T + bias, Y[M,512] (bf16) = LayerNorm(X).  The
 * residual is table[row / rows_per_group] when table is set, else the fp32 rows R (left unchanged) when R is set, else X itself
 * (in place).  A, W, X, Y, R and table 16-byte aligned; table and R exclude each other; rows_per_group >= 1. */
typedef struct {
  const void* A;
  const void* W;
  float* X;
  void* Y;
  const float* table;
  const float* R;
  int32_t rows_per_group;
  int32_t M;
} m3pc_ln_job_t;
/* 1 .. 4 jobs of the fused residual GEMM + LayerNorm in one launch (shared K, bias (512) or NULL, gamma, beta).  out_kernel: NULL,
 * or HOST int32[2] that receives {rows per CTA-pair unit (128 or 256), CTA pairs} of the launch. */
int m3pc_gemm_ln_bf16_grouped(const m3pc_ln_job_t* jobs, int32_t n, const float* bias, const float* gamma, const float* beta, int32_t K,
                              int32_t* out_kernel, void* stream);
/* y = LayerNorm(x) over the last dim (eps 1e-5); x fp32 (M,D); y bf16 (out_bf16=1) or fp32. */
int m3pc_layernorm(const float* x, const float* gamma, const float* beta, void* y, int32_t M, int32_t D,
                   int32_t out_bf16, void* stream);
/* Bidirectional attention over token-major qkv (S*B rows, 3*D cols), head_dim 128; out (S*B, D). */
int m3pc_attention(const void* qkv, void* out, int32_t B, int32_t S, int32_t n_head, int32_t is_bf16, void* stream);
/* One token of m3pc_attention_gather: its row for batch row b starts at ptr + (bdiv > 0 ? b / bdiv : b) * bstride elements
 * (bstride 0: one row for the whole batch; bdiv > 0: one row per group of bdiv batch rows).  Head h is columns h*128 .. h*128+127. */
typedef struct {
  const void* ptr;
  int32_t bstride;
  int32_t bdiv;
} m3pc_attn_tok_t;
/* The token-gather attention the engine runs in pass 2 (queries, keys and values each from their own rows):
 * out[i*B + b, h*128 + d] = softmax_j(q_i(b,h) . k_j(b,h) / sqrt(128)) v_j(b,h)[d], out (n_q*B, n_head*128) device, bf16
 * (is_bf16) or fp32 like every operand.  q, k, v are HOST arrays of n_q, n_kv, n_kv headers; n_q, n_kv in [1, 64].
 * n_kv_batch > 0 names keys [0, n_kv_batch) per-batch-row and keys [n_kv_batch, n_kv) shared: the bf16 path then takes the
 * shared-key kernel (constant K / V staged once per CTA of 8 batch rows) when n_q <= 16, B >= 64, at least 8 shared keys, at
 * most 32 per-batch and 48 shared keys, every per-batch key's K and V have one bstride and bdiv, and the shared keys are all
 * batch-constant (bstride 0, bdiv 0) or all per-group with one common bdiv that is a multiple of 8; otherwise the per-row kernel.
 * ptr and out must be 16-byte aligned and bstride a multiple of 8 (bf16) or 4 (fp32) elements; M3PC_ERR_INVALID otherwise.
 * out_kernel: NULL, or HOST int32[4] that receives {kind, a, b, grid_x} of the launch: kind 0 = the fp32 kernel, 1 = the bf16
 * per-row kernel with a = ceil(n_q/16) query and b = ceil(n_kv/16) key tiles, 2 = the shared-key kernel with a per-batch and b
 * shared key tiles; grid_x < ceil(B/8) there means each CTA walked several blocks of 8 batch rows. */
int m3pc_attention_gather(const m3pc_attn_tok_t* q, int32_t n_q, const m3pc_attn_tok_t* k, const m3pc_attn_tok_t* v, int32_t n_kv,
                          int32_t n_kv_batch, int32_t B, int32_t n_head, void* out, int32_t is_bf16, int32_t* out_kernel, void* stream);

/* ---- the fused memory-bound kernels of the path, one entry each (SURVEY.md section 8b K1, K4..K8) ----
 * The activation layout these expose is the library's internal one: token-major matrices, row = token * batch + b, fp32
 * residual stream (x) and operands in the activation type of the handle (bf16 for M3PC_PREC_BF16, else fp32). */

/* K1 -- tokens -> encoder input: omtm.trajectory_encoding + the kept-token gather of forward_encoder (mtm_model.py:546-557,
 * :619-632) + norm1 of the first encoder block.  tok_*, masks as in m3pc_forward.  S = number of kept tokens (modality-major).
 *   x_out  device fp32 (S*batch, D): W_enc x + b + per-dim + pos[t] of every kept token
 *   y_out  device (S*batch, D) activation type: LayerNorm(x_out; encoder.layers.0.norm1) */
int m3pc_embed_gather(m3pc_handle_t h, int32_t batch, const float* tok_states, const float* tok_actions, const float* tok_rewards,
                      const float* tok_returns, const uint8_t* masks, float* x_out, void* y_out, void* stream);
/* K2 + K3 -- ONE pre-LN transformer block (nn.TransformerEncoderLayer(norm_first=True, activation="gelu"), built at
 * mtm_model.py:379-409, run by forward_encoder :619-644 / forward_decoder :698-706): x += MHA(LN1(x)); x += W2 gelu(W1 LN2(x) + b1) + b2.
 * The same launch sequence m3pc_forward uses for a block (QKV GEMM, attention, out-projection + residual + norm2, linear1 + GELU,
 * linear2 + residual + the LayerNorm that follows).
 *   stack   0 = encoder.layers[layer], 1 = decoder.layers[layer]
 *   x       device fp32 (n_tok*batch, D), token-major (row = token * batch + b): the residual stream, updated in place
 *   y_next  device (n_tok*batch, D) activation type or NULL: LayerNorm of the result by the NEXT block's norm1, or by the
 *           stack's final norm after its last layer (the operand the next block / the decoder embedding / K5 consumes)
 *   n_tok <= 4T (attention keys of one batch row), batch <= the engine's chunk, n_tok*batch <= 4T*chunk workspace rows. */
int m3pc_block_forward(m3pc_handle_t h, int32_t stack, int32_t layer, int32_t batch, int32_t n_tok, float* x, void* y_next, void* stream);
/* K4 -- encoder output -> decoder input: mask-token scatter + decoder_embed + per-dim + pos (mtm_model.py:646-696).
 *   enc_out device (S*batch, D) activation type: final-normed encoder output of the kept tokens, token-major
 *   x_out   device fp32 (4T*batch, D): row block j = decoder token j (modality-major, time-minor); masked tokens get the
 *           batch-constant row W_dec mask_token + b + per-dim + pos[t].  batch <= the engine's chunk. */
int m3pc_decoder_scatter_embed(m3pc_handle_t h, int32_t batch, const void* enc_out, const uint8_t* masks, float* x_out, void* stream);
/* K5 -- decoder block output -> predictions: final decoder norm, per-modality head LayerNorm -> Linear -> GELU -> Linear
 * (mtm_model.py:397-433, :708-714) and the DiagGaussianActor mu / std (mtm_model.py:313-321).
 *   x_dec device fp32 (4T*batch, D): residual stream after the last decoder block, BEFORE decoder.norm
 *   out_* as in m3pc_forward, (batch, T, d); any may be NULL.  batch <= the engine's chunk. */
int m3pc_heads(m3pc_handle_t h, int32_t batch, const float* x_dec, float* out_states, float* out_act_mu, float* out_act_std,
               float* out_rewards, float* out_returns, void* stream);
/* K6 -- candidate action sequences (finetune_omtm/learner.py:285-287, :156-167):
 *   noise_mode 0: cand[n,t,:] = tanh(mu[T-h+t] + std[T-h+t] * eps[n,t,:]);  1: clamp(tanh(mu[T-h+t]) + 0.09 eps[n,t,:], +-0.99999)
 *   mu, std device (T, A); eps device (n_cand, h, A) or NULL = Philox keyed by (seed, cand_offset + n); out (n_cand, h, A). */
int m3pc_sample_candidates(const float* mu, const float* std, const float* eps, uint64_t seed, int32_t n_cand, int32_t horizon, int32_t act_dim,
                           int32_t traj_length, int32_t noise_mode, int32_t cand_offset, float* out_candidates, void* stream);
/* K7 -- TwinQ on every (candidate, step): q[n*h + t] = min(Q1, Q2)((s_hat - obs_mean) / obs_std, a) with
 * s_hat = states_pred[n, T-h+t] * tok_std + tok_mean (finetune_omtm/learner.py:250-252, model.py:146-171).
 *   states_pred device (n_cand, T, obs) raw head output; candidates device (n_cand, h, A); out_q device (n_cand*h). */
int m3pc_twinq(m3pc_handle_t h, const float* states_pred, const float* candidates, int32_t n_cand, int32_t horizon, float* out_q, void* stream);
/* K8 -- TD(lambda) score + softmax selection (finetune_omtm/learner.py:301-325) of ONE shard of candidates:
 *   rewards_pred (n_cand, T) raw head output; exactly one of returns_pred (n_cand, T) [rtg_guiding: V_t = 1000 * return] and
 *   qvals (n_cand*h) [critic guidance]; candidates (n_cand, h, A); expq (n_cand) injected Exp(1) draws or NULL = Philox;
 *   norm_stats HOST float[4] = {rewards mean, rewards std, returns mean, returns std} of the tokenizers;
 *   out_J (n_cand); out_eval_action / out_sample_action (A); out_partials (M3PC_PARTIAL_FLOATS) or NULL; out_indices (2) or NULL. */
int m3pc_score_select(const float* rewards_pred, const float* returns_pred, const float* qvals, const float* candidates, const float* expq,
                      const float* norm_stats, float discount, float lmbda, float temperature, int32_t n_cand, int32_t horizon,
                      int32_t traj_length, int32_t act_dim, uint64_t seed, int32_t cand_offset, float* out_J, float* out_eval_action,
                      float* out_sample_action, float* out_partials, int32_t* out_indices, void* stream);

/* Device-side time (ms) spent between the first and last kernel of the most recent m3pc_plan / m3pc_forward
 * on this handle, measured with CUDA events on the caller's stream (valid after the stream is synchronised). */
int m3pc_last_device_ms(m3pc_handle_t h, float* ms);
/* Number of kernels the most recent m3pc_plan / m3pc_forward call launched. */
int m3pc_last_launch_count(m3pc_handle_t h, int32_t* n);

/* Profiling mode (off by default): when on, every tensor-core / fp32 GEMM launch of m3pc_plan / m3pc_forward /
 * m3pc_backward_plan is bracketed by its own CUDA event pair on the caller's stream.  m3pc_get_profile synchronises
 * those events and reports, for the most recent call: summed GEMM device time (ms), the algorithmic FLOPs those
 * launches executed (2*M*N*K each) and their count.  Used by bench.py for the live roofline numerator. */
int m3pc_set_profile(m3pc_handle_t h, int32_t on);
int m3pc_get_profile(m3pc_handle_t h, double* gemm_ms, double* gemm_flops, int32_t* gemm_launches);

#ifdef __cplusplus
}
#endif
#endif /* M3PC_H_ */
