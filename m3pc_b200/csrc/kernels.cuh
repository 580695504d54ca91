// Launcher declarations for the memory-bound fused kernels of the MTM forward and the M^3PC candidate loop.
#pragma once
#include "common.cuh"

namespace m3pc {

constexpr int MAX_TOK = 64;  // 4 * traj_length, traj_length <= 16

// ---- K1: tokenise + embed + positional/per-dim + unmasked gather (+ LayerNorm of the first block) -------
struct EmbedTok {
  const float* src;    // first element of this token's feature vector for batch row 0
  const float* wt;     // W_enc^T of the token's modality, (d, D) row-major
  const float* cvec;   // (D): bias + per-dim encoding + pos[t]
  const float* nmean;  // (d) tokenizer mean or nullptr (already tokenised / un-normalised modality)
  const float* nstd;   // (d)
  int bstride;         // floats between consecutive batch rows (0 = shared by all rows)
  int d;               // feature dim
  int bdiv;            // > 0: rows come in groups of bdiv consecutive GLOBAL batch rows (one group per environment) that share
                       // one source row; bstride is then the stride between groups (m3pc_plan with n_env > 1)
};
struct EmbedParams {
  EmbedTok tok[MAX_TOK];
  int n_tok;
  int B;
  int b0;   // global batch row of this chunk's row 0 (only read for tokens with bdiv > 0)
};
// x (n_tok*B, D) fp32 residual stream, y (n_tok*B, D) = LayerNorm(x; gamma, beta) in AT.
int launch_embed(const EmbedParams& p, int D, float* x, void* y, bool y_bf16, const float* gamma, const float* beta, cudaStream_t st);

// ---- fused B = 1 forward (fused_b1.cu): encoder + restricted single-layer decoder in one cooperative kernel -------
constexpr int FB_MAX_ROWS = 32;    // encoder tokens / needed decoder rows
constexpr int FB_MAX_LAYERS = 4;   // encoder layers
struct FusedLayer {
  const __nv_bfloat16 *in_w, *out_w, *l1_w, *l2_w;
  const float *in_b, *out_b, *l1_b, *l2_b, *n1_w, *n1_b, *n2_w, *n2_b;
};
struct FusedB1Params {
  int S, n_enc, T4, n_need;
  EmbedTok tok[FB_MAX_ROWS];             // encoder (kept) tokens, modality-major
  FusedLayer enc[FB_MAX_LAYERS];
  FusedLayer dec;
  const float *enc_norm_w, *enc_norm_b;  // final encoder norm
  const float *fnorm_w, *fnorm_b;        // final decoder norm
  const float* head_g[4];                // head LayerNorm per modality (null: actions, the actor reads the final norm)
  const float* head_b[4];
  const __nv_bfloat16* dec_w[4];         // decoder_embed weights per modality
  const float* dec_cvec;                 // (4T, D) bias + per-dim + pos
  const float* dec_maskrow;              // (4T, D) decoder input of a masked token
  const __nv_bfloat16* const_qkv;        // (4T, 3D) [Q | K | V] of the masked-token rows
  int mod_row0[5];                       // encoder rows of modality k: [mod_row0[k], mod_row0[k + 1])
  signed char dec_src[MAX_TOK];          // decoder token j -> encoder row, or -1 (masked)
  unsigned char enc_dectok[FB_MAX_ROWS]; // encoder row -> decoder token
  unsigned char need_tok[FB_MAX_ROWS];   // needed decoder tokens
  unsigned char need_mod[FB_MAX_ROWS];   // their modality
  // scratch (global; every buffer at least 32 rows)
  float* X;             // (S, D) encoder residual stream
  float* Xd;            // (S, D) decoder embedding of the kept tokens
  float* XS;            // (n_need, D) decoder residual stream of the needed rows
  __nv_bfloat16* QKV;   // (S, 3D)
  __nv_bfloat16* ATT;   // (max(S, n_need), D)
  __nv_bfloat16* HID;   // (max(S, n_need), 4D)
  // outputs
  __nv_bfloat16* Y;     // (n_need, D) final norm
  __nv_bfloat16* Y2;    // (n_need, D) head norm
  // optional fused actor head (DiagGaussianActor) for the needed action rows: out_mu / out_std are (T, A) of this batch row
  const float *mu_w, *mu_b, *ls_w, *ls_b;
  float *out_mu, *out_std;
  int act_dim;
  unsigned* bar;        // grid barrier state {count, generation}, zero-initialised once
};
size_t fused_b1_smem_bytes(int D, int S, int n_need);
int launch_fused_b1(const FusedB1Params& p, int D, cudaStream_t st);

// ---- LayerNorm family ---------------------------------------------------------------------------------
// y1 = LN(x; g1, b1) (optional), y2 = LN(y1; g2[grp], b2[grp]) (optional, grp = row / rows_per_group, skipped where g2[grp]==0)
struct LnParams {
  const float* x;
  int rows;
  const float* g1;
  const float* b1;
  void* y1;  // may be null
  const float* g2[4];
  const float* b2[4];
  int rows_per_group;            // rows per token block (B); the second LN's parameter set is tok_group[row / rows_per_group]
  unsigned char tok_group[MAX_TOK];
  void* y2;  // may be null
};
int launch_layernorm(const LnParams& p, int D, bool out_bf16, cudaStream_t st);

// ---- K4 helper: broadcast batch-constant decoder rows (mask tokens after decoder embedding) ------------
struct FillParams {
  const float* row[MAX_TOK];  // source row of batch row 0 for each listed token
  int bstride[MAX_TOK];       // floats between batch rows of the source (0 = one constant row broadcast to all)
  int tok[MAX_TOK];           // destination token index j (row block j*B .. j*B+B)
  int n;
  int B;
};
int launch_fill_rows(const FillParams& p, int D, float* x, cudaStream_t st);

// ---- K5: skinny output projections (512 -> d) ----------------------------------------------------------
// out[b, t, o] = dot(Y[(tok0 + t) * B + b, :], W[o, :]) + bias[o]     for t < n_t, o < d_out  (out is (B, T_out, d_out), t written at t + t_out0)
// actor mode: second weight set gives std = exp(-5 + 3.5 (tanh(.) + 1))   (DiagGaussianActor, mtm_model.py:313-321)
struct RowDotParams {
  const void* y;   // (rows, D) AT
  int B, tok0, n_t, t_out0, T_out, d_out;
  const float* w;   // (d_out, D)
  const float* b;   // (d_out)
  float* out;       // (B, T_out, d_out)
  const float* w2;  // actor log_std weights or null
  const float* b2;
  float* out2;      // std
};
int launch_rowdot(const RowDotParams& p, int D, bool y_bf16, cudaStream_t st);
constexpr int ROWDOT_MAX_JOBS = 4;
struct RowDotGroup {
  RowDotParams p[ROWDOT_MAX_JOBS];
  int block0[ROWDOT_MAX_JOBS];  // first block of each job
  int n;
};
// several projections (the heads of the consumed modalities) in one launch; per-row arithmetic as in launch_rowdot
int launch_rowdot_group(const RowDotParams* jobs, int n, int D, bool y_bf16, cudaStream_t st);

// ---- K3: small-sequence bidirectional attention ----------------------------------------------------------
// Token-gather form: every query / key / value token names its own source row block (row for batch b = ptr + b*bstride
// elements, bstride = 0 for rows shared by the whole batch: history tokens, batch-constant mask-token rows).
struct AttnTok {
  const void* ptr;
  int bstride;
  int bdiv;  // > 0: the row of batch row b is ptr + (b / bdiv) * bstride -- one row per group of bdiv batch rows (history tokens of
             // an environment, shared by all of its candidates); 0: ptr + b * bstride
};
struct AttnParams {
  AttnTok q[MAX_TOK], k[MAX_TOK], v[MAX_TOK];
  int n_q, n_kv, B, n_head;
  int n_kv_batch;  // > 0: keys [0, n_kv_batch) are per-batch rows and keys [n_kv_batch, n_kv) are shared by batch rows, all
                   // batch-constant (bstride 0) or all per-group with one bdiv; the bf16 kernel then stages them once per CTA instead
                   // of once per batch row (any other key list runs on the per-row kernel)
  void* out;  // (n_q * B, n_head * 128), row = query token * B + b
};
// launched: null, or int[4] that receives {kind, a, b, grid_x} of the kernel it launched (kind 0 = fp32 attention_kernel,
// 1 = attention_mma_kernel<a, b>, 2 = attention_mma_shared_kernel<a, b>)
int launch_attention_gather(const AttnParams& p, bool bf16, cudaStream_t st, int* launched = nullptr);
// self-attention over token-major qkv (S*B rows, [Q | K | V] columns)
int launch_attention(const void* qkv, void* out, int B, int S, int n_head, bool bf16, cudaStream_t st);

// ---- K6..K8: the candidate loop ---------------------------------------------------------------------------
struct CandParams {
  const float* mu;   // (T, A) action-head mu of pass 1 (B = 1)
  const float* std;  // (T, A)
  const float* eps;  // (N, h, A) injected noise or null (Philox)
  float* cand;       // (N, h, A)
  int N, h, A, T;
  int n_per_env;     // > 0: candidate n belongs to environment n / n_per_env and mu / std are (E, T, A)
  int noise_mode;    // 0: tanh(mu + std*eps) (learner.py:285-287); 1: clamp(tanh(mu) + 0.09*eps) (learner.py:156-167)
  unsigned long long seed;
  int cand_offset;
  const unsigned long long* seed_ptr;  // if non-null the Philox key is read from device memory (CUDA-graph replay)
  const int* env_id;  // (E) or null: device table local environment -> the caller's environment index.  Philox is then keyed by
                      // the caller's index (gid = env_id * n_per_env + n), so an environment's draws do not depend on which other
                      // environments share the call; null: gid = cand_offset + n
};
int launch_candidates(const CandParams& p, cudaStream_t st);

struct CriticInParams {
  const float* states_pred;  // (N, T, obs) raw head output (tokenised space)
  const float* cand;         // (N, h, A)
  const float* tok_mean;     // (obs) tokenizer stats of states
  const float* tok_std;
  const float* obs_mean;     // (obs) critic normaliser
  const float* obs_std;
  void* sa;                  // (N*h, ld), row = n*h + t: fp32 (ld = obs+A) or bf16 zero-padded to ld (tensor-core critic)
  int N, h, T, obs, A;
  int ld;
  int out_bf16;
};
int launch_critic_input(const CriticInParams& p, cudaStream_t st);
// q = min(h1 . w1 + b1, h2 . w2 + b2) per row; h1, h2 (rows, H) fp32
int launch_critic_out(const float* h1, const float* h2, const float* w1, const float* b1, const float* w2, const float* b2, float* q,
                      int rows, int H, cudaStream_t st);

struct ScoreParams {
  const float* rewards_pred;  // (N, T) raw head output
  const float* returns_pred;  // (N, T) raw head output (rtg_guiding) or null
  const float* qvals;         // (N*h) critic values or null
  float rw_mean, rw_std, rt_mean, rt_std;
  float discount, lmbda;
  int N, h, T;
  float* J;  // (N)
};
int launch_score(const ScoreParams& p, cudaStream_t st);

// Peer exchange of the per-shard records (candidate sharding over GPUs, SURVEY.md section 8e): every rank owns one buffer that
// ALL ranks can store into (peer-mapped over NVLink: CUDA IPC between processes, plain pointers inside one process):
//     float    rec [2][world][M3PC_PARTIAL_FLOATS]     record of rank g for plans of parity s at rec[s][g]
//     uint64   flag[2][world]                           epoch of the record that is complete in rec[s][g]
// The select kernel of rank r stores its record into slot [epoch & 1][r] of every rank's buffer (its own included), publishes
// it with a system-scope release store of the epoch, waits until all `world` flags of its own buffer show the epoch and merges
// the records -- ONE kernel does the selection, the all-gather and the merge; no NCCL launch, nothing outside the CUDA graph.
// Two slots suffice: a rank can only be one plan ahead of the slowest rank (it needs everybody's record to finish a plan).
constexpr int XCH_MAX_RANKS = 32;
constexpr size_t XCH_FLAG_OFFSET = sizeof(float) * 2 * XCH_MAX_RANKS * M3PC_PARTIAL_FLOATS;
constexpr size_t XCH_ERR_OFFSET = XCH_FLAG_OFFSET + sizeof(unsigned long long) * 2 * XCH_MAX_RANKS;  // uint64: epoch of a timed-out wait
constexpr size_t XCH_BYTES = XCH_ERR_OFFSET + 64;
struct ExchangeParams {
  void* peer[XCH_MAX_RANKS];      // exchange buffer of every rank, as addressable from THIS device
  int rank, world;                // world == 0: no exchange
  unsigned long long* epoch;      // device scalar of this handle: plans exchanged so far
  unsigned long long timeout_ns;  // give up (NaN actions, error word set) instead of spinning forever if a peer never arrives
};

// One thread block per environment e (grid = n_env): J, cand, expq are offset by e*N, the outputs by e*A (indices by 2e).
struct SelectParams {
  int n_env;          // >= 1
  const float* J;     // (N)
  const float* cand;  // (N, h, A): a0 = cand[n, 0, :]
  const float* expq;  // (N) or null
  int N, h, A;
  float temperature;
  unsigned long long seed;
  int cand_offset;
  const unsigned long long* seed_ptr;  // see CandParams
  float* eval_action;    // (A)
  float* sample_action;  // (A)
  float* partials;       // (M3PC_PARTIAL_FLOATS) or null
  int* indices;          // (2) or null
  ExchangeParams xch;    // xch.world > 0 (n_env == 1 only): exchange + merge inside the kernel; the outputs are the GLOBAL result
  ScoreParams score;     // score.J == J: the TD(lambda) scores are computed by this launch first (one launch less per plan); null J: not
  const int* env_id;     // (n_env) or null: as CandParams::env_id; the outputs of block e go to row env_id[e] (indices 2 env_id[e])
};
int launch_select(const SelectParams& p, cudaStream_t st);
int launch_merge(const float* partials, int n_shards, int A, float temperature, float* eval_action, float* sample_action, int* indices,
                 cudaStream_t st);

// mtm_sampling tail (learner.py:103-115): eval = tanh(mu[T-h]), sample = tanh(mu[T-h] + std[T-h]*eps)
// C > 1: C draws per environment, sample_action is (E, C, A) and eps (E, C, A)
// env_id (E) or null: as CandParams::env_id (Philox keyed by, and outputs written to, the caller's environment index)
// eps_at_env_id (needs env_id): eps is the caller's (E_caller, C, A) noise, read at the row of env_id[e] instead of row e
int launch_sampling_tail(const float* mu, const float* std, const float* eps, int T, int h, int A, int E, float* eval_action,
                         float* sample_action, unsigned long long seed, const unsigned long long* seed_ptr, cudaStream_t st, int C = 1,
                         const int* env_id = nullptr, bool eps_at_env_id = false);

// ---- m3pc_plan with one horizon per environment: the environments of one horizon class are planned as one uniform sub-plan on
// contiguous copies of their inputs.  One launch gathers every class at once (classes are disjoint, so nothing is overwritten
// while a later class runs).  The class order is a kernel parameter: a captured plan holds no host-to-device copy. ----
constexpr int MIX_MAX_ENV = 256;
struct MixGatherParams {
  const float *ws, *wa, *wr, *wt;  // caller windows (E, T, .)
  float *gs, *ga, *gr, *gt;        // gathered windows (E, T, .), gathered slot s = caller environment src[s]
  const float* eps;                // caller noise: eps_rows rows of eps_ld floats per environment, or null
  float* geps;                     // gathered noise: slot s keeps the first (eps_off[s+1]-eps_off[s]) / eps_rows floats of each row
  const float* expq;               // caller (E, N) or null
  float* gexpq;                    // gathered (E, N)
  int* env_id;                     // out (E): gathered slot -> caller environment (the sub-plans' id tables)
  int E, T, obs, A, N, eps_rows, eps_ld;
  short src[MIX_MAX_ENV];          // gathered slot -> caller environment
  short slot_of[MIX_MAX_ENV];      // caller environment -> gathered slot
  int eps_off[MIX_MAX_ENV + 1];    // first gathered noise float of each slot
};
int launch_mix_gather(const MixGatherParams& p, cudaStream_t st);
int launch_set_seed(unsigned long long* dst, unsigned long long seed, cudaStream_t st);

// zero-shot piid fill (zeroshot_omtm/learner.py:240-246): states[:, T-h+2:-1] and states[:, :T-h+1] <- decode(pred)
int launch_piid_fill(const float* win_states, const float* states_pred, const float* tok_mean, const float* tok_std, float* filled, int E,
                     int T, int h, int obs, cudaStream_t st);

// device-resident episode ring (include/m3pc.h: m3pc_ring_reset / m3pc_ring_append_slots / m3pc_ring_windows_slots): slots and
// horizons are host lists, t / path_length device (E) tables indexed by slot; per-slot inputs and outputs are in list order
int launch_ring_reset(float* ring, int E, int L, int obs, int act, const int* slots, int n, cudaStream_t st);
int launch_ring_append_slots(float* ring, int E, int L, int obs, int act, const int* t, const int* slots, int n, const float* o, const float* pa,
                             const float* pr, cudaStream_t st);
int launch_ring_write_obs(float* ring, int E, int L, int obs, int act, const int* slots, int n, int first, int n_rows, const float* rows,
                          cudaStream_t st);
int launch_ring_windows_slots(const float* ring, int E, int L, int obs, int act, const int* pl, const int* slots, const int* horizons, int n,
                              int T, int future_obs, const float* rtg_tok, float* ws, float* wa, float* wr, float* wt, cudaStream_t st);

// conversions
int launch_f32_to_bf16(const float* in, __nv_bfloat16* out, size_t n, cudaStream_t st);

}  // namespace m3pc
