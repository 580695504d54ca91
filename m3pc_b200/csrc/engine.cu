// Engine: the handle behind include/m3pc.h -- parameter packing, workspaces, and the launch sequences of
// omtm.forward (mtm_model.py:593-607) and of the M^3PC planners (finetune_omtm/learner.py:103-327,
// zeroshot_omtm/learner.py:60-261).  Host code only; every kernel lives in the sibling .cu files.
//
// HBM layout: all activations are token-major matrices, row = token * Bc + b for the Bc batch rows (candidates
// or environments) of the current chunk.  A chunk is run through the whole network before the next one starts,
// so its working set (<= ~80 bytes/feature/row) stays L2-resident; weights (22.7 MB bf16) stay L2-resident too.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "kernels.cuh"

namespace m3pc {

thread_local int g_launch_count = 0;
static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }

int device_num_sms() {
  static PerDevice<int> sms;
  int& n = sms.here();
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n = 0;
  }
  return n;
}

namespace {

const char* kMod[4] = {"states", "actions", "rewards", "returns"};

constexpr int TAB_ROWS = 4096;  // capacity (token x group rows) of the shared-history tables

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int alloc(size_t n) {
    free();
    if (n == 0) n = 16;
    M3PC_CHECK_CUDA(cudaMalloc(&p, n));
    bytes = n;
    return M3PC_OK;
  }
  void free() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  ~DevBuf() { free(); }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct LayerW {
  const float *in_w, *in_b, *out_w, *out_b, *l1_w, *l1_b, *l2_w, *l2_b, *n1_w, *n1_b, *n2_w, *n2_b;
  const __nv_bfloat16 *in_w16, *out_w16, *l1_w16, *l2_w16;
};
struct StackW {
  std::vector<LayerW> layers;
  const float *norm_w, *norm_b;
};

// source of one modality's tokens for the embedding kernel
struct ModSrc {
  const float* base = nullptr;  // token t of batch row b at base + b*bstride + t*d
  long bstride = 0;
  bool normalize = false;       // apply the tokenizer's (x-mean)/std
  const float* base2 = nullptr; // tokens t >= t_split come from base2 + b*bstride2 + (t-t_split)*d
  long bstride2 = 0;
  int t_split = 1 << 30;
  int bdiv = 0;                 // > 0: `base` rows are shared by groups of bdiv consecutive batch rows (row b reads
                                // base + (b / bdiv)*bstride + t*d): the E windows of an n_env > 1 plan
};

struct FwdIO {
  ModSrc src[4];
  uint8_t mask[4 * M3PC_MAX_T];
  float* out_states = nullptr;
  float* out_mu = nullptr;
  float* out_std = nullptr;
  float* out_rewards = nullptr;
  float* out_returns = nullptr;
  // time steps whose head outputs the caller consumes, per modality: [need_t0, need_t0 + need_nt); need_nt < 0 = all T.
  // Rows outside these ranges are never written (dead-row elimination in the last decoder layer).
  int need_t0[4] = {0, 0, 0, 0};
  int need_nt[4] = {-1, -1, -1, -1};
};

}  // namespace
}  // namespace m3pc

using namespace m3pc;

struct m3pc_engine {
  m3pc_config_t cfg{};
  int D = 0, H = 0, T = 0, F = 0, obs = 0, act = 0, Le = 0, Ld = 0, QH = 0;
  int dims[4] = {0, 0, 0, 0};
  bool bf16 = true;
  bool tf32x3 = false;  // M3PC_PREC_TF32X3: the fp32 mode with its contractions on the tensor cores (gemm_tf32x3)
  int chunk = 0;
  bool finalized = false;
  std::map<std::string, std::vector<float>> staged;

  DevBuf arena_f32, arena_bf16;  // packed parameters

  // derived device pointers
  const float* enc_wt[4] = {};    // W_enc^T (d, D)
  const float* enc_cvec = nullptr;  // (4, T, D) bias + perdim + pos
  const float* dec_cvec = nullptr;  // (4T, D)   bias + perdim + pos
  const float* dec_maskrow = nullptr;  // (4T, D) W_dec mask_token + dec_cvec
  const float* dec_w[4] = {};
  const __nv_bfloat16* dec_w16[4] = {};
  StackW enc, dec;
  const float *head_ln_w[4] = {}, *head_ln_b[4] = {}, *head_w1[4] = {}, *head_b1[4] = {}, *head_w3[4] = {}, *head_b3[4] = {};
  const __nv_bfloat16* head_w1_16[4] = {};
  const float *mu_w = nullptr, *mu_b = nullptr, *ls_w = nullptr, *ls_b = nullptr;
  const float *tok_mean[4] = {}, *tok_std[4] = {};
  float h_tok_mean[4] = {0, 0, 0, 0}, h_tok_std[4] = {1, 1, 1, 1};  // scalar modalities (rewards, returns) on host
  bool has_critic = false;
  const float *q_w[2][3] = {}, *q_b[2][3] = {}, *obs_mean = nullptr, *obs_std = nullptr;
  const __nv_bfloat16* q_w16[2][2] = {};  // bf16 copies of the two hidden layers (layer 0 zero-padded to q_kp inputs)
  int q_kp = 0;                            // critic input width padded to a multiple of 64 (tensor-core critic)
  bool critic_tc = false;

  // batch-constant decoder rows (single-layer decoder only): [Q | K | V] of LN1(decoder_embed(mask token) + per-dim + pos[t])
  // for every decoder token, (4T, 3D) in the activation type; independent of inputs and of the mask layout
  DevBuf const_qkv;

  // workspaces (per chunk)
  DevBuf X, XS, Y, Y2, QKV, QSEL, ATT, HID, ENC;
  DevBuf XT, YT, QKVT;  // shared-history tables of the first encoder block (TAB_ROWS rows)
  DevBuf fb_xd, fb_bar;  // fused B = 1 path: decoder-embedding scratch, grid-barrier state
  bool use_fused_b1 = true;
  int fuse_ln_min_rows = 1024;  // residual GEMM + LayerNorm in one kernel (gemm_ln.cu) from this many rows up; option "fused_ln_min_rows"
                                // (the kernel-level parity tests call the kernel at any size)
  bool restrict_deep = true;  // decoders with > 1 layer: last layer on the consumed rows only; option "restrict_deep_decoder"
  // planner buffers
  DevBuf p1_mu, p1_std, cand, pred_states, pred_rewards, pred_returns, sa, qa, qb1, qb2, qvals, J, filled, e_mu, e_std;
  // plans with one horizon per environment: every class's windows, noise rows and id table, gathered (launch_mix_gather)
  DevBuf mix_ws, mix_wa, mix_wr, mix_wt, mix_eps, mix_expq, mix_id;

  // CUDA-graph replay of m3pc_plan (production path: on-device Philox noise, no debug outputs)
  struct PlanKey {
    int guidance, horizon, n_cand, cand_offset, n_env, exchange;
    float discount, temperature, lmbda;
    const void *ws, *wa, *wr, *wt, *ev, *sm, *pt;
    unsigned char env_h[MIX_MAX_ENV];  // per-environment horizons of a mixed plan (all zero otherwise)
    bool operator<(const PlanKey& o) const { return std::memcmp(this, &o, sizeof(PlanKey)) < 0; }
  };
  struct PlanGraph {
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
    int seen = 0;  // eager calls before capture (lazy one-time initialisation must not happen inside a capture)
  };
  std::map<PlanKey, PlanGraph> plan_graphs;
  bool use_graphs = true;
  DevBuf seed_scalar;
  const unsigned long long* seed_ptr_active = nullptr;  // non-null while (re)building / replaying a graph

  // peer exchange of per-shard records (candidate sharding over GPUs; kernels.cuh ExchangeParams)
  DevBuf xch_buf, xch_epoch;
  void* xch_peer[XCH_MAX_RANKS] = {};
  std::vector<void*> xch_opened;  // cudaIpcOpenMemHandle'd peers (closed in the destructor)
  int xch_rank = 0, xch_world = 0;

  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaStream_t cap_stream = nullptr;  // private stream the plan graphs are captured on
  int last_launches = 0;
  // profiling mode: one event pair per GEMM launch
  bool profile = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
  std::vector<double> prof_flops;
  size_t prof_used = 0;

  // Every captured plan has the weight / tokenizer / critic arena addresses and the scalar statistics baked into its kernel
  // nodes: whenever any of those may change (m3pc_set_param, m3pc_finalize_params, m3pc_set_option) the graphs are dropped
  // and the next plan re-captures.
  void drop_graphs() {
    for (auto& kv : plan_graphs)
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    plan_graphs.clear();
  }

  ~m3pc_engine() {
    drop_graphs();
    for (void* q : xch_opened) cudaIpcCloseMemHandle(q);
    if (cap_stream) cudaStreamDestroy(cap_stream);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    for (auto& pr : prof_events) {
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
  }
};

namespace m3pc {
namespace {

size_t act_bytes(const m3pc_engine* e) { return e->bf16 ? 2 : 4; }

// ------------------------------------------------------------------------------------------------ params
int need(m3pc_engine* e, const std::string& name, size_t count, const std::vector<float>** out) {
  auto it = e->staged.find(name);
  if (it == e->staged.end()) {
    set_error("missing parameter '" + name + "'");
    return M3PC_ERR_STATE;
  }
  if (it->second.size() != count) {
    set_error("parameter '" + name + "' has " + std::to_string(it->second.size()) + " values, expected " + std::to_string(count));
    return M3PC_ERR_INVALID;
  }
  *out = &it->second;
  return M3PC_OK;
}

// Lays the parameters out in the fp32 arena and (bf16 mode) the bf16 arena, and records for every tensor the engine field that
// receives its device pointer; finalize() writes those fields once the arenas are uploaded.
struct Packer {
  bool bf16 = false;  // bf16 mode: tensors given a bf16 slot also get a bf16 copy
  std::vector<float> f32;
  struct Slot { size_t off; const float** p; };
  struct Slot16 { size_t src, n, off; const __nv_bfloat16** p; };  // bf16 copy of f32[src, src + n) at element `off`
  std::vector<Slot> slots;
  std::vector<Slot16> slots16;
  size_t n16 = 0;
  void add(const float* data, size_t n, const float** slot, const __nv_bfloat16** slot16 = nullptr) {
    // 64-float (256 B) alignment keeps every tensor TMA/float4 friendly
    while (f32.size() % 64) f32.push_back(0.f);
    const size_t o = f32.size();
    f32.insert(f32.end(), data, data + n);
    if (slot != nullptr) slots.push_back({o, slot});
    if (bf16 && slot16 != nullptr) {
      while (n16 % 128) ++n16;
      slots16.push_back({o, n, n16, slot16});
      n16 += n;
    }
  }
};

// packs the staged parameter `name` of `n` values
int pack(m3pc_engine* e, Packer& pk, const std::string& name, size_t n, const float** slot, const __nv_bfloat16** slot16 = nullptr) {
  const std::vector<float>* v;
  M3PC_TRY(need(e, name, n, &v));
  pk.add(v->data(), n, slot, slot16);
  return M3PC_OK;
}

int pack_stack(m3pc_engine* e, Packer& pk, StackW& s, const std::string& prefix, int n_layer) {
  const size_t D = e->D, F = e->F;
  s.layers.resize(n_layer);  // before packing: the slots point into it
  for (int l = 0; l < n_layer; ++l) {
    const std::string p = prefix + ".layers." + std::to_string(l);
    LayerW& w = s.layers[l];
    struct Item { const char* suffix; size_t n; const float** slot; const __nv_bfloat16** slot16; } items[] = {
        {".self_attn.in_proj_weight", 3 * D * D, &w.in_w, &w.in_w16}, {".self_attn.in_proj_bias", 3 * D, &w.in_b, nullptr},
        {".self_attn.out_proj.weight", D * D, &w.out_w, &w.out_w16},   {".self_attn.out_proj.bias", D, &w.out_b, nullptr},
        {".linear1.weight", F * D, &w.l1_w, &w.l1_w16},                {".linear1.bias", F, &w.l1_b, nullptr},
        {".linear2.weight", D * F, &w.l2_w, &w.l2_w16},                {".linear2.bias", D, &w.l2_b, nullptr},
        {".norm1.weight", D, &w.n1_w, nullptr},                        {".norm1.bias", D, &w.n1_b, nullptr},
        {".norm2.weight", D, &w.n2_w, nullptr},                        {".norm2.bias", D, &w.n2_b, nullptr}};
    for (auto& it : items) M3PC_TRY(pack(e, pk, p + it.suffix, it.n, it.slot, it.slot16));
  }
  M3PC_TRY(pack(e, pk, prefix + ".norm.weight", D, &s.norm_w));
  return pack(e, pk, prefix + ".norm.bias", D, &s.norm_b);
}

int build_const_rows(m3pc_engine* e);

int finalize(m3pc_engine* e) {
  const size_t D = e->D, T = e->T;
  // the arenas are about to be freed and re-allocated: no graph captured against the old addresses may survive, and no
  // kernel still reading them may be in flight
  M3PC_CHECK_CUDA(cudaDeviceSynchronize());
  e->drop_graphs();
  Packer pk;
  pk.bf16 = e->bf16;
  const std::vector<float>* v;
  const std::vector<float>* pos;
  M3PC_TRY(need(e, "pos_embed", T * D, &pos));

  std::vector<float> enc_cvec(4 * T * D), dec_cvec(4 * T * D), dec_maskrow(4 * T * D);
  for (int k = 0; k < 4; ++k) {
    const size_t d = e->dims[k];
    const std::string m = kMod[k];
    const std::vector<float>*ew, *eb, *epd, *dw, *db, *dpd, *mt;
    M3PC_TRY(need(e, "encoder_embed_dict." + m + ".weight", D * d, &ew));
    M3PC_TRY(need(e, "encoder_embed_dict." + m + ".bias", D, &eb));
    M3PC_TRY(need(e, "encoder_per_dim_encoding." + m, D, &epd));
    M3PC_TRY(need(e, "decoder_embed_dict." + m + ".weight", D * D, &dw));
    M3PC_TRY(need(e, "decoder_embed_dict." + m + ".bias", D, &db));
    M3PC_TRY(need(e, "decoder_per_dim_encoding." + m, D, &dpd));
    M3PC_TRY(need(e, "mask_token_dict." + m, D, &mt));
    // W_enc^T (d, D): lanes of the embedding kernel read it coalesced along D
    std::vector<float> wt(d * D);
    for (size_t c = 0; c < D; ++c)
      for (size_t i = 0; i < d; ++i) wt[i * D + c] = (*ew)[c * d + i];
    pk.add(wt.data(), wt.size(), &e->enc_wt[k]);
    pk.add(dw->data(), D * D, &e->dec_w[k], &e->dec_w16[k]);
    // W_dec mask_token (fp64 accumulate, rounded once)
    std::vector<float> wm(D);
    for (size_t c = 0; c < D; ++c) {
      double s = 0.0;
      for (size_t i = 0; i < D; ++i) s += static_cast<double>((*dw)[c * D + i]) * static_cast<double>((*mt)[i]);
      wm[c] = static_cast<float>(s);
    }
    for (size_t t = 0; t < T; ++t)
      for (size_t c = 0; c < D; ++c) {
        const size_t o = (k * T + t) * D + c;
        enc_cvec[o] = ((*eb)[c] + (*epd)[c]) + (*pos)[t * D + c];
        dec_cvec[o] = ((*db)[c] + (*dpd)[c]) + (*pos)[t * D + c];
        dec_maskrow[o] = ((wm[c] + (*db)[c]) + (*dpd)[c]) + (*pos)[t * D + c];
      }
  }
  pk.add(enc_cvec.data(), enc_cvec.size(), &e->enc_cvec);
  pk.add(dec_cvec.data(), dec_cvec.size(), &e->dec_cvec);
  pk.add(dec_maskrow.data(), dec_maskrow.size(), &e->dec_maskrow);
  M3PC_TRY(pack_stack(e, pk, e->enc, "encoder", e->Le));
  M3PC_TRY(pack_stack(e, pk, e->dec, "decoder", e->Ld));
  for (int k = 0; k < 4; ++k) {
    const std::string m = kMod[k];
    const size_t d = e->dims[k];
    if (k == M3PC_ACTIONS) {
      M3PC_TRY(pack(e, pk, "output_head_dict.actions.mu.weight", d * D, &e->mu_w));
      M3PC_TRY(pack(e, pk, "output_head_dict.actions.mu.bias", d, &e->mu_b));
      M3PC_TRY(pack(e, pk, "output_head_dict.actions.log_std.weight", d * D, &e->ls_w));
      M3PC_TRY(pack(e, pk, "output_head_dict.actions.log_std.bias", d, &e->ls_b));
    } else {
      const std::string p = "output_head_dict." + m;
      M3PC_TRY(pack(e, pk, p + ".0.weight", D, &e->head_ln_w[k]));
      M3PC_TRY(pack(e, pk, p + ".0.bias", D, &e->head_ln_b[k]));
      M3PC_TRY(pack(e, pk, p + ".1.weight", D * D, &e->head_w1[k], &e->head_w1_16[k]));
      M3PC_TRY(pack(e, pk, p + ".1.bias", D, &e->head_b1[k]));
      M3PC_TRY(pack(e, pk, p + ".3.weight", d * D, &e->head_w3[k]));
      M3PC_TRY(pack(e, pk, p + ".3.bias", d, &e->head_b3[k]));
      // tokenizer statistics (decode needs them for all three; encode for states/rewards)
      M3PC_TRY(need(e, "tokenizer." + m + ".mean", d, &v));
      pk.add(v->data(), d, &e->tok_mean[k]);
      if (d == 1) e->h_tok_mean[k] = (*v)[0];
      M3PC_TRY(need(e, "tokenizer." + m + ".std", d, &v));
      pk.add(v->data(), d, &e->tok_std[k]);
      if (d == 1) e->h_tok_std[k] = (*v)[0];
    }
  }
  e->has_critic = false;
  if (e->QH > 0 && e->staged.count("critic.q1.net.0.weight")) {
    const size_t in = e->obs + e->act, Hq = e->QH;
    e->q_kp = static_cast<int>((in + 63) / 64 * 64);
    e->critic_tc = e->bf16 && Hq % 128 == 0;
    const size_t wn[3] = {Hq * in, Hq * Hq, Hq}, bn[3] = {Hq, Hq, 1};
    for (int q = 0; q < 2; ++q)
      for (int l = 0; l < 3; ++l) {
        const std::string p = "critic.q" + std::to_string(q + 1) + ".net." + std::to_string(2 * l);
        M3PC_TRY(need(e, p + ".weight", wn[l], &v));
        pk.add(v->data(), wn[l], &e->q_w[q][l], l == 1 && e->critic_tc ? &e->q_w16[q][1] : nullptr);
        if (l == 0 && e->critic_tc) {  // zero-pad the input dimension to a TMA/UMMA friendly multiple of 64
          std::vector<float> wp(Hq * e->q_kp, 0.f);
          for (size_t r = 0; r < Hq; ++r)
            for (size_t c = 0; c < in; ++c) wp[r * e->q_kp + c] = (*v)[r * in + c];
          pk.add(wp.data(), wp.size(), nullptr, &e->q_w16[q][0]);
        }
        M3PC_TRY(pack(e, pk, p + ".bias", bn[l], &e->q_b[q][l]));
      }
    M3PC_TRY(pack(e, pk, "critic.obs_mean", e->obs, &e->obs_mean));
    M3PC_TRY(pack(e, pk, "critic.obs_std", e->obs, &e->obs_std));
    e->has_critic = true;
  }

  // upload, then point every slot into the arenas
  M3PC_TRY(e->arena_f32.alloc(pk.f32.size() * sizeof(float)));
  M3PC_CHECK_CUDA(cudaMemcpy(e->arena_f32.p, pk.f32.data(), pk.f32.size() * sizeof(float), cudaMemcpyHostToDevice));
  for (const Packer::Slot& s : pk.slots) *s.p = e->arena_f32.as<float>() + s.off;
  if (e->bf16) {
    M3PC_TRY(e->arena_bf16.alloc((pk.n16 + 128) * sizeof(__nv_bfloat16)));
    M3PC_CHECK_CUDA(cudaMemset(e->arena_bf16.p, 0, e->arena_bf16.bytes));
    for (const Packer::Slot16& s : pk.slots16) {
      M3PC_TRY(launch_f32_to_bf16(e->arena_f32.as<float>() + s.src, e->arena_bf16.as<__nv_bfloat16>() + s.off, s.n, 0));
      *s.p = e->arena_bf16.as<__nv_bfloat16>() + s.off;
    }
    M3PC_CHECK_CUDA(cudaDeviceSynchronize());
  }
  e->finalized = true;  // `staged` is kept: a later m3pc_set_param of a subset + finalize re-packs (include/m3pc.h)
  if (e->Ld == 1) M3PC_TRY(build_const_rows(e));
  return M3PC_OK;
}

// ------------------------------------------------------------------------------------------------ forward
int gemm(m3pc_engine* e, const void* A, const float* w32, const __nv_bfloat16* w16, void* C, int M, int N, int K, const GemmEpilogue& epi,
         cudaStream_t st);

// y = LayerNorm(x; gamma, beta) on `rows` rows of D features, y in bf16 or fp32
int layernorm(const float* x, int rows, const float* gamma, const float* beta, void* y, int D, bool y_bf16, cudaStream_t st) {
  LnParams ln{};
  ln.x = x;
  ln.rows = rows;
  ln.rows_per_group = 1;
  ln.g1 = gamma;
  ln.b1 = beta;
  ln.y1 = y;
  return launch_layernorm(ln, D, y_bf16, st);
}

// Batch-constant decoder rows.  With a single decoder layer, a masked token's decoder input is the same vector for every
// batch row: decoder_embed(mask_token) + per-dim + pos[t] (dec_maskrow, mtm_model.py:646-696).  Its LayerNorm and its Q / K / V
// projections are therefore constants of the weights: computed once here, with the same kernels the per-batch rows use.
int build_const_rows(m3pc_engine* e) {
  const int D = e->D, rows = 4 * e->T;
  const LayerW& w = e->dec.layers[0];
  M3PC_TRY(layernorm(e->dec_maskrow, rows, w.n1_w, w.n1_b, e->Y.p, D, e->bf16, 0));
  GemmEpilogue ge;
  ge.bias = w.in_b;
  M3PC_TRY(gemm(e, e->Y.p, w.in_w, w.in_w16, e->const_qkv.p, rows, 3 * D, D, ge, 0));
  M3PC_CHECK_CUDA(cudaDeviceSynchronize());
  return M3PC_OK;
}

// Runs `launch` (one GEMM-family launch); with profiling on (m3pc_set_profile) it is bracketed by an event pair and `flops`
// are booked against it for m3pc_get_profile.
template <typename Launch>
int profiled(m3pc_engine* e, double flops, cudaStream_t st, Launch&& launch) {
  if (!e->profile) return launch();
  const size_t slot = e->prof_used++;
  if (slot >= e->prof_events.size()) {
    cudaEvent_t a, b;
    M3PC_CHECK_CUDA(cudaEventCreate(&a));
    M3PC_CHECK_CUDA(cudaEventCreate(&b));
    e->prof_events.push_back({a, b});
    e->prof_flops.push_back(0.0);
  }
  e->prof_flops[slot] = flops;
  M3PC_CHECK_CUDA(cudaEventRecord(e->prof_events[slot].first, st));
  M3PC_TRY(launch());
  M3PC_CHECK_CUDA(cudaEventRecord(e->prof_events[slot].second, st));
  return M3PC_OK;
}

// C = epilogue(A W^T) on fp32 operands, with the kernel the precision mode runs fp32 contractions on: the 3xTF32 tensor-core kernel
// in tf32x3 mode, the CUDA-core kernel otherwise (fp32 mode; the fp32 critic layers of bf16 mode, when its width is not a multiple
// of 128).
int gemm_f32(const m3pc_engine* e, const float* A, const float* W, float* C, int M, int N, int K, const GemmEpilogue& epi, cudaStream_t st) {
  return e->tf32x3 ? gemm_tf32x3(A, W, C, M, N, K, epi, st) : gemm_fp32(A, W, C, M, N, K, epi, st);
}

// Independent GEMMs C = epilogue(A W^T) on activations of the mode's type, with the weights in both precisions.  bf16 mode:
// kMaxGroup at a time, each such group one launch of the CTA-pair tensor-core kernel where it applies (gemm_bf16) and booked as one
// profile entry; fp32 and tf32x3 modes: one launch each (gemm_f32).
struct GemmJob {
  const void* A;
  const float* w32;
  const __nv_bfloat16* w16;
  void* C;
  int M, N, K;
  GemmEpilogue epi;
};
int gemm_group(m3pc_engine* e, const GemmJob* jobs, int n, cudaStream_t st) {
  const int group = e->bf16 ? kMaxGroup : 1;
  for (int i0 = 0; i0 < n; i0 += group) {
    const int m = std::min(group, n - i0);
    GemmProblem pr[kMaxGroup];
    double flops = 0.0;
    for (int i = 0; i < m; ++i) {
      const GemmJob& j = jobs[i0 + i];
      pr[i] = GemmProblem{reinterpret_cast<const __nv_bfloat16*>(j.A), j.w16, j.C, j.M, j.N, j.K, j.epi};
      flops += 2.0 * j.M * static_cast<double>(j.N) * j.K;
    }
    const GemmJob& j = jobs[i0];
    M3PC_TRY(profiled(e, flops, st, [&] {
      return e->bf16 ? gemm_bf16(pr, m, st)
                     : gemm_f32(e, reinterpret_cast<const float*>(j.A), j.w32, reinterpret_cast<float*>(j.C), j.M, j.N, j.K, j.epi, st);
    }));
  }
  return M3PC_OK;
}

int gemm(m3pc_engine* e, const void* A, const float* w32, const __nv_bfloat16* w16, void* C, int M, int N, int K, const GemmEpilogue& epi,
         cudaStream_t st) {
  const GemmJob job{A, w32, w16, C, M, N, K, epi};
  return gemm_group(e, &job, 1, st);
}

// Whether the residual GEMM + LayerNorm of `rows` rows runs as ONE tensor-core kernel whose epilogue owns whole rows (gemm_ln.cu):
// bf16 mode, n_embd 512, and one CTA pair per 256 rows -- not for the few hundred rows of pass 1 of a multi-environment plan,
// where a single pair would do the work of 4 .. 16.  (The switch is kept well below any pass-2 chunk or candidate shard, so the
// kernel choice -- and with it the bit pattern of the scores -- does not depend on how candidates are chunked or sharded.)
// Which rows decide: a problem of its own decides on its own rows (a block, an MLP half, each part of the shared-history block);
// the decoder embedding's runs of kept tokens fuse only when every run is large enough; the restricted decoder layer's runs, which
// only split its needed rows by where their residual comes from, decide on their total: the fused kernel gives every row the same
// bits whether those rows run as one problem or as one per residual source.
bool fuse_ln(const m3pc_engine* e, int rows) { return e->bf16 && e->D == 512 && rows >= e->fuse_ln_min_rows; }

// X = R + A W^T + bias, Y = LayerNorm(X; g, b), with the residual R = X itself (in place), table[row / rpg] (`table`) or the fp32
// rows `res_src`
struct ResLnJob {
  const void* A;
  const float* w32;
  const __nv_bfloat16* w16;
  float* X;
  void* Y;
  const float* table;
  int rpg;
  int M;
  const float* res_src;
};

// `n` residual GEMM + LayerNorm jobs that share K, bias and the LayerNorm parameters.  `fused` (fuse_ln): the fused kernel, up to
// kMaxGroup jobs per launch (the ~10 us fixed cost of a launch is paid once per group).  Otherwise one grouped GEMM over all jobs,
// each residual added in its epilogue as (A W^T + bias) + R -- the same sum for an in-place residual and a row table -- and one
// LayerNorm launch over the jobs' rows, which therefore must tile one row range of X and of Y in order.
int gemm_res_ln(m3pc_engine* e, const ResLnJob* jobs, int n, const float* bias, const float* g, const float* b, int K, bool fused,
                cudaStream_t st) {
  const int D = e->D;
  M3PC_REQUIRE(n >= 1 && n <= MAX_TOK, "gemm_res_ln: 1 .. MAX_TOK jobs");
  if (!fused) {
    const size_t ab = act_bytes(e);
    GemmJob gj[MAX_TOK];
    int rows = 0;
    for (int i = 0; i < n; ++i) {
      const ResLnJob& j = jobs[i];
      M3PC_REQUIRE(j.X == jobs[0].X + static_cast<size_t>(rows) * D &&
                       static_cast<char*>(j.Y) == static_cast<char*>(jobs[0].Y) + static_cast<size_t>(rows) * D * ab,
                   "gemm_res_ln: the jobs must tile one row range of X and of Y in order");
      GemmEpilogue ep;
      ep.bias = bias;
      if (j.table != nullptr || j.res_src != nullptr) {
        ep.table = j.table != nullptr ? j.table : j.res_src;
        ep.rows_per_group = j.table != nullptr ? j.rpg : 1;
        ep.flags = EPI_OUT_F32 | EPI_ROWTABLE;
      } else {
        ep.flags = EPI_RESIDUAL;
      }
      gj[i] = GemmJob{j.A, j.w32, j.w16, j.X, j.M, D, K, ep};
      rows += j.M;
    }
    M3PC_TRY(gemm_group(e, gj, n, st));
    return layernorm(jobs[0].X, rows, g, b, jobs[0].Y, D, e->bf16, st);
  }
  for (int i0 = 0; i0 < n; i0 += kMaxGroup) {
    const int m = std::min(kMaxGroup, n - i0);
    LnJob lj[kMaxGroup];
    double flops = 0.0;
    for (int i = 0; i < m; ++i) {
      const ResLnJob& j = jobs[i0 + i];
      lj[i] = LnJob{reinterpret_cast<const __nv_bfloat16*>(j.A), j.w16, j.X, reinterpret_cast<__nv_bfloat16*>(j.Y), j.table, j.rpg, j.M, j.res_src};
      flops += 2.0 * j.M * static_cast<double>(D) * K;
    }
    M3PC_TRY(profiled(e, flops, st, [&] { return gemm_ln_bf16_grouped(lj, m, bias, g, b, K, st); }));
  }
  return M3PC_OK;
}

// LayerNorm applied to the residual stream right after a block: the next block's norm1 or a stack's final norm
struct PostLn {
  const float* g = nullptr;
  const float* b = nullptr;
  void* y = nullptr;
};

// second half of a pre-LN transformer block on `rows` token-major rows: expects Y = LN2(X); X += MLP(Y); then `post` (optional)
int mlp_half(m3pc_engine* e, const LayerW& w, int rows, cudaStream_t st, const PostLn& post) {
  const int D = e->D, F = e->F;
  GemmEpilogue ep;
  ep.bias = w.l1_b;
  ep.flags = EPI_GELU;
  M3PC_TRY(gemm(e, e->Y.p, w.l1_w, w.l1_w16, e->HID.p, rows, F, D, ep, st));
  if (post.y != nullptr) {
    const ResLnJob l2{e->HID.p, w.l2_w, w.l2_w16, e->X.as<float>(), post.y, nullptr, 1, rows, nullptr};
    return gemm_res_ln(e, &l2, 1, w.l2_b, post.g, post.b, F, fuse_ln(e, rows), st);
  }
  ep = GemmEpilogue{};
  ep.bias = w.l2_b;
  ep.flags = EPI_RESIDUAL;
  return gemm(e, e->HID.p, w.l2_w, w.l2_w16, e->X.p, rows, D, F, ep, st);
}

// one pre-LN transformer block on `rows` = S * Bc token-major rows; expects Y = LN1(X) on entry
int block(m3pc_engine* e, const LayerW& w, int Bc, int S, cudaStream_t st, const PostLn& post = PostLn{}) {
  const int D = e->D, rows = S * Bc;
  GemmEpilogue ep;
  ep.bias = w.in_b;
  M3PC_TRY(gemm(e, e->Y.p, w.in_w, w.in_w16, e->QKV.p, rows, 3 * D, D, ep, st));
  M3PC_TRY(launch_attention(e->QKV.p, e->ATT.p, Bc, S, e->H, e->bf16, st));
  const ResLnJob outp{e->ATT.p, w.out_w, w.out_w16, e->X.as<float>(), e->Y.p, nullptr, 1, rows, nullptr};
  M3PC_TRY(gemm_res_ln(e, &outp, 1, w.out_b, w.n2_w, w.n2_b, D, fuse_ln(e, rows), st));
  return mlp_half(e, w, rows, st, post);
}

// First encoder block when the first `n_sh` tokens are history tokens shared by groups of `grp` batch rows (the candidates of
// one environment): their embedding, LayerNorm and Q / K / V are computed once per group (tables XT / YT / QKVT, row =
// token * nG + group) instead of once per candidate.  The attention output differs per candidate, so from the
// out-projection on every row exists; for the shared tokens the residual is the table row, added in the epilogue.
// Expects: XT / YT = embedding / LN1 of the shared tokens, X / Y rows [n_sh*Bc, S*Bc) = the per-candidate tokens.
int block_shared_history(m3pc_engine* e, const LayerW& w, int Bc, int S, int n_sh, int grp, cudaStream_t st, const PostLn& post) {
  const int D = e->D, nG = Bc / grp;
  const size_t ab = act_bytes(e);
  const size_t off = static_cast<size_t>(n_sh) * Bc;  // first per-candidate row
  GemmJob qkv[2];
  GemmEpilogue ep;
  ep.bias = w.in_b;
  qkv[0] = GemmJob{e->YT.p, w.in_w, w.in_w16, e->QKVT.p, n_sh * nG, 3 * D, D, ep};
  qkv[1] = GemmJob{reinterpret_cast<const char*>(e->Y.p) + off * D * ab, w.in_w, w.in_w16, reinterpret_cast<char*>(e->QKV.p) + off * 3 * D * ab,
                   (S - n_sh) * Bc, 3 * D, D, ep};
  M3PC_TRY(gemm_group(e, qkv, 2, st));
  AttnParams ap{};
  ap.n_q = ap.n_kv = S;
  ap.B = Bc;
  ap.n_head = e->H;
  ap.out = e->ATT.p;
  // queries in token order (the output row block is the query's token); keys / values with the per-candidate tokens first and the
  // shared history tokens after them, which lets the bf16 kernel stage the shared ones once per CTA
  auto tok = [&](int s, int part) {
    const bool sh = s < n_sh;
    const char* row = sh ? reinterpret_cast<const char*>(e->QKVT.p) + static_cast<size_t>(s) * nG * 3 * D * ab
                         : reinterpret_cast<const char*>(e->QKV.p) + static_cast<size_t>(s) * Bc * 3 * D * ab;
    return AttnTok{row + static_cast<size_t>(part) * D * ab, 3 * D, sh ? grp : 0};
  };
  for (int s = 0; s < S; ++s) ap.q[s] = tok(s, 0);
  int nk = 0;
  for (int s = n_sh; s < S; ++s, ++nk) { ap.k[nk] = tok(s, 1); ap.v[nk] = tok(s, 2); }
  ap.n_kv_batch = nk;
  for (int s = 0; s < n_sh; ++s, ++nk) { ap.k[nk] = tok(s, 1); ap.v[nk] = tok(s, 2); }
  M3PC_TRY(launch_attention_gather(ap, e->bf16, st));
  // out-projection + norm2.  Shared tokens: X = table[token, group] + att W^T + b (row / grp = token * nG + group);
  // per-candidate tokens: X += att W^T + b.
  const ResLnJob outp[2] = {
      {e->ATT.p, w.out_w, w.out_w16, e->X.as<float>(), e->Y.p, e->XT.as<float>(), grp, static_cast<int>(off), nullptr},
      {reinterpret_cast<const char*>(e->ATT.p) + off * D * ab, w.out_w, w.out_w16, e->X.as<float>() + off * D, reinterpret_cast<char*>(e->Y.p) + off * D * ab,
       nullptr, 1, (S - n_sh) * Bc, nullptr}};
  const bool fused[2] = {fuse_ln(e, outp[0].M), fuse_ln(e, outp[1].M)};
  if (fused[0] == fused[1]) {
    M3PC_TRY(gemm_res_ln(e, outp, 2, w.out_b, w.n2_w, w.n2_b, D, fused[0], st));
  } else {
    for (int i = 0; i < 2; ++i) M3PC_TRY(gemm_res_ln(e, &outp[i], 1, w.out_b, w.n2_w, w.n2_b, D, fused[i], st));
  }
  return mlp_half(e, w, S * Bc, st, post);
}

struct NeedSet {
  int n = 0;
  int tok[MAX_TOK];  // needed decoder tokens (k*T + t), modality-major
  int q0[4] = {0, 0, 0, 0};  // first index in tok[] of each modality
  int t0[4] = {0, 0, 0, 0}, nt[4] = {0, 0, 0, 0};
};

// Calls fn(j, k, len) for every run of kept tokens of one modality k: decoder tokens j .. j+len-1, whose encoder rows
// dec_src[j] .. dec_src[j]+len-1 are consecutive too.
template <typename Fn>
void for_each_kept_run(const int* dec_src, int T, Fn&& fn) {
  for (int j = 0; j < 4 * T;) {
    if (dec_src[j] < 0) { ++j; continue; }
    const int k = j / T;
    int len = 1;
    while (j + len < (k + 1) * T && dec_src[j + len] == dec_src[j] + len) ++len;
    fn(j, k, len);
    j += len;
  }
}

// the masked decoder tokens of a layout, each broadcast from its batch-constant row dec_maskrow[j] into row block j
FillParams mask_rows(const m3pc_engine* e, const int* dec_src, int Bc) {
  FillParams fp{};
  fp.B = Bc;
  for (int j = 0; j < 4 * e->T; ++j)
    if (dec_src[j] < 0) {
      fp.row[fp.n] = e->dec_maskrow + static_cast<size_t>(j) * e->D;
      fp.bstride[fp.n] = 0;
      fp.tok[fp.n] = j;
      ++fp.n;
    }
  return fp;
}

// decoder_embed of the encoder outputs: one grouped GEMM per run of kept tokens of one modality (mtm_model.py:646-661), rows in
// decoder order (row block = decoder token j).
int decoder_embed(m3pc_engine* e, const void* enc_out, const int* dec_src, int Bc, cudaStream_t st, float* xout = nullptr) {
  const int D = e->D;
  const size_t ab = act_bytes(e);
  GemmJob jobs[MAX_TOK];
  int n = 0;
  for_each_kept_run(dec_src, e->T, [&](int j, int k, int len) {
    GemmEpilogue ge;
    ge.table = e->dec_cvec + static_cast<size_t>(j) * D;
    ge.rows_per_group = Bc;
    ge.flags = EPI_OUT_F32 | EPI_ROWTABLE;
    const char* a = reinterpret_cast<const char*>(enc_out) + static_cast<size_t>(dec_src[j]) * Bc * D * ab;
    float* c = (xout != nullptr ? xout : e->X.as<float>()) + static_cast<size_t>(j) * Bc * D;
    jobs[n++] = GemmJob{a, e->dec_w[k], e->dec_w16[k], c, len * Bc, D, D, ge};
  });
  return gemm_group(e, jobs, n, st);  // the runs of all modalities in one launch
}

// K5: per-modality output heads on `y2` (head-LayerNorm'ed) / `y1` (final-norm only, for the actor), whose row blocks are
// the needed tokens in NeedSet order.
int heads(m3pc_engine* e, const FwdIO& io, const NeedSet& need, const void* y1, const void* y2, int b0, int Bc, cudaStream_t st) {
  const int D = e->D, T = e->T;
  const size_t ab = act_bytes(e);
  float* outs[4] = {io.out_states, nullptr, io.out_rewards, io.out_returns};
  // hidden layers of all consumed modalities in one grouped launch, each into its own row range of HID
  GemmJob jobs[4];
  char* hid[4] = {nullptr, nullptr, nullptr, nullptr};
  int nj = 0;
  size_t hid_rows = 0;
  for (int k = 0; k < 4; ++k) {
    if (k == M3PC_ACTIONS || outs[k] == nullptr || need.nt[k] == 0) continue;
    GemmEpilogue ge;
    ge.bias = e->head_b1[k];
    ge.flags = EPI_GELU;
    const char* a = reinterpret_cast<const char*>(y2) + static_cast<size_t>(need.q0[k]) * Bc * D * ab;
    hid[k] = reinterpret_cast<char*>(e->HID.p) + hid_rows * D * ab;
    jobs[nj++] = GemmJob{a, e->head_w1[k], e->head_w1_16[k], hid[k], need.nt[k] * Bc, D, D, ge};
    hid_rows += static_cast<size_t>(need.nt[k]) * Bc + 128;  // slack rows: tile tails of one problem never touch the next one's rows
  }
  if (nj > 0) M3PC_TRY(gemm_group(e, jobs, nj, st));
  RowDotParams rps[4];
  int nr = 0;
  for (int k = 0; k < 4; ++k) {  // the output projections of all consumed modalities in one launch
    if (hid[k] == nullptr) continue;
    const int d = e->dims[k];
    RowDotParams rp{};
    rp.y = hid[k];
    rp.B = Bc; rp.tok0 = 0; rp.n_t = need.nt[k]; rp.t_out0 = need.t0[k]; rp.T_out = T; rp.d_out = d;
    rp.w = e->head_w3[k];
    rp.b = e->head_b3[k];
    rp.out = outs[k] + static_cast<size_t>(b0) * T * d;
    rps[nr++] = rp;
  }
  M3PC_TRY(launch_rowdot_group(rps, nr, D, e->bf16, st));
  if (io.out_mu != nullptr && need.nt[M3PC_ACTIONS] > 0) {
    RowDotParams rp{};
    rp.y = y1;
    rp.B = Bc; rp.tok0 = need.q0[M3PC_ACTIONS]; rp.n_t = need.nt[M3PC_ACTIONS]; rp.t_out0 = need.t0[M3PC_ACTIONS]; rp.T_out = T;
    rp.d_out = e->act;
    rp.w = e->mu_w; rp.b = e->mu_b;
    rp.out = io.out_mu + static_cast<size_t>(b0) * T * e->act;
    rp.w2 = e->ls_w; rp.b2 = e->ls_b;
    rp.out2 = io.out_std + static_cast<size_t>(b0) * T * e->act;
    M3PC_TRY(launch_rowdot(rp, D, e->bf16, st));
  }
  return M3PC_OK;
}

// final decoder norm (-> Y) chained with each head's own LayerNorm (-> Y2), mtm_model.py:428-433
int final_norms(m3pc_engine* e, const float* x, int n_tok, const int* tok, int Bc, cudaStream_t st, bool want_y1 = true) {
  LnParams ln{};
  ln.x = x;
  ln.rows = n_tok * Bc;
  ln.g1 = e->dec.norm_w;
  ln.b1 = e->dec.norm_b;
  ln.y1 = want_y1 ? e->Y.p : nullptr;  // only the actor head reads the final norm itself; the MLP heads read their own LayerNorm of it
  ln.y2 = e->Y2.p;
  ln.rows_per_group = Bc;
  for (int i = 0; i < n_tok; ++i) ln.tok_group[i] = static_cast<unsigned char>(tok[i] / e->T);
  for (int k = 0; k < 4; ++k) {
    ln.g2[k] = e->head_ln_w[k];  // null for actions: the actor reads the final norm directly
    ln.b2[k] = e->head_ln_b[k];
  }
  return launch_layernorm(ln, e->D, e->bf16, st);
}

// final norms + heads over all 4T decoder rows of `x` (token blocks in decoder order); reads need.t0 / need.nt
int heads_all_rows(m3pc_engine* e, const FwdIO& io, const float* x, NeedSet need, int b0, int Bc, cudaStream_t st) {
  const int T = e->T;
  int all_tok[MAX_TOK];
  for (int j = 0; j < 4 * T; ++j) all_tok[j] = j;
  M3PC_TRY(final_norms(e, x, 4 * T, all_tok, Bc, st));
  for (int k = 0; k < 4; ++k) need.q0[k] = k * T + need.t0[k];  // row block of (k, t0) in decoder order
  return heads(e, io, need, e->Y.p, e->Y2.p, b0, Bc, st);
}

// Last decoder layer restricted to the rows the caller consumes.  Identical results to the full layer for those rows:
//   * keys / values still cover all 4T tokens; queries, out-projection, MLP, norms and heads run on the needed tokens only;
//   * `src[j]` names the row block of X / Y (layer input and its LayerNorm) that holds decoder token j, or -1 for a token
//     whose layer input is batch-constant (single-layer decoder: mask-token rows) -- its Q / K / V come from the table built
//     once at finalize (const_qkv) and only the other tokens' K / V are projected per batch row.
// Expects X[0 : S*Bc) = layer input and Y = LN1(X) on entry.
int restricted_last_layer(m3pc_engine* e, const FwdIO& io, const LayerW& w, const int* src, int S, const NeedSet& need, int b0, int Bc,
                          cudaStream_t st) {
  const int D = e->D, T = e->T, F = e->F;
  const size_t ab = act_bytes(e);
  // (c) K, V of the per-batch tokens: rows D..3D of in_proj -> QKV as (S*Bc, 2D)
  GemmEpilogue ge;
  ge.bias = w.in_b + D;
  GemmJob kvq[MAX_TOK + 1];
  int nkvq = 0;
  kvq[nkvq++] = GemmJob{e->Y.p, w.in_w + static_cast<size_t>(D) * D, e->bf16 ? w.in_w16 + static_cast<size_t>(D) * D : nullptr, e->QKV.p, S * Bc, 2 * D, D, ge};
  // (d) Q of needed per-batch tokens -> QSEL row block qi (same launch as the K/V projection); runs of needed tokens whose
  //     source row blocks are consecutive share one problem
  for (int qi = 0; qi < need.n;) {
    const int s0 = src[need.tok[qi]];
    if (s0 < 0) { ++qi; continue; }
    int len = 1;
    while (qi + len < need.n && src[need.tok[qi + len]] == s0 + len) ++len;
    GemmEpilogue gq;
    gq.bias = w.in_b;
    const char* a = reinterpret_cast<const char*>(e->Y.p) + static_cast<size_t>(s0) * Bc * D * ab;
    char* c = reinterpret_cast<char*>(e->QSEL.p) + static_cast<size_t>(qi) * Bc * D * ab;
    kvq[nkvq++] = GemmJob{a, w.in_w, w.in_w16, c, len * Bc, D, D, gq};
    qi += len;
  }
  M3PC_TRY(gemm_group(e, kvq, nkvq, st));
  // (e) attention: needed queries x all 4T keys
  AttnParams ap{};
  ap.n_q = need.n;
  ap.n_kv = 4 * T;
  ap.B = Bc;
  ap.n_head = e->H;
  ap.out = e->ATT.p;
  const char* cq = reinterpret_cast<const char*>(e->const_qkv.p);
  for (int qi = 0; qi < need.n; ++qi) {
    const int j = need.tok[qi];
    if (src[j] < 0)
      ap.q[qi] = AttnTok{cq + static_cast<size_t>(j) * 3 * D * ab, 0};
    else
      ap.q[qi] = AttnTok{reinterpret_cast<const char*>(e->QSEL.p) + static_cast<size_t>(qi) * Bc * D * ab, D};
  }
  // keys / values: per-batch tokens first, batch-constant tokens after (attention is invariant to the key order; the bf16
  // kernel stages the constant ones once per CTA)
  int nk = 0;
  for (int pass = 0; pass < 2; ++pass)
    for (int j = 0; j < 4 * T; ++j) {
      if ((src[j] < 0) != (pass == 1)) continue;
      if (src[j] < 0) {
        ap.k[nk] = AttnTok{cq + (static_cast<size_t>(j) * 3 * D + D) * ab, 0};
        ap.v[nk] = AttnTok{cq + (static_cast<size_t>(j) * 3 * D + 2 * D) * ab, 0};
      } else {
        const char* row = reinterpret_cast<const char*>(e->QKV.p) + static_cast<size_t>(src[j]) * Bc * 2 * D * ab;
        ap.k[nk] = AttnTok{row, 2 * D};
        ap.v[nk] = AttnTok{row + D * ab, 2 * D};
      }
      ++nk;
      if (pass == 0) ap.n_kv_batch = nk;
    }
  if (ap.n_kv_batch == 4 * T) ap.n_kv_batch = 0;  // no constant keys (deeper decoders): plain kernel
  M3PC_TRY(launch_attention_gather(ap, e->bf16, st));
  // (f) out-projection + residual + norm2 of the needed tokens -> XS (compact, one row block per needed token) / Y.
  // A run = needed tokens with consecutive row blocks whose residual comes from one place: masked tokens take the batch-constant
  // row dec_maskrow[token] (consecutive tokens of a modality are consecutive table rows), kept tokens their own residual-stream rows.
  const int rows = need.n * Bc;
  ResLnJob jobs[MAX_TOK];
  int n_runs = 0;
  for (int qi = 0; qi < need.n;) {
    const int j = need.tok[qi];
    int len = 1;
    const float *table = nullptr, *res = nullptr;
    if (src[j] < 0) {
      while (qi + len < need.n && need.tok[qi + len] == j + len && src[j + len] < 0) ++len;
      table = e->dec_maskrow + static_cast<size_t>(j) * D;
    } else {
      while (qi + len < need.n && src[need.tok[qi + len]] == src[j] + len) ++len;
      res = e->X.as<float>() + static_cast<size_t>(src[j]) * Bc * D;
    }
    const size_t off = static_cast<size_t>(qi) * Bc;
    jobs[n_runs++] = ResLnJob{reinterpret_cast<const char*>(e->ATT.p) + off * D * ab, w.out_w, w.out_w16, e->XS.as<float>() + off * D,
                              reinterpret_cast<char*>(e->Y.p) + off * D * ab, table, Bc, len * Bc, res};
    qi += len;
  }
  M3PC_TRY(gemm_res_ln(e, jobs, n_runs, w.out_b, w.n2_w, w.n2_b, D, fuse_ln(e, rows), st));
  ge = GemmEpilogue{};
  ge.bias = w.l1_b;
  ge.flags = EPI_GELU;
  M3PC_TRY(gemm(e, e->Y.p, w.l1_w, w.l1_w16, e->HID.p, rows, F, D, ge, st));
  ge = GemmEpilogue{};
  ge.bias = w.l2_b;
  ge.flags = EPI_RESIDUAL;
  M3PC_TRY(gemm(e, e->HID.p, w.l2_w, w.l2_w16, e->XS.p, rows, D, F, ge, st));
  // (h) norms + heads
  M3PC_TRY(final_norms(e, e->XS.as<float>(), need.n, need.tok, Bc, st, io.out_mu != nullptr && need.nt[M3PC_ACTIONS] > 0));
  return heads(e, io, need, e->Y.p, e->Y2.p, b0, Bc, st);
}

// Single-layer decoder: the masked tokens' layer input is batch-constant, so only the kept tokens are embedded (compact,
// encoder order) and the rest comes from the constant table.
int decode_restricted(m3pc_engine* e, const FwdIO& io, const void* enc_out, const int* dec_src, int S, const NeedSet& need, int b0, int Bc,
                      cudaStream_t st) {
  const LayerW& w = e->dec.layers[0];
  const int D = e->D;
  const size_t ab = act_bytes(e);
  // (a) + (b), one job per run of kept tokens of a modality: X = dec_cvec[token] + enc_out W_dec^T (compact, encoder order:
  // X[0 : S*Bc)), Y = LN1(X) -- the table-residual form of the residual GEMM + LayerNorm (no residual traffic at all)
  ResLnJob jobs[MAX_TOK];
  int nj = 0, min_rows = 1 << 30;
  for_each_kept_run(dec_src, e->T, [&](int j, int k, int len) {
    const size_t r0 = static_cast<size_t>(dec_src[j]) * Bc;
    jobs[nj++] = ResLnJob{reinterpret_cast<const char*>(enc_out) + r0 * D * ab, e->dec_w[k], e->dec_w16[k], e->X.as<float>() + r0 * D,
                          reinterpret_cast<char*>(e->Y.p) + r0 * D * ab, e->dec_cvec + static_cast<size_t>(j) * D, Bc, len * Bc, nullptr};
    min_rows = std::min(min_rows, len * Bc);
  });
  M3PC_TRY(gemm_res_ln(e, jobs, nj, nullptr, w.n1_w, w.n1_b, D, fuse_ln(e, min_rows), st));
  return restricted_last_layer(e, io, w, dec_src, S, need, b0, Bc, st);
}

// Decoder on all 4T rows (mtm_model.py:663-716 computes every row of every layer).  `restrict_last` (deeper decoders; after the
// first layer no row is batch-constant any more): layers 0 .. Ld-2 run on all rows, the last layer only on the rows the caller
// consumes.  Otherwise every layer and the heads run on all rows.
int decode_full(m3pc_engine* e, const FwdIO& io, const void* enc_out, const int* dec_src, const NeedSet& need, int b0, int Bc,
                bool restrict_last, cudaStream_t st) {
  const int D = e->D, Sd = 4 * e->T;
  M3PC_TRY(launch_fill_rows(mask_rows(e, dec_src, Bc), D, e->X.as<float>(), st));
  M3PC_TRY(decoder_embed(e, enc_out, dec_src, Bc, st));
  M3PC_TRY(layernorm(e->X.as<float>(), Sd * Bc, e->dec.layers[0].n1_w, e->dec.layers[0].n1_b, e->Y.p, D, e->bf16, st));
  const int n_full = restrict_last ? e->Ld - 1 : e->Ld;
  for (int l = 0; l < n_full; ++l) {
    PostLn post;  // the next layer's norm1 rides on this layer's linear2
    if (l + 1 < e->Ld) post = PostLn{e->dec.layers[l + 1].n1_w, e->dec.layers[l + 1].n1_b, e->Y.p};
    M3PC_TRY(block(e, e->dec.layers[l], Bc, Sd, st, post));
  }
  if (!restrict_last) return heads_all_rows(e, io, e->X.as<float>(), need, b0, Bc, st);
  int ident[MAX_TOK];
  for (int j = 0; j < Sd; ++j) ident[j] = j;
  return restricted_last_layer(e, io, e->dec.layers[e->Ld - 1], ident, Sd, need, b0, Bc, st);
}

// Token tables of a mask layout (omtm._index / process_masks, mtm_model.py:534-591): kept tokens keep their order, modality-major;
// every inference mask keeps per-modality order, so the restore permutation reduces to "decoder token j <- encoder row dec_src[j]".
struct TokTables {
  int enc_mod[MAX_TOK], enc_t[MAX_TOK], dec_src[MAX_TOK];
  int S = 0;
};
TokTables token_tables(const uint8_t* mask, int T) {
  TokTables tt;
  for (int k = 0; k < 4; ++k)
    for (int t = 0; t < T; ++t) {
      if (mask[k * T + t]) {
        tt.enc_mod[tt.S] = k;
        tt.enc_t[tt.S] = t;
        tt.dec_src[k * T + t] = tt.S++;
      } else {
        tt.dec_src[k * T + t] = -1;
      }
    }
  return tt;
}

// K1 parameters: one EmbedTok per kept token (trajectory_encoding + the gather of forward_encoder, mtm_model.py:546-557, 619-632)
EmbedParams embed_params(const m3pc_engine* e, const FwdIO& io, const TokTables& tt, int b0, int Bc) {
  const int D = e->D, T = e->T;
  EmbedParams ep{};
  ep.n_tok = tt.S;
  ep.B = Bc;
  ep.b0 = b0;
  for (int s = 0; s < tt.S; ++s) {
    const int k = tt.enc_mod[s], t = tt.enc_t[s], d = e->dims[k];
    const ModSrc& ms = io.src[k];
    EmbedTok& tk = ep.tok[s];
    if (ms.base2 != nullptr && t >= ms.t_split) {
      tk.src = ms.base2 + static_cast<size_t>(b0) * ms.bstride2 + static_cast<size_t>(t - ms.t_split) * d;
      tk.bstride = static_cast<int>(ms.bstride2);
    } else if (ms.bdiv > 0) {
      tk.src = ms.base + static_cast<size_t>(t) * d;  // the kernel adds ((b0 + b) / bdiv) * bstride
      tk.bstride = static_cast<int>(ms.bstride);
      tk.bdiv = ms.bdiv;
    } else {
      tk.src = ms.base + static_cast<size_t>(b0) * ms.bstride + static_cast<size_t>(t) * d;
      tk.bstride = static_cast<int>(ms.bstride);
    }
    tk.wt = e->enc_wt[k];
    tk.cvec = e->enc_cvec + (static_cast<size_t>(k) * T + t) * D;
    tk.nmean = ms.normalize ? e->tok_mean[k] : nullptr;
    tk.nstd = ms.normalize ? e->tok_std[k] : nullptr;
    tk.d = d;
  }
  return ep;
}

int forward_chunk(m3pc_engine* e, const FwdIO& io, int b0, int Bc, cudaStream_t st) {
  const int D = e->D, T = e->T;
  const size_t ab = act_bytes(e);
  const TokTables tt = token_tables(io.mask, T);
  const int S = tt.S;
  const int* dec_src = tt.dec_src;
  M3PC_REQUIRE(S > 0, "forward: every token is masked");

  // ---- which head rows does the caller consume? ----
  NeedSet need;
  const float* outp[4] = {io.out_states, io.out_mu, io.out_rewards, io.out_returns};
  for (int k = 0; k < 4; ++k) {
    need.q0[k] = need.n;
    if (outp[k] == nullptr) continue;
    const int t0 = io.need_nt[k] < 0 ? 0 : io.need_t0[k];
    const int nt = io.need_nt[k] < 0 ? T : io.need_nt[k];
    M3PC_REQUIRE(t0 >= 0 && nt >= 0 && t0 + nt <= T, "need range out of bounds");
    need.t0[k] = t0;
    need.nt[k] = nt;
    for (int t = t0; t < t0 + nt; ++t) need.tok[need.n++] = k * T + t;
  }
  const EmbedParams ep = embed_params(e, io, tt, b0, Bc);  // the encoder tokens, for K1 or the fused B = 1 kernel

  // ---- B = 1: the whole encoder + restricted decoder in one cooperative kernel (fused_b1.cu) ----
  bool grouped_src = false;
  for (int k = 0; k < 4; ++k) grouped_src = grouped_src || io.src[k].bdiv > 0;
  if (Bc == 1 && !grouped_src && e->bf16 && e->use_fused_b1 && e->Ld == 1 && e->Le >= 1 && e->Le <= FB_MAX_LAYERS && need.n >= 1 && need.n < 4 * T &&
      need.n <= FB_MAX_ROWS && S <= FB_MAX_ROWS && D == 512 && fused_b1_smem_bytes(D, S, need.n) <= 200 * 1024) {
    FusedB1Params fp{};
    fp.S = S; fp.n_enc = e->Le; fp.T4 = 4 * T; fp.n_need = need.n;
    auto fill_layer = [](FusedLayer& f, const LayerW& w) {
      f.in_w = w.in_w16; f.out_w = w.out_w16; f.l1_w = w.l1_w16; f.l2_w = w.l2_w16;
      f.in_b = w.in_b; f.out_b = w.out_b; f.l1_b = w.l1_b; f.l2_b = w.l2_b;
      f.n1_w = w.n1_w; f.n1_b = w.n1_b; f.n2_w = w.n2_w; f.n2_b = w.n2_b;
    };
    for (int l = 0; l < e->Le; ++l) fill_layer(fp.enc[l], e->enc.layers[l]);
    fill_layer(fp.dec, e->dec.layers[0]);
    fp.enc_norm_w = e->enc.norm_w; fp.enc_norm_b = e->enc.norm_b;
    fp.fnorm_w = e->dec.norm_w; fp.fnorm_b = e->dec.norm_b;
    for (int k = 0; k < 4; ++k) {
      fp.head_g[k] = e->head_ln_w[k]; fp.head_b[k] = e->head_ln_b[k];
      fp.dec_w[k] = e->dec_w16[k];
    }
    fp.dec_cvec = e->dec_cvec; fp.dec_maskrow = e->dec_maskrow;
    fp.const_qkv = e->const_qkv.as<__nv_bfloat16>();
    for (int s = 0; s < S; ++s) {  // the kernel reads src, wt, cvec, nmean, nstd and d of a token (the single batch row's source)
      const int k = tt.enc_mod[s];
      fp.tok[s] = ep.tok[s];
      fp.enc_dectok[s] = static_cast<unsigned char>(k * T + tt.enc_t[s]);
      for (int kk = k + 1; kk <= 4; ++kk) fp.mod_row0[kk] = s + 1;
    }
    for (int j = 0; j < 4 * T; ++j) fp.dec_src[j] = static_cast<signed char>(dec_src[j]);
    for (int qi = 0; qi < need.n; ++qi) {
      fp.need_tok[qi] = static_cast<unsigned char>(need.tok[qi]);
      fp.need_mod[qi] = static_cast<unsigned char>(need.tok[qi] / T);
    }
    fp.X = e->X.as<float>(); fp.Xd = e->fb_xd.as<float>(); fp.XS = e->XS.as<float>();
    fp.QKV = e->QKV.as<__nv_bfloat16>(); fp.ATT = e->ATT.as<__nv_bfloat16>(); fp.HID = e->HID.as<__nv_bfloat16>();
    fp.Y = e->Y.as<__nv_bfloat16>(); fp.Y2 = e->Y2.as<__nv_bfloat16>();
    fp.bar = e->fb_bar.as<unsigned>();
    // the actor head is folded into the kernel's last phase; the MLP heads of the other modalities keep their own launches
    FwdIO io_rest = io;
    if (io.out_mu != nullptr && need.nt[M3PC_ACTIONS] > 0) {
      fp.mu_w = e->mu_w; fp.mu_b = e->mu_b; fp.ls_w = e->ls_w; fp.ls_b = e->ls_b;
      fp.out_mu = io.out_mu + static_cast<size_t>(b0) * T * e->act;
      fp.out_std = io.out_std + static_cast<size_t>(b0) * T * e->act;
      fp.act_dim = e->act;
      io_rest.out_mu = io_rest.out_std = nullptr;
    }
    M3PC_TRY(launch_fused_b1(fp, D, st));
    return heads(e, io_rest, need, e->Y.p, e->Y2.p, b0, 1, st);
  }

  // ---- K1: embed + gather + first LayerNorm ----
  const LayerW& first = e->Le > 0 ? e->enc.layers[0] : e->dec.layers[0];
  // shared-history analysis: the leading encoder tokens whose source row is shared by whole groups of batch rows (one window
  // for the whole batch: bstride 0; one window per environment: bdiv rows each) -- the chunk must hold whole groups
  int n_sh = 0, grp = 0;
  if (e->Le >= 1 && Bc >= 64) {
    for (int s = 0; s < S; ++s) {
      const EmbedTok& tk = ep.tok[s];
      const int g = tk.bdiv > 0 ? tk.bdiv : (tk.bstride == 0 ? Bc : 0);
      if (g == 0 || (grp != 0 && g != grp)) break;
      grp = g;
      ++n_sh;
    }
    const bool aligned = grp > 0 && Bc % grp == 0 && (grp == Bc || b0 % grp == 0);
    if (!aligned || n_sh == S || static_cast<long>(n_sh) * (Bc / std::max(grp, 1)) > TAB_ROWS) n_sh = 0;
  }
  if (n_sh > 0) {
    const int nG = Bc / grp;
    EmbedParams ea{};  // shared tokens, one row per group
    ea.n_tok = n_sh;
    ea.B = nG;
    for (int s = 0; s < n_sh; ++s) {
      ea.tok[s] = ep.tok[s];
      if (ea.tok[s].bdiv > 0) ea.tok[s].src += static_cast<size_t>(b0 / grp) * ea.tok[s].bstride;  // first group of this chunk
      ea.tok[s].bdiv = 0;
    }
    M3PC_TRY(launch_embed(ea, D, e->XT.as<float>(), e->YT.p, e->bf16, first.n1_w, first.n1_b, st));
    EmbedParams eb{};  // per-candidate tokens, written at their usual rows
    eb.n_tok = S - n_sh;
    eb.B = Bc;
    eb.b0 = b0;
    for (int s = n_sh; s < S; ++s) eb.tok[s - n_sh] = ep.tok[s];
    const size_t off = static_cast<size_t>(n_sh) * Bc * D;
    M3PC_TRY(launch_embed(eb, D, e->X.as<float>() + off, reinterpret_cast<char*>(e->Y.p) + off * ab, e->bf16, first.n1_w, first.n1_b, st));
  } else {
    M3PC_TRY(launch_embed(ep, D, e->X.as<float>(), e->Y.p, e->bf16, e->Le > 0 ? first.n1_w : e->enc.norm_w,
                          e->Le > 0 ? first.n1_b : e->enc.norm_b, st));
  }
  void* enc_out = e->Le > 0 ? e->ENC.p : e->Y.p;

  // ---- encoder stack (mtm_model.py:379-391, 619-644) ----
  for (int l = 0; l < e->Le; ++l) {
    // the LayerNorm that follows the block (next block's norm1, or the final encoder norm -> ENC) rides on its linear2
    PostLn post;
    if (l + 1 < e->Le)
      post = PostLn{e->enc.layers[l + 1].n1_w, e->enc.layers[l + 1].n1_b, e->Y.p};
    else
      post = PostLn{e->enc.norm_w, e->enc.norm_b, e->ENC.p};
    if (l == 0 && n_sh > 0)
      M3PC_TRY(block_shared_history(e, e->enc.layers[0], Bc, S, n_sh, grp, st, post));
    else
      M3PC_TRY(block(e, e->enc.layers[l], Bc, S, st, post));
  }

  if (need.n == 0) return M3PC_OK;
  if (e->Ld == 1 && need.n < 4 * T) return decode_restricted(e, io, enc_out, dec_src, S, need, b0, Bc, st);
  return decode_full(e, io, enc_out, dec_src, need, b0, Bc, e->Ld > 1 && need.n < 4 * T && e->restrict_deep, st);
}

int forward(m3pc_engine* e, const FwdIO& io, int B, cudaStream_t st) {
  M3PC_REQUIRE(e->finalized, "forward before m3pc_finalize_params");
  M3PC_REQUIRE(B >= 1 && B <= e->cfg.max_batch, "batch exceeds cfg.max_batch");
  M3PC_REQUIRE((io.out_mu == nullptr) == (io.out_std == nullptr), "out_act_mu and out_act_std go together");
  for (int b0 = 0; b0 < B; b0 += e->chunk) M3PC_TRY(forward_chunk(e, io, b0, std::min(e->chunk, B - b0), st));
  return M3PC_OK;
}

// K7: TwinQ on all (candidate, step) rows at once (the reference calls it h times on N rows, learner.py:250-252).
// bf16 mode: the two hidden layers run on the tcgen05 GEMM (bf16 operands, fp32 accumulate, second layer written in fp32);
// otherwise (and in the fp32 / tf32x3 modes) fp32 GEMMs on the mode's fp32 kernel (gemm_f32).  The final 256 -> 1 layer and
// min(q1, q2) are fp32 in all modes.
int critic(m3pc_engine* e, int N, int h, cudaStream_t st, const float* states_pred = nullptr, const float* cand = nullptr, float* q_out = nullptr) {
  const int rows = N * h, in = e->obs + e->act, Hq = e->QH;
  float* qv = q_out != nullptr ? q_out : e->qvals.as<float>();
  CriticInParams ci{};
  ci.states_pred = states_pred != nullptr ? states_pred : e->pred_states.as<float>();
  ci.cand = cand != nullptr ? cand : e->cand.as<float>();
  ci.tok_mean = e->tok_mean[M3PC_STATES];
  ci.tok_std = e->tok_std[M3PC_STATES];
  ci.obs_mean = e->obs_mean;
  ci.obs_std = e->obs_std;
  ci.sa = e->sa.p;
  ci.N = N; ci.h = h; ci.T = e->T; ci.obs = e->obs; ci.A = e->act;
  ci.ld = e->critic_tc ? e->q_kp : in;
  ci.out_bf16 = e->critic_tc;
  M3PC_TRY(launch_critic_input(ci, st));
  float* outs[2] = {e->qb1.as<float>(), e->qb2.as<float>()};
  if (e->critic_tc) {  // both nets per layer in one grouped launch (qa holds two bf16 activations side by side)
    char* qa2 = reinterpret_cast<char*>(e->qa.p) + (static_cast<size_t>(rows) + 128) * Hq * 2;
    void* qa[2] = {e->qa.p, qa2};
    GemmJob l1[2], l2[2];
    for (int q = 0; q < 2; ++q) {
      GemmEpilogue g1, g2;
      g1.bias = e->q_b[q][0];
      g1.flags = EPI_RELU;
      g2.bias = e->q_b[q][1];
      g2.flags = EPI_RELU | EPI_OUT_F32;
      l1[q] = GemmJob{e->sa.p, nullptr, e->q_w16[q][0], qa[q], rows, Hq, e->q_kp, g1};
      l2[q] = GemmJob{qa[q], nullptr, e->q_w16[q][1], outs[q], rows, Hq, Hq, g2};
    }
    M3PC_TRY(gemm_group(e, l1, 2, st));
    M3PC_TRY(gemm_group(e, l2, 2, st));
    return launch_critic_out(outs[0], outs[1], e->q_w[0][2], e->q_b[0][2], e->q_w[1][2], e->q_b[1][2], qv, rows, Hq, st);
  }
  for (int q = 0; q < 2; ++q) {
    GemmEpilogue ge;
    ge.bias = e->q_b[q][0];
    ge.flags = EPI_RELU;
    M3PC_TRY(profiled(e, 2.0 * rows * Hq * in, st, [&] { return gemm_f32(e, e->sa.as<float>(), e->q_w[q][0], e->qa.as<float>(), rows, Hq, in, ge, st); }));
    ge.bias = e->q_b[q][1];
    M3PC_TRY(profiled(e, 2.0 * rows * Hq * Hq, st, [&] { return gemm_f32(e, e->qa.as<float>(), e->q_w[q][1], outs[q], rows, Hq, Hq, ge, st); }));
  }
  return launch_critic_out(outs[0], outs[1], e->q_w[0][2], e->q_b[0][2], e->q_w[1][2], e->q_b[1][2], qv, rows, Hq, st);
}

void set_window_sources(m3pc_engine* e, FwdIO& io, const float* ws, const float* wa, const float* wr, const float* wrt, long stride_mul) {
  const int T = e->T;
  io.src[M3PC_STATES] = ModSrc{ws, stride_mul * T * e->obs, true};
  io.src[M3PC_ACTIONS] = ModSrc{wa, stride_mul * T * e->act, false};
  io.src[M3PC_REWARDS] = ModSrc{wr, stride_mul * T, true};
  io.src[M3PC_RETURNS] = ModSrc{wrt, stride_mul * T, false};
}

// sources and mask of a forward on already tokenised (batch, T, d) inputs
int io_from_tokens(const m3pc_engine* e, FwdIO& io, const float* ts, const float* ta, const float* tr, const float* tt, const uint8_t* masks) {
  M3PC_REQUIRE(masks != nullptr, "null masks");
  const int T = e->T;
  io.src[M3PC_STATES] = ModSrc{ts, static_cast<long>(T) * e->obs, false};
  io.src[M3PC_ACTIONS] = ModSrc{ta, static_cast<long>(T) * e->act, false};
  io.src[M3PC_REWARDS] = ModSrc{tr, static_cast<long>(T), false};
  io.src[M3PC_RETURNS] = ModSrc{tt, static_cast<long>(T), false};
  for (int i = 0; i < 4 * T; ++i) {
    M3PC_REQUIRE(masks[i] <= 1, "mask entries must be 0 or 1");
    io.mask[i] = masks[i];
  }
  return M3PC_OK;
}

// env_id: null, or the device id table of a horizon class planned by plan_mixed (local environment -> the caller's index)
int plan_body(m3pc_engine* e, const m3pc_plan_args_t* a, cudaStream_t st, const int* env_id = nullptr) {
  M3PC_REQUIRE(e->finalized, "plan before m3pc_finalize_params");
  const int T = e->T, h = a->horizon, N = a->n_cand, A = e->act, idx = T - h;
  const int E = a->n_env > 1 ? a->n_env : 1;  // lock-step environments planned by this call
  const long R = static_cast<long>(E) * N;    // pass-2 rows: environment-major, candidate-minor
  M3PC_REQUIRE(a->n_env >= 0, "n_env must be >= 0");
  M3PC_REQUIRE(E == 1 || (a->out_partials == nullptr && a->cand_offset == 0 && a->exchange == 0), "n_env > 1 cannot be combined with candidate sharding");
  M3PC_REQUIRE(a->exchange == 0 || a->exchange == 1, "exchange must be 0 or 1");
  M3PC_REQUIRE(a->exchange == 0 || (e->xch_world >= 1 && a->guidance != M3PC_GUIDE_SAMPLING), "exchange requested but m3pc_exchange_connect was not called (or plan = False)");
  M3PC_REQUIRE(E <= e->cfg.max_batch, "n_env exceeds cfg.max_batch");
  M3PC_REQUIRE(h >= 1 && h <= T, "horizon must be in [1, traj_length]");
  M3PC_REQUIRE(a->guidance >= 0 && a->guidance <= 3, "unknown guidance");
  M3PC_REQUIRE(a->win_states && a->win_actions && a->win_rewards && a->win_returns_tok, "window pointers must be set");
  M3PC_REQUIRE(a->out_eval_action && a->out_sample_action, "output pointers must be set");
  const bool needs_critic = a->guidance == M3PC_GUIDE_CRITIC || a->guidance == M3PC_GUIDE_NOISE_CRITIC;
  M3PC_REQUIRE(!needs_critic || e->has_critic, "critic guidance requested but no critic parameters were loaded");
  if (a->guidance != M3PC_GUIDE_SAMPLING) M3PC_REQUIRE(N >= 1 && R <= e->cfg.max_batch, "n_env * n_cand exceeds cfg.max_batch");

  // ---- pass 1: B = 1, rcbc mask (finetune_omtm/masks.py:7-27) -> action distribution ----
  FwdIO io{};
  set_window_sources(e, io, a->win_states, a->win_actions, a->win_rewards, a->win_returns_tok, E > 1 ? 1 : 0);
  for (int t = 0; t < T; ++t) {
    io.mask[M3PC_STATES * T + t] = t <= idx;
    io.mask[M3PC_ACTIONS * T + t] = t < idx;
    io.mask[M3PC_REWARDS * T + t] = 0;
    io.mask[M3PC_RETURNS * T + t] = 1;
  }
  io.out_mu = E > 1 ? e->e_mu.as<float>() : e->p1_mu.as<float>();  // (E, T, A)
  io.out_std = E > 1 ? e->e_std.as<float>() : e->p1_std.as<float>();
  io.need_t0[M3PC_ACTIONS] = idx;  // only the planned steps of the action head are consumed
  io.need_nt[M3PC_ACTIONS] = h;
  M3PC_TRY(forward(e, io, E, st));
  if (a->guidance == M3PC_GUIDE_SAMPLING)
    return launch_sampling_tail(io.out_mu, io.out_std, a->eps, T, h, A, E, a->out_eval_action, a->out_sample_action, a->seed,
                                e->seed_ptr_active, st, 1, env_id);

  // ---- K6: candidates ----
  CandParams cp{};
  cp.mu = io.out_mu; cp.std = io.out_std; cp.eps = a->eps; cp.cand = e->cand.as<float>();
  cp.N = static_cast<int>(R); cp.h = h; cp.A = A; cp.T = T;
  cp.n_per_env = E > 1 ? N : 0;
  cp.noise_mode = a->guidance == M3PC_GUIDE_NOISE_CRITIC ? 1 : 0;
  cp.seed = a->seed; cp.cand_offset = a->cand_offset; cp.seed_ptr = e->seed_ptr_active; cp.env_id = env_id;
  M3PC_TRY(launch_candidates(cp, st));
  if (a->dbg_candidates)
    M3PC_CHECK_CUDA(cudaMemcpyAsync(a->dbg_candidates, cp.cand, sizeof(float) * R * h * A, cudaMemcpyDeviceToDevice, st));

  // ---- pass 2: B = N, fd mask (finetune_omtm/masks.py:30-44); history shared, planned actions per candidate ----
  FwdIO io2{};
  set_window_sources(e, io2, a->win_states, a->win_actions, a->win_rewards, a->win_returns_tok, E > 1 ? 1 : 0);
  if (E > 1)
    for (int k = 0; k < 4; ++k) io2.src[k].bdiv = N;  // rows [e*N, (e+1)*N) share window e
  io2.src[M3PC_ACTIONS].base2 = cp.cand;
  io2.src[M3PC_ACTIONS].bstride2 = static_cast<long>(h) * A;
  io2.src[M3PC_ACTIONS].t_split = idx;
  for (int t = 0; t < T; ++t) {
    io2.mask[M3PC_STATES * T + t] = t <= idx;
    io2.mask[M3PC_ACTIONS * T + t] = 1;
    io2.mask[M3PC_REWARDS * T + t] = 0;
    io2.mask[M3PC_RETURNS * T + t] = 0;
  }
  // consumed by the scorer (learner.py:301-316): rewards[idx .. T-2], and returns[idx ..] (rtg) or states[idx ..] (critic)
  io2.out_rewards = e->pred_rewards.as<float>();
  io2.need_t0[M3PC_REWARDS] = idx;
  io2.need_nt[M3PC_REWARDS] = h - 1;
  if (needs_critic) {
    io2.out_states = e->pred_states.as<float>();
    io2.need_t0[M3PC_STATES] = idx;
    io2.need_nt[M3PC_STATES] = h;
  } else {
    io2.out_returns = e->pred_returns.as<float>();
    io2.need_t0[M3PC_RETURNS] = idx;
    io2.need_nt[M3PC_RETURNS] = h;
  }
  M3PC_TRY(forward(e, io2, static_cast<int>(R), st));

  // ---- K7 + K8 ----
  if (needs_critic) M3PC_TRY(critic(e, static_cast<int>(R), h, st));
  ScoreParams sp{};
  sp.rewards_pred = io2.out_rewards;
  sp.returns_pred = needs_critic ? nullptr : io2.out_returns;
  sp.qvals = needs_critic ? e->qvals.as<float>() : nullptr;
  sp.rw_mean = e->h_tok_mean[M3PC_REWARDS]; sp.rw_std = e->h_tok_std[M3PC_REWARDS];
  sp.rt_mean = e->h_tok_mean[M3PC_RETURNS]; sp.rt_std = e->h_tok_std[M3PC_RETURNS];
  sp.discount = a->discount; sp.lmbda = a->lmbda;
  sp.N = static_cast<int>(R); sp.h = h; sp.T = T;
  sp.J = e->J.as<float>();
  SelectParams sl{};
  sl.score = sp;  // the score pass rides in the select launch
  sl.J = sp.J; sl.cand = cp.cand; sl.expq = a->expq;
  sl.n_env = E; sl.N = N; sl.h = h; sl.A = A;
  sl.temperature = a->temperature; sl.seed = a->seed; sl.cand_offset = a->cand_offset; sl.seed_ptr = e->seed_ptr_active;
  sl.eval_action = a->out_eval_action; sl.sample_action = a->out_sample_action;
  sl.partials = a->out_partials; sl.indices = a->dbg_indices; sl.env_id = env_id;
  if (a->exchange) {
    for (int g = 0; g < e->xch_world; ++g) sl.xch.peer[g] = e->xch_peer[g];
    sl.xch.rank = e->xch_rank;
    sl.xch.world = e->xch_world;
    sl.xch.epoch = e->xch_epoch.as<unsigned long long>();
    sl.xch.timeout_ns = 2000000000ull;  // 2 s: a peer that never launches its plan must not hang this GPU
  }
  M3PC_TRY(launch_select(sl, st));
  if (a->dbg_expect_return) M3PC_CHECK_CUDA(cudaMemcpyAsync(a->dbg_expect_return, sp.J, sizeof(float) * R, cudaMemcpyDeviceToDevice, st));
  return M3PC_OK;
}

// Horizon classes of a plan with env_horizons: class c holds the environments of horizon h[c] (ascending), in the caller's order,
// as gathered slots [off[c], off[c + 1]); src maps a gathered slot to the caller's environment.
struct MixPlan {
  int n_class = 0;
  int h[M3PC_MAX_T] = {}, off[M3PC_MAX_T + 1] = {};
  short src[MIX_MAX_ENV] = {};
};

// Splits E <= MIX_MAX_ENV environments with horizons hz[i] in [1, T] into their classes.
void horizon_classes(const int32_t* hz, int E, int T, MixPlan& m) {
  int n = 0;
  for (int hh = 1; hh <= T; ++hh) {
    const int start = n;
    for (int i = 0; i < E; ++i)
      if (hz[i] == hh) m.src[n++] = static_cast<short>(i);
    if (n > start) {
      m.h[m.n_class] = hh;
      m.off[m.n_class++] = start;
    }
  }
  m.off[m.n_class] = n;
}

// Validates env_horizons.  *mixed is false when it is null or all its entries are equal: the plan is then exactly the uniform one.
int mix_classes(const m3pc_engine* e, const m3pc_plan_args_t* a, MixPlan& m, bool* mixed) {
  *mixed = false;
  if (a->env_horizons == nullptr) return M3PC_OK;
  const int E = a->n_env > 1 ? a->n_env : 1;
  M3PC_REQUIRE(a->n_env >= 0, "n_env must be >= 0");
  M3PC_REQUIRE(a->exchange == 0 && a->out_partials == nullptr && a->cand_offset == 0, "env_horizons cannot be combined with candidate sharding");
  int hmax = 0;
  bool equal = true;
  for (int i = 0; i < E; ++i) {
    const int hi = a->env_horizons[i];
    M3PC_REQUIRE(hi >= 1 && hi <= e->T, "env_horizons entries must be in [1, traj_length]");
    hmax = std::max(hmax, hi);
    equal = equal && hi == a->env_horizons[0];
  }
  M3PC_REQUIRE(a->horizon == hmax, "with env_horizons, horizon must equal its largest entry");
  if (equal) return M3PC_OK;
  M3PC_REQUIRE(E <= MIX_MAX_ENV, "env_horizons: more environments than one mixed plan takes (256)");
  horizon_classes(a->env_horizons, E, e->T, m);
  *mixed = true;
  return M3PC_OK;
}

// A plan whose environments have different horizons: one gather launch, then per horizon class the uniform plan sequence at
// n_env = E_c on the class's contiguous windows (and noise rows), with the class's id table so Philox keys and outputs use the
// caller's environment index.  Each class computes exactly what the uniform call on its windows computes.
int plan_mixed(m3pc_engine* e, const m3pc_plan_args_t* a, const MixPlan& m, cudaStream_t st) {
  M3PC_REQUIRE(e->finalized, "plan before m3pc_finalize_params");
  M3PC_REQUIRE(a->win_states && a->win_actions && a->win_rewards && a->win_returns_tok, "window pointers must be set");
  const int T = e->T, A = e->act, N = a->n_cand, E = m.off[m.n_class], hmax = a->horizon;
  const bool g3 = a->guidance == M3PC_GUIDE_SAMPLING;
  M3PC_REQUIRE(E <= e->cfg.max_batch && (g3 || (N >= 1 && static_cast<long>(E) * N <= e->cfg.max_batch)), "n_env * n_cand exceeds cfg.max_batch");
  MixGatherParams g{};
  g.ws = a->win_states; g.wa = a->win_actions; g.wr = a->win_rewards; g.wt = a->win_returns_tok;
  g.gs = e->mix_ws.as<float>(); g.ga = e->mix_wa.as<float>(); g.gr = e->mix_wr.as<float>(); g.gt = e->mix_wt.as<float>();
  g.eps = a->eps; g.geps = e->mix_eps.as<float>();
  g.expq = g3 ? nullptr : a->expq; g.gexpq = e->mix_expq.as<float>();
  g.env_id = e->mix_id.as<int>();
  g.E = E; g.T = T; g.obs = e->obs; g.A = A; g.N = g3 ? 0 : N;
  g.eps_rows = g3 ? 1 : N;            // guidance 3: eps is (E, A)
  g.eps_ld = g3 ? A : hmax * A;
  for (int c = 0; c < m.n_class; ++c)
    for (int s = m.off[c]; s < m.off[c + 1]; ++s) {
      g.src[s] = m.src[s];
      g.slot_of[m.src[s]] = static_cast<short>(s);
      g.eps_off[s + 1] = g.eps_off[s] + g.eps_rows * (g3 ? A : m.h[c] * A);
    }
  M3PC_TRY(launch_mix_gather(g, st));
  for (int c = 0; c < m.n_class; ++c) {
    const int off = m.off[c], Ec = m.off[c + 1] - off, h = m.h[c];
    m3pc_plan_args_t sub = *a;
    sub.env_horizons = nullptr;
    sub.n_env = Ec;
    sub.horizon = h;
    sub.win_states = g.gs + static_cast<size_t>(off) * T * e->obs;
    sub.win_actions = g.ga + static_cast<size_t>(off) * T * A;
    sub.win_rewards = g.gr + static_cast<size_t>(off) * T;
    sub.win_returns_tok = g.gt + static_cast<size_t>(off) * T;
    sub.eps = a->eps ? g.geps + g.eps_off[off] : nullptr;
    sub.expq = g.expq ? g.gexpq + static_cast<size_t>(off) * N : nullptr;
    sub.dbg_expect_return = nullptr;
    sub.dbg_candidates = nullptr;
    M3PC_TRY(plan_body(e, &sub, st, g.env_id + off));
    // debug outputs (eager calls only) in the caller's environment order; steps >= h of a candidate row are not written
    for (int i = 0; i < Ec && !g3; ++i) {
      const size_t ce = static_cast<size_t>(m.src[off + i]);
      if (a->dbg_expect_return)
        M3PC_CHECK_CUDA(cudaMemcpyAsync(a->dbg_expect_return + ce * N, e->J.as<float>() + static_cast<size_t>(i) * N, sizeof(float) * N,
                                        cudaMemcpyDeviceToDevice, st));
      if (a->dbg_candidates)
        M3PC_CHECK_CUDA(cudaMemcpy2DAsync(a->dbg_candidates + ce * N * hmax * A, sizeof(float) * hmax * A,
                                          e->cand.as<float>() + static_cast<size_t>(i) * N * h * A, sizeof(float) * h * A, sizeof(float) * h * A, N,
                                          cudaMemcpyDeviceToDevice, st));
    }
  }
  return M3PC_OK;
}

// m3pc_plan: eager for parity / debug calls (injected noise, debug outputs, profiling); otherwise the launch sequence is
// captured once per (arguments, buffer addresses) into a CUDA graph and replayed -- ~70 dependent launches become one
// submission, which is what bounds the B = 1 pass.  The Philox key travels through a device scalar so replays differ.
int plan(m3pc_engine* e, const m3pc_plan_args_t* args, cudaStream_t st) {
  MixPlan mix;
  bool mixed = false;
  M3PC_TRY(mix_classes(e, args, mix, &mixed));
  m3pc_plan_args_t uniform;
  const m3pc_plan_args_t* a = args;
  if (args->env_horizons != nullptr && !mixed) {  // all horizons equal: the uniform plan, launch for launch and graph for graph
    uniform = *args;
    uniform.env_horizons = nullptr;
    a = &uniform;
  }
  auto body = [&](cudaStream_t s) { return mixed ? plan_mixed(e, a, mix, s) : plan_body(e, a, s); };
  const bool eager = !e->use_graphs || e->profile || a->eps || a->expq || a->dbg_expect_return || a->dbg_candidates || a->dbg_indices;
  if (eager) {
    e->seed_ptr_active = nullptr;
    return body(st);
  }
  m3pc_engine::PlanKey key;
  std::memset(&key, 0, sizeof(key));
  key.guidance = a->guidance; key.horizon = a->horizon; key.n_cand = a->n_cand; key.cand_offset = a->cand_offset; key.n_env = a->n_env > 1 ? a->n_env : 1;
  key.exchange = a->exchange;
  key.discount = a->discount; key.temperature = a->temperature; key.lmbda = a->lmbda;
  key.ws = a->win_states; key.wa = a->win_actions; key.wr = a->win_rewards; key.wt = a->win_returns_tok;
  key.ev = a->out_eval_action; key.sm = a->out_sample_action; key.pt = a->out_partials;
  if (mixed)
    for (int i = 0; i < mix.off[mix.n_class]; ++i) key.env_h[i] = static_cast<unsigned char>(a->env_horizons[i]);
  if (e->plan_graphs.size() > 64) e->drop_graphs();  // callers that keep changing buffers would otherwise grow the cache without bound
  m3pc_engine::PlanGraph& pg = e->plan_graphs[key];
  if (pg.exec == nullptr) {
    if (pg.seen++ < 1) {  // first sighting: run eagerly (also performs every lazy cudaFuncSetAttribute)
      e->seed_ptr_active = nullptr;
      return body(st);
    }
    // captured on a private stream: the caller's stream may be the legacy default stream, which cannot be captured;
    // the instantiated graph is then launched on the caller's stream
    cudaGraph_t graph = nullptr;
    if (e->cap_stream == nullptr) M3PC_CHECK_CUDA(cudaStreamCreateWithFlags(&e->cap_stream, cudaStreamNonBlocking));
    e->seed_ptr_active = e->seed_scalar.as<unsigned long long>();
    M3PC_CHECK_CUDA(cudaStreamBeginCapture(e->cap_stream, cudaStreamCaptureModeThreadLocal));
    const int before = g_launch_count;
    const int rc = body(e->cap_stream);
    pg.launches = g_launch_count - before;
    const cudaError_t ce = cudaStreamEndCapture(e->cap_stream, &graph);
    e->seed_ptr_active = nullptr;
    if (rc != M3PC_OK) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    M3PC_CHECK_CUDA(ce);
    M3PC_CHECK_CUDA(cudaGraphInstantiate(&pg.exec, graph, 0));
    M3PC_CHECK_CUDA(cudaGraphDestroy(graph));
    g_launch_count = before;
  }
  M3PC_TRY(launch_set_seed(e->seed_scalar.as<unsigned long long>(), a->seed, st));
  M3PC_CHECK_CUDA(cudaGraphLaunch(pg.exec, st));
  g_launch_count += pg.launches;
  return M3PC_OK;
}

// env_id: null, or the device id table of a horizon class planned by backward_plan_env (local environment -> the caller's index):
// outputs go to the caller's rows, Philox is keyed by the caller's index and eps is read from the caller's rows in place
int backward_plan(m3pc_engine* e, int mode, int E, int h, const float* ws, const float* wa, const float* wr, const float* wrt,
                  const float* eps, float* out_eval, float* out_sample, float* dbg_filled, cudaStream_t st, int n_draws = 1,
                  unsigned long long seed = 0ull, const int* env_id = nullptr) {
  M3PC_REQUIRE(e->finalized, "backward_plan before m3pc_finalize_params");
  const int T = e->T, idx = T - h, A = e->act;
  M3PC_REQUIRE(mode == 0 || mode == 1, "mode must be 0 (id) or 1 (piid)");
  M3PC_REQUIRE(h >= 1 && h <= T && E >= 1 && E <= e->cfg.max_batch, "bad horizon / n_env");
  FwdIO io{};
  set_window_sources(e, io, ws, wa, wr, wrt, 1);
  // gid == pi mask (zeroshot_omtm/masks.py:50-91): all states except (idx+1 .. T-2) when idx > 0; actions < idx
  for (int t = 0; t < T; ++t) {
    io.mask[M3PC_STATES * T + t] = !(idx > 0 && t >= idx + 1 && t < T - 1);
    io.mask[M3PC_ACTIONS * T + t] = t < idx;
    io.mask[M3PC_REWARDS * T + t] = 0;
    io.mask[M3PC_RETURNS * T + t] = 0;
  }
  if (mode == 0) {
    io.out_mu = e->e_mu.as<float>();
    io.out_std = e->e_std.as<float>();
    io.need_t0[M3PC_ACTIONS] = idx;
    io.need_nt[M3PC_ACTIONS] = 1;
    M3PC_TRY(forward(e, io, E, st));
  } else {
    io.out_states = e->pred_states.as<float>();
    M3PC_TRY(forward(e, io, E, st));
    M3PC_TRY(launch_piid_fill(ws, io.out_states, e->tok_mean[M3PC_STATES], e->tok_std[M3PC_STATES], e->filled.as<float>(), E, T, h, e->obs, st));
    if (dbg_filled)
      M3PC_CHECK_CUDA(cudaMemcpyAsync(dbg_filled, e->filled.p, sizeof(float) * E * T * e->obs, cudaMemcpyDeviceToDevice, st));
    FwdIO io2{};
    set_window_sources(e, io2, e->filled.as<float>(), wa, wr, wrt, 1);
    // fid mask (zeroshot_omtm/masks.py:30-47): all states, actions < idx
    for (int t = 0; t < T; ++t) {
      io2.mask[M3PC_STATES * T + t] = 1;
      io2.mask[M3PC_ACTIONS * T + t] = t < idx;
    }
    io2.out_mu = e->e_mu.as<float>();
    io2.out_std = e->e_std.as<float>();
    io2.need_t0[M3PC_ACTIONS] = idx;
    io2.need_nt[M3PC_ACTIONS] = 1;
    M3PC_TRY(forward(e, io2, E, st));
  }
  return launch_sampling_tail(e->e_mu.as<float>(), e->e_std.as<float>(), eps, T, h, A, E, out_eval, out_sample, seed, nullptr, st, n_draws,
                              env_id, env_id != nullptr);
}

// m3pc_backward_plan_env: one horizon per environment.  All equal: exactly the uniform call.  Otherwise one gather launch puts every
// horizon class's windows side by side, then backward_plan runs once per class at n_env = E_c on its contiguous windows with the
// class's id table.  The injected eps (E, C, A) is not gathered: it depends on no horizon, and E * C rows can exceed the gather buffer.
int backward_plan_env(m3pc_engine* e, int mode, int E, const int32_t* hz, int n_draws, const float* ws, const float* wa, const float* wr,
                      const float* wt, const float* eps, unsigned long long seed, float* out_eval, float* out_sample, cudaStream_t st) {
  M3PC_REQUIRE(e->finalized, "backward_plan before m3pc_finalize_params");
  M3PC_REQUIRE(mode == 0 || mode == 1, "mode must be 0 (id) or 1 (piid)");
  M3PC_REQUIRE(E >= 1 && E <= MIX_MAX_ENV && E <= e->cfg.max_batch, "n_env must be in [1, min(256, cfg.max_batch)]");
  bool equal = true;
  for (int i = 0; i < E; ++i) {
    M3PC_REQUIRE(hz[i] >= 1 && hz[i] <= e->T, "env_horizons entries must be in [1, traj_length]");
    equal = equal && hz[i] == hz[0];
  }
  if (equal) return backward_plan(e, mode, E, hz[0], ws, wa, wr, wt, eps, out_eval, out_sample, nullptr, st, n_draws, seed);
  MixPlan m;
  horizon_classes(hz, E, e->T, m);
  const int T = e->T, A = e->act;
  MixGatherParams g{};
  g.ws = ws; g.wa = wa; g.wr = wr; g.wt = wt;
  g.gs = e->mix_ws.as<float>(); g.ga = e->mix_wa.as<float>(); g.gr = e->mix_wr.as<float>(); g.gt = e->mix_wt.as<float>();
  g.env_id = e->mix_id.as<int>();
  g.E = E; g.T = T; g.obs = e->obs; g.A = A;
  for (int s = 0; s < E; ++s) {
    g.src[s] = m.src[s];
    g.slot_of[m.src[s]] = static_cast<short>(s);
  }
  M3PC_TRY(launch_mix_gather(g, st));
  for (int c = 0; c < m.n_class; ++c) {
    const size_t off = m.off[c];
    M3PC_TRY(backward_plan(e, mode, m.off[c + 1] - m.off[c], m.h[c], g.gs + off * T * e->obs, g.ga + off * T * A, g.gr + off * T, g.gt + off * T,
                           eps, out_eval, out_sample, nullptr, st, n_draws, seed, g.env_id + off));
  }
  return M3PC_OK;
}

int create(m3pc_handle_t* out, const m3pc_config_t* cfg) {
  M3PC_REQUIRE(out != nullptr && cfg != nullptr, "null argument");
  M3PC_REQUIRE(cfg->n_embd > 0 && cfg->n_embd % 128 == 0 && cfg->n_embd <= 1024, "n_embd must be a multiple of 128, <= 1024");
  M3PC_REQUIRE(cfg->n_head * 128 == cfg->n_embd, "head_dim must be 128 (n_head == n_embd / 128)");
  M3PC_REQUIRE(cfg->traj_length >= 1 && cfg->traj_length <= M3PC_MAX_T, "traj_length out of range");
  M3PC_REQUIRE(cfg->obs_dim >= 1 && cfg->obs_dim <= M3PC_MAX_OBS && cfg->act_dim >= 1 && cfg->act_dim <= M3PC_MAX_ACT, "obs/act dim out of range");
  M3PC_REQUIRE(cfg->n_enc_layer >= 1 && cfg->n_dec_layer >= 1, "need at least one encoder and one decoder layer");
  M3PC_REQUIRE(cfg->precision == M3PC_PREC_BF16 || cfg->precision == M3PC_PREC_FP32 || cfg->precision == M3PC_PREC_TF32X3,
               "unknown precision");
  M3PC_REQUIRE(cfg->max_batch >= 1, "max_batch must be positive");
  int dev = 0;
  M3PC_CHECK_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  M3PC_CHECK_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) {
    set_error(std::string("this library is built for sm_100a only; device is ") + prop.name + " (sm_" + std::to_string(prop.major) +
              std::to_string(prop.minor) + ")");
    return M3PC_ERR_CUDA;
  }
  std::unique_ptr<m3pc_engine> e(new m3pc_engine());
  e->cfg = *cfg;
  e->D = cfg->n_embd; e->H = cfg->n_head; e->T = cfg->traj_length; e->F = 4 * cfg->n_embd;
  e->obs = cfg->obs_dim; e->act = cfg->act_dim; e->Le = cfg->n_enc_layer; e->Ld = cfg->n_dec_layer; e->QH = cfg->critic_hidden;
  e->dims[0] = e->obs; e->dims[1] = e->act; e->dims[2] = 1; e->dims[3] = 1;
  e->bf16 = cfg->precision == M3PC_PREC_BF16;
  e->tf32x3 = cfg->precision == M3PC_PREC_TF32X3;
  e->chunk = cfg->chunk > 0 ? cfg->chunk : 8192;  // measured (profiles/r1e_chunk_sweep.txt, 8 x 1024 rows per step): 3.86 ms in chunks of 1024, 3.28 ms at 4096, 3.20 ms at 8192
  e->chunk = std::min(e->chunk, cfg->max_batch);
  if (e->bf16 || e->tf32x3) M3PC_TRY(gemm_init_driver_api());
  const size_t rows = static_cast<size_t>(4) * e->T * e->chunk + 128;  // +128: slack rows for tile tails
  const size_t ab = act_bytes(e.get()), D = e->D;
  M3PC_TRY(e->X.alloc(rows * D * 4));
  M3PC_TRY(e->XS.alloc(rows * D * 4));
  M3PC_TRY(e->QSEL.alloc(rows * D * ab));
  M3PC_TRY(e->const_qkv.alloc(static_cast<size_t>(4) * e->T * 3 * D * ab));
  M3PC_TRY(e->Y.alloc(rows * D * ab));
  M3PC_TRY(e->Y2.alloc(rows * D * ab));
  M3PC_TRY(e->QKV.alloc(rows * 3 * D * ab));
  M3PC_TRY(e->ATT.alloc(rows * D * ab));
  M3PC_TRY(e->HID.alloc(rows * 4 * D * ab));
  M3PC_TRY(e->ENC.alloc(rows * D * ab));
  M3PC_TRY(e->XT.alloc(static_cast<size_t>(TAB_ROWS + 128) * D * 4));
  M3PC_TRY(e->YT.alloc(static_cast<size_t>(TAB_ROWS + 128) * D * ab));
  M3PC_TRY(e->QKVT.alloc(static_cast<size_t>(TAB_ROWS + 128) * 3 * D * ab));
  for (DevBuf* b : {&e->X, &e->XS, &e->Y, &e->Y2, &e->QKV, &e->QSEL, &e->ATT, &e->HID, &e->ENC})
    M3PC_CHECK_CUDA(cudaMemset(b->p, 0, b->bytes));
  const size_t N = cfg->max_batch, T = e->T;
  M3PC_TRY(e->p1_mu.alloc(T * e->act * 4));
  M3PC_TRY(e->p1_std.alloc(T * e->act * 4));
  M3PC_TRY(e->cand.alloc(N * T * e->act * 4));
  M3PC_TRY(e->pred_states.alloc(N * T * e->obs * 4));
  M3PC_TRY(e->pred_rewards.alloc(N * T * 4));
  M3PC_TRY(e->pred_returns.alloc(N * T * 4));
  M3PC_TRY(e->J.alloc(N * 4));
  M3PC_TRY(e->filled.alloc(N * T * e->obs * 4));
  M3PC_TRY(e->e_mu.alloc(N * T * e->act * 4));
  M3PC_TRY(e->e_std.alloc(N * T * e->act * 4));
  const size_t NE = std::min<size_t>(N, MIX_MAX_ENV);  // environments of a mixed plan
  M3PC_TRY(e->mix_ws.alloc(NE * T * e->obs * 4));
  M3PC_TRY(e->mix_wa.alloc(NE * T * e->act * 4));
  M3PC_TRY(e->mix_wr.alloc(NE * T * 4));
  M3PC_TRY(e->mix_wt.alloc(NE * T * 4));
  M3PC_TRY(e->mix_eps.alloc(N * T * e->act * 4));  // sum_c E_c n_cand h_c A <= max_batch T A
  M3PC_TRY(e->mix_expq.alloc(N * 4));
  M3PC_TRY(e->mix_id.alloc(NE * 4));
  if (e->QH > 0) {
    M3PC_TRY(e->sa.alloc((N * T + 128) * static_cast<size_t>((e->obs + e->act + 63) / 64 * 64) * 4));
    M3PC_TRY(e->qa.alloc((N * T + 128) * e->QH * 4));
    M3PC_TRY(e->qb1.alloc(N * T * e->QH * 4));
    M3PC_TRY(e->qb2.alloc(N * T * e->QH * 4));
    M3PC_TRY(e->qvals.alloc(N * T * 4));
  }
  M3PC_TRY(e->seed_scalar.alloc(16));
  M3PC_TRY(e->fb_xd.alloc(static_cast<size_t>(FB_MAX_ROWS) * D * 4));
  M3PC_TRY(e->fb_bar.alloc(16));
  M3PC_CHECK_CUDA(cudaMemset(e->fb_bar.p, 0, 16));
  M3PC_CHECK_CUDA(cudaEventCreate(&e->ev0));
  M3PC_CHECK_CUDA(cudaEventCreate(&e->ev1));
  M3PC_CHECK_CUDA(cudaDeviceSynchronize());
  *out = e.release();
  return M3PC_OK;
}

template <typename Fn>
int timed(m3pc_engine* e, cudaStream_t st, Fn&& fn) {
  g_launch_count = 0;
  e->prof_used = 0;
  M3PC_CHECK_CUDA(cudaEventRecord(e->ev0, st));
  const int rc = fn();
  e->last_launches = g_launch_count;
  if (rc != M3PC_OK) return rc;
  M3PC_CHECK_CUDA(cudaEventRecord(e->ev1, st));
  return M3PC_OK;
}

}  // namespace
}  // namespace m3pc

// ================================================================================================ C ABI
extern "C" {

const char* m3pc_last_error(void) { return m3pc::g_error.c_str(); }
const char* m3pc_version(void) { return "m3pc-b200 0.3.0 (sm_100a)"; }

int m3pc_create(m3pc_handle_t* out, const m3pc_config_t* cfg) { return m3pc::create(out, cfg); }

int m3pc_destroy(m3pc_handle_t h) {
  if (h == nullptr) return M3PC_OK;
  cudaDeviceSynchronize();
  delete h;
  return M3PC_OK;
}

int m3pc_set_param(m3pc_handle_t h, const char* name, const float* data, size_t count) {
  M3PC_REQUIRE(h != nullptr && name != nullptr && data != nullptr, "null argument");
  h->finalized = false;
  h->drop_graphs();
  h->staged[name].assign(data, data + count);
  return M3PC_OK;
}

int m3pc_set_option(m3pc_handle_t h, const char* name, int32_t value) {
  M3PC_REQUIRE(h != nullptr && name != nullptr, "null argument");
  const std::string n(name);
  h->drop_graphs();  // the launch sequence a graph froze may no longer be the selected one
  if (n == "graphs") h->use_graphs = value != 0;
  else if (n == "fused_b1") h->use_fused_b1 = value != 0;
  else if (n == "fused_ln_min_rows") h->fuse_ln_min_rows = std::max(129, static_cast<int>(value));
  else if (n == "restrict_deep_decoder") h->restrict_deep = value != 0;
  else if (n == "gemm_ln_unit_rows") {
    M3PC_REQUIRE(value == 0 || value == 128 || value == 256, "gemm_ln_unit_rows must be 0 (per launch), 128 or 256");
    m3pc::g_ln_unit_rows = value;
  }
  else {
    m3pc::set_error("m3pc_set_option: unknown option '" + n + "'");
    return M3PC_ERR_INVALID;
  }
  return M3PC_OK;
}

int m3pc_finalize_params(m3pc_handle_t h) {
  M3PC_REQUIRE(h != nullptr, "null handle");
  return m3pc::finalize(h);
}

int m3pc_forward(m3pc_handle_t h, int32_t batch, const float* tok_states, const float* tok_actions, const float* tok_rewards,
                 const float* tok_returns, const uint8_t* masks, float* out_states, float* out_act_mu, float* out_act_std,
                 float* out_rewards, float* out_returns, void* stream) {
  M3PC_REQUIRE(h != nullptr && masks != nullptr, "null argument");
  M3PC_REQUIRE(tok_states && tok_actions && tok_rewards && tok_returns, "all four modalities must be given");
  m3pc::FwdIO io{};
  M3PC_TRY(m3pc::io_from_tokens(h, io, tok_states, tok_actions, tok_rewards, tok_returns, masks));
  io.out_states = out_states; io.out_mu = out_act_mu; io.out_std = out_act_std;
  io.out_rewards = out_rewards; io.out_returns = out_returns;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return m3pc::timed(h, st, [&] { return m3pc::forward(h, io, batch, st); });
}

int m3pc_plan(m3pc_handle_t h, const m3pc_plan_args_t* args, void* stream) {
  M3PC_REQUIRE(h != nullptr && args != nullptr, "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return m3pc::timed(h, st, [&] { return m3pc::plan(h, args, st); });
}

int m3pc_merge_partials(m3pc_handle_t h, const float* partials, int32_t n_shards, float temperature, float* out_eval_action,
                        float* out_sample_action, int32_t* out_indices, void* stream) {
  M3PC_REQUIRE(h != nullptr && partials && out_eval_action && out_sample_action && n_shards >= 1, "bad argument");
  return m3pc::launch_merge(partials, n_shards, h->act, temperature, out_eval_action, out_sample_action, out_indices,
                            reinterpret_cast<cudaStream_t>(stream));
}

// ---- peer exchange wiring (candidate sharding over GPUs) ----
namespace {
int xch_alloc(m3pc_handle_t h) {
  if (h->xch_buf.p != nullptr) return M3PC_OK;
  M3PC_TRY(h->xch_buf.alloc(m3pc::XCH_BYTES));
  M3PC_CHECK_CUDA(cudaMemset(h->xch_buf.p, 0, m3pc::XCH_BYTES));
  M3PC_TRY(h->xch_epoch.alloc(16));
  M3PC_CHECK_CUDA(cudaMemset(h->xch_epoch.p, 0, 16));
  M3PC_CHECK_CUDA(cudaDeviceSynchronize());
  return M3PC_OK;
}
}  // namespace

int m3pc_exchange_local(m3pc_handle_t h, uint8_t* out_ipc_handle, void** out_device_ptr) {
  M3PC_REQUIRE(h != nullptr, "null handle");
  M3PC_TRY(xch_alloc(h));
  if (out_ipc_handle != nullptr) {
    static_assert(sizeof(cudaIpcMemHandle_t) == M3PC_IPC_HANDLE_BYTES, "CUDA IPC handle size");
    cudaIpcMemHandle_t ih;
    M3PC_CHECK_CUDA(cudaIpcGetMemHandle(&ih, h->xch_buf.p));
    std::memcpy(out_ipc_handle, &ih, sizeof(ih));
  }
  if (out_device_ptr != nullptr) *out_device_ptr = h->xch_buf.p;
  return M3PC_OK;
}

int m3pc_exchange_connect(m3pc_handle_t h, int32_t rank, int32_t world, const uint8_t* ipc_handles, void* const* device_ptrs) {
  M3PC_REQUIRE(h != nullptr, "null handle");
  M3PC_REQUIRE(world >= 1 && world <= m3pc::XCH_MAX_RANKS && rank >= 0 && rank < world, "rank / world out of range");
  M3PC_REQUIRE((ipc_handles != nullptr) != (device_ptrs != nullptr), "give either IPC handles (peers in other processes) or device pointers (same process)");
  M3PC_TRY(xch_alloc(h));
  M3PC_CHECK_CUDA(cudaDeviceSynchronize());
  h->drop_graphs();  // captured plans hold the previous peer table
  for (void* q : h->xch_opened) cudaIpcCloseMemHandle(q);
  h->xch_opened.clear();
  for (int g = 0; g < world; ++g) {
    if (g == rank) {
      h->xch_peer[g] = h->xch_buf.p;
    } else if (device_ptrs != nullptr) {
      M3PC_REQUIRE(device_ptrs[g] != nullptr, "null peer pointer");
      h->xch_peer[g] = device_ptrs[g];
    } else {
      cudaIpcMemHandle_t ih;
      std::memcpy(&ih, ipc_handles + static_cast<size_t>(g) * sizeof(ih), sizeof(ih));
      void* q = nullptr;
      M3PC_CHECK_CUDA(cudaIpcOpenMemHandle(&q, ih, cudaIpcMemLazyEnablePeerAccess));
      h->xch_opened.push_back(q);
      h->xch_peer[g] = q;
    }
  }
  // a (re)connected group starts a fresh epoch sequence; every rank must (re)connect together
  M3PC_CHECK_CUDA(cudaMemset(h->xch_buf.p, 0, m3pc::XCH_BYTES));
  M3PC_CHECK_CUDA(cudaMemset(h->xch_epoch.p, 0, 16));
  M3PC_CHECK_CUDA(cudaDeviceSynchronize());
  h->xch_rank = rank;
  h->xch_world = world;
  return M3PC_OK;
}

int m3pc_exchange_status(m3pc_handle_t h, uint64_t* out_epoch, uint64_t* out_failed_epoch) {
  M3PC_REQUIRE(h != nullptr && h->xch_buf.p != nullptr && out_epoch && out_failed_epoch, "bad argument (or exchange not set up)");
  M3PC_CHECK_CUDA(cudaMemcpy(out_epoch, h->xch_epoch.p, 8, cudaMemcpyDeviceToHost));
  M3PC_CHECK_CUDA(cudaMemcpy(out_failed_epoch, reinterpret_cast<const char*>(h->xch_buf.p) + m3pc::XCH_ERR_OFFSET, 8, cudaMemcpyDeviceToHost));
  return M3PC_OK;
}

int m3pc_backward_plan(m3pc_handle_t h, int32_t mode, int32_t n_env, int32_t horizon, const float* win_states, const float* win_actions,
                       const float* win_rewards, const float* win_returns_tok, const float* eps, float* out_eval_action,
                       float* out_sample_action, float* dbg_states_filled, void* stream) {
  M3PC_REQUIRE(h != nullptr && win_states && win_actions && win_rewards && win_returns_tok && out_eval_action && out_sample_action,
               "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return m3pc::timed(h, st, [&] {
    return m3pc::backward_plan(h, mode, n_env, horizon, win_states, win_actions, win_rewards, win_returns_tok, eps, out_eval_action,
                               out_sample_action, dbg_states_filled, st);
  });
}

int m3pc_backward_plan_draws(m3pc_handle_t h, int32_t mode, int32_t n_env, int32_t horizon, int32_t n_draws, const float* win_states,
                             const float* win_actions, const float* win_rewards, const float* win_returns_tok, const float* eps,
                             uint64_t seed, float* out_eval_action, float* out_sample_actions, void* stream) {
  M3PC_REQUIRE(h != nullptr && win_states && win_actions && win_rewards && win_returns_tok && out_eval_action && out_sample_actions,
               "null argument");
  M3PC_REQUIRE(n_draws >= 1 && n_draws <= (1 << 20), "n_draws out of range");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return m3pc::timed(h, st, [&] {
    return m3pc::backward_plan(h, mode, n_env, horizon, win_states, win_actions, win_rewards, win_returns_tok, eps, out_eval_action,
                               out_sample_actions, nullptr, st, n_draws, seed);
  });
}

int m3pc_backward_plan_env(m3pc_handle_t h, int32_t mode, int32_t n_env, const int32_t* env_horizons, int32_t n_draws, const float* win_states,
                           const float* win_actions, const float* win_rewards, const float* win_returns_tok, const float* eps, uint64_t seed,
                           float* out_eval_action, float* out_sample_actions, void* stream) {
  M3PC_REQUIRE(h != nullptr && env_horizons && win_states && win_actions && win_rewards && win_returns_tok && out_eval_action && out_sample_actions,
               "null argument");
  M3PC_REQUIRE(n_draws >= 1 && n_draws <= (1 << 20), "n_draws out of range");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return m3pc::timed(h, st, [&] {
    return m3pc::backward_plan_env(h, mode, n_env, env_horizons, n_draws, win_states, win_actions, win_rewards, win_returns_tok, eps, seed,
                                   out_eval_action, out_sample_actions, st);
  });
}

int m3pc_ring_reset(float* ring, int32_t n_env, int32_t ring_len, int32_t obs_dim, int32_t act_dim, const int32_t* slots, int32_t n_slots,
                    void* stream) {
  return m3pc::launch_ring_reset(ring, n_env, ring_len, obs_dim, act_dim, slots, n_slots, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_ring_append_slots(float* ring, int32_t n_env, int32_t ring_len, int32_t obs_dim, int32_t act_dim, const int32_t* t, const int32_t* slots,
                           int32_t n_slots, const float* obs, const float* prev_action, const float* prev_reward, void* stream) {
  return m3pc::launch_ring_append_slots(ring, n_env, ring_len, obs_dim, act_dim, t, slots, n_slots, obs, prev_action, prev_reward,
                                        reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_ring_write_obs(float* ring, int32_t n_env, int32_t ring_len, int32_t obs_dim, int32_t act_dim, const int32_t* slots, int32_t n_slots,
                        int32_t first_row, int32_t n_rows, const float* obs_rows, void* stream) {
  return m3pc::launch_ring_write_obs(ring, n_env, ring_len, obs_dim, act_dim, slots, n_slots, first_row, n_rows, obs_rows,
                                     reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_ring_windows_slots(const float* ring, int32_t n_env, int32_t ring_len, int32_t obs_dim, int32_t act_dim, const int32_t* path_length,
                            const int32_t* slots, const int32_t* horizons, int32_t n_slots, int32_t traj_length, int32_t future_obs,
                            const float* rtg_tok, float* win_states, float* win_actions, float* win_rewards, float* win_returns_tok,
                            void* stream) {
  return m3pc::launch_ring_windows_slots(ring, n_env, ring_len, obs_dim, act_dim, path_length, slots, horizons, n_slots, traj_length, future_obs,
                                         rtg_tok, win_states, win_actions, win_rewards, win_returns_tok, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_gemm_bf16(const void* A, const void* W, const float* bias, void* C, int32_t M, int32_t N, int32_t K, int32_t flags, void* stream) {
  M3PC_REQUIRE(A && W && C, "null argument");
  M3PC_REQUIRE((flags & ~7) == 0, "unknown flag");
  m3pc::GemmEpilogue ep;
  ep.bias = bias;
  ep.flags = flags;
  const m3pc::GemmProblem pr{reinterpret_cast<const __nv_bfloat16*>(A), reinterpret_cast<const __nv_bfloat16*>(W), C, M, N, K, ep};
  return m3pc::gemm_bf16(&pr, 1, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_gemm_bf16_grouped(int32_t n, const void* const* A, const void* const* W, const float* const* bias, void* const* C, const int32_t* M,
                           const int32_t* N, const int32_t* K, const int32_t* flags, void* stream) {
  M3PC_REQUIRE(n >= 1 && n <= 16 && A && W && C && M && N && K && flags, "bad argument");
  m3pc::GemmProblem pr[16];
  for (int i = 0; i < n; ++i) {
    M3PC_REQUIRE(A[i] && W[i] && C[i], "null operand");
    M3PC_REQUIRE((flags[i] & ~7) == 0, "unknown flag");
    m3pc::GemmEpilogue ep;
    ep.bias = bias ? bias[i] : nullptr;
    ep.flags = flags[i];
    pr[i] = m3pc::GemmProblem{reinterpret_cast<const __nv_bfloat16*>(A[i]), reinterpret_cast<const __nv_bfloat16*>(W[i]), C[i], M[i], N[i], K[i], ep};
  }
  return m3pc::gemm_bf16(pr, n, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_gemm_ln_bf16(const void* A, const void* W, const float* bias, float* X, void* Y, const float* gamma, const float* beta,
                      const float* table, int32_t rows_per_group, int32_t M, int32_t K, void* stream) {
  const m3pc::LnJob job{reinterpret_cast<const __nv_bfloat16*>(A), reinterpret_cast<const __nv_bfloat16*>(W), X,
                        reinterpret_cast<__nv_bfloat16*>(Y), table, rows_per_group, M, nullptr};
  return m3pc::gemm_ln_bf16_grouped(&job, 1, bias, gamma, beta, K, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_gemm_bf16_problems(const m3pc_gemm_problem_t* p, int32_t n, int32_t* out_kernel, void* stream) {
  static_assert(M3PC_EPI_GELU == m3pc::EPI_GELU && M3PC_EPI_RESIDUAL == m3pc::EPI_RESIDUAL && M3PC_EPI_RELU == m3pc::EPI_RELU &&
                    M3PC_EPI_ROWTABLE == m3pc::EPI_ROWTABLE && M3PC_EPI_OUT_F32 == m3pc::EPI_OUT_F32,
                "public epilogue flags");
  M3PC_REQUIRE(p != nullptr && n >= 1 && n <= m3pc::MAX_TOK, "gemm_bf16_problems: 1 .. 64 problems");
  m3pc::GemmProblem pr[m3pc::MAX_TOK];
  for (int i = 0; i < n; ++i) {
    const m3pc_gemm_problem_t& q = p[i];
    M3PC_REQUIRE(q.A && q.W && q.C, "null operand");
    m3pc::GemmEpilogue ep;
    ep.bias = q.bias;
    ep.table = q.table;
    ep.rows_per_group = q.rows_per_group;
    ep.flags = q.flags;
    pr[i] = m3pc::GemmProblem{reinterpret_cast<const __nv_bfloat16*>(q.A), reinterpret_cast<const __nv_bfloat16*>(q.W), q.C, q.M, q.N, q.K, ep};
  }
  return m3pc::gemm_bf16(pr, n, reinterpret_cast<cudaStream_t>(stream), out_kernel);
}

int m3pc_gemm_ln_bf16_grouped(const m3pc_ln_job_t* jobs, int32_t n, const float* bias, const float* gamma, const float* beta, int32_t K,
                              int32_t* out_kernel, void* stream) {
  M3PC_REQUIRE(jobs != nullptr && n >= 1 && n <= m3pc::kMaxGroup, "gemm_ln_bf16_grouped: 1 .. 4 jobs");
  m3pc::LnJob lj[m3pc::kMaxGroup];
  for (int i = 0; i < n; ++i) {
    const m3pc_ln_job_t& j = jobs[i];
    lj[i] = m3pc::LnJob{reinterpret_cast<const __nv_bfloat16*>(j.A), reinterpret_cast<const __nv_bfloat16*>(j.W), j.X,
                        reinterpret_cast<__nv_bfloat16*>(j.Y), j.table, j.rows_per_group, j.M, j.R};
  }
  return m3pc::gemm_ln_bf16_grouped(lj, n, bias, gamma, beta, K, reinterpret_cast<cudaStream_t>(stream), out_kernel);
}

int m3pc_gemm_fp32(const float* A, const float* W, const float* bias, float* C, int32_t M, int32_t N, int32_t K, int32_t flags, void* stream) {
  M3PC_REQUIRE(A && W && C, "null argument");
  M3PC_REQUIRE((flags & ~7) == 0, "unknown flag");
  m3pc::GemmEpilogue ep;
  ep.bias = bias;
  ep.flags = flags;
  return m3pc::gemm_fp32(A, W, C, M, N, K, ep, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_gemm_tf32x3(const float* A, const float* W, const float* bias, float* C, int32_t M, int32_t N, int32_t K, int32_t flags, void* stream) {
  M3PC_REQUIRE(A && W && C, "null argument");
  M3PC_REQUIRE((flags & ~7) == 0, "unknown flag");
  m3pc::GemmEpilogue ep;
  ep.bias = bias;
  ep.flags = flags;
  return m3pc::gemm_tf32x3(A, W, C, M, N, K, ep, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_layernorm(const float* x, const float* gamma, const float* beta, void* y, int32_t M, int32_t D, int32_t out_bf16, void* stream) {
  M3PC_REQUIRE(x && gamma && beta && y, "null argument");
  return m3pc::layernorm(x, M, gamma, beta, y, D, out_bf16 != 0, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_attention(const void* qkv, void* out, int32_t B, int32_t S, int32_t n_head, int32_t is_bf16, void* stream) {
  M3PC_REQUIRE(qkv && out, "null argument");
  return m3pc::launch_attention(qkv, out, B, S, n_head, is_bf16 != 0, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_attention_gather(const m3pc_attn_tok_t* q, int32_t n_q, const m3pc_attn_tok_t* k, const m3pc_attn_tok_t* v, int32_t n_kv,
                          int32_t n_kv_batch, int32_t B, int32_t n_head, void* out, int32_t is_bf16, int32_t* out_kernel, void* stream) {
  M3PC_REQUIRE(q && k && v && out, "null argument");
  M3PC_REQUIRE(n_q >= 1 && n_q <= m3pc::MAX_TOK && n_kv >= 1 && n_kv <= m3pc::MAX_TOK, "attention_gather: n_q and n_kv must be in [1, 64]");
  M3PC_REQUIRE(n_kv_batch >= 0 && n_kv_batch <= n_kv, "attention_gather: n_kv_batch must be in [0, n_kv]");
  M3PC_REQUIRE(B >= 1 && n_head >= 1 && static_cast<int64_t>(B) * n_head <= INT32_MAX, "attention_gather: bad B / n_head");
  M3PC_REQUIRE(reinterpret_cast<uintptr_t>(out) % 16 == 0, "attention_gather: out must be 16-byte aligned");
  const int align = is_bf16 ? 8 : 4;  // elements per 16-byte load: cp.async of bf16 rows, float4 of fp32 rows
  m3pc::AttnParams p{};
  const m3pc_attn_tok_t* const src[3] = {q, k, v};
  m3pc::AttnTok* const dst[3] = {p.q, p.k, p.v};
  for (int l = 0; l < 3; ++l)
    for (int i = 0; i < (l == 0 ? n_q : n_kv); ++i) {
      const m3pc_attn_tok_t& t = src[l][i];
      M3PC_REQUIRE(t.ptr != nullptr, "null token pointer");
      M3PC_REQUIRE(reinterpret_cast<uintptr_t>(t.ptr) % 16 == 0 && t.bstride >= 0 && t.bstride % align == 0 && t.bdiv >= 0,
                   "attention_gather: a token's ptr must be 16-byte aligned and its bstride a non-negative multiple of 16 bytes");
      dst[l][i] = m3pc::AttnTok{t.ptr, t.bstride, t.bdiv};
    }
  p.n_q = n_q;
  p.n_kv = n_kv;
  p.B = B;
  p.n_head = n_head;
  p.n_kv_batch = n_kv_batch;
  p.out = out;
  return m3pc::launch_attention_gather(p, is_bf16 != 0, reinterpret_cast<cudaStream_t>(stream), out_kernel);
}

// ---- kernel-level entries K1 / K4 / K5 / K6 / K7 / K8 (SURVEY.md section 8b): the same launchers m3pc_forward / m3pc_plan use ----
int m3pc_embed_gather(m3pc_handle_t h, int32_t batch, const float* tok_states, const float* tok_actions, const float* tok_rewards,
                      const float* tok_returns, const uint8_t* masks, float* x_out, void* y_out, void* stream) {
  M3PC_REQUIRE(tok_states && tok_actions && tok_rewards && tok_returns && x_out && y_out, "null argument");
  M3PC_REQUIRE(h != nullptr && h->finalized, "kernel-level call before m3pc_finalize_params");
  m3pc::FwdIO io{};
  M3PC_TRY(m3pc::io_from_tokens(h, io, tok_states, tok_actions, tok_rewards, tok_returns, masks));
  M3PC_REQUIRE(batch >= 1 && batch <= h->cfg.max_batch, "batch exceeds cfg.max_batch");
  const m3pc::TokTables tt = m3pc::token_tables(io.mask, h->T);
  M3PC_REQUIRE(tt.S > 0, "every token is masked");
  const m3pc::EmbedParams ep = m3pc::embed_params(h, io, tt, 0, batch);
  const m3pc::LayerW& first = h->enc.layers[0];
  return m3pc::launch_embed(ep, h->D, x_out, y_out, h->bf16, first.n1_w, first.n1_b, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_block_forward(m3pc_handle_t h, int32_t stack, int32_t layer, int32_t batch, int32_t n_tok, float* x, void* y_next, void* stream) {
  M3PC_REQUIRE(h != nullptr && h->finalized && x != nullptr, "bad argument");
  M3PC_REQUIRE(stack == 0 || stack == 1, "stack must be 0 (encoder) or 1 (decoder)");
  const m3pc::StackW& sw = stack == 0 ? h->enc : h->dec;
  const int n_layer = stack == 0 ? h->Le : h->Ld;
  M3PC_REQUIRE(layer >= 0 && layer < n_layer, "layer out of range");
  M3PC_REQUIRE(batch >= 1 && batch <= h->chunk && n_tok >= 1 && n_tok <= 4 * h->T, "batch exceeds the engine's chunk, or more tokens than 4T");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const size_t rows = static_cast<size_t>(batch) * n_tok, D = h->D, ab = m3pc::act_bytes(h);
  const m3pc::LayerW& w = sw.layers[layer];
  M3PC_CHECK_CUDA(cudaMemcpyAsync(h->X.p, x, rows * D * 4, cudaMemcpyDeviceToDevice, st));
  M3PC_TRY(m3pc::layernorm(h->X.as<float>(), static_cast<int>(rows), w.n1_w, w.n1_b, h->Y.p, h->D, h->bf16, st));
  m3pc::PostLn post;
  if (y_next != nullptr)
    post = layer + 1 < n_layer ? m3pc::PostLn{sw.layers[layer + 1].n1_w, sw.layers[layer + 1].n1_b, h->ENC.p} : m3pc::PostLn{sw.norm_w, sw.norm_b, h->ENC.p};
  M3PC_TRY(m3pc::block(h, w, batch, n_tok, st, post));
  M3PC_CHECK_CUDA(cudaMemcpyAsync(x, h->X.p, rows * D * 4, cudaMemcpyDeviceToDevice, st));
  if (y_next != nullptr) M3PC_CHECK_CUDA(cudaMemcpyAsync(y_next, h->ENC.p, rows * D * ab, cudaMemcpyDeviceToDevice, st));
  return M3PC_OK;
}

int m3pc_decoder_scatter_embed(m3pc_handle_t h, int32_t batch, const void* enc_out, const uint8_t* masks, float* x_out, void* stream) {
  M3PC_REQUIRE(h != nullptr && h->finalized && enc_out && masks && x_out, "bad argument");
  M3PC_REQUIRE(batch >= 1 && batch <= h->chunk, "batch exceeds the engine's chunk (workspace rows)");
  const int T = h->T;
  for (int i = 0; i < 4 * T; ++i) M3PC_REQUIRE(masks[i] <= 1, "mask entries must be 0 or 1");
  const m3pc::TokTables tt = m3pc::token_tables(masks, T);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  M3PC_TRY(m3pc::launch_fill_rows(m3pc::mask_rows(h, tt.dec_src, batch), h->D, x_out, st));  // no launch when every token is kept
  if (tt.S == 0) return M3PC_OK;
  return m3pc::decoder_embed(h, enc_out, tt.dec_src, batch, st, x_out);
}

int m3pc_heads(m3pc_handle_t h, int32_t batch, const float* x_dec, float* out_states, float* out_act_mu, float* out_act_std,
               float* out_rewards, float* out_returns, void* stream) {
  M3PC_REQUIRE(h != nullptr && h->finalized && x_dec, "bad argument");
  M3PC_REQUIRE(batch >= 1 && batch <= h->chunk, "batch exceeds the engine's chunk (workspace rows)");
  M3PC_REQUIRE((out_act_mu == nullptr) == (out_act_std == nullptr), "out_act_mu and out_act_std go together");
  m3pc::FwdIO io{};
  io.out_states = out_states; io.out_mu = out_act_mu; io.out_std = out_act_std; io.out_rewards = out_rewards; io.out_returns = out_returns;
  m3pc::NeedSet need;
  const float* outp[4] = {out_states, out_act_mu, out_rewards, out_returns};
  for (int k = 0; k < 4; ++k) need.nt[k] = outp[k] != nullptr ? h->T : 0;
  return m3pc::heads_all_rows(h, io, x_dec, need, 0, batch, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_sample_candidates(const float* mu, const float* std, const float* eps, uint64_t seed, int32_t n_cand, int32_t horizon, int32_t act_dim,
                           int32_t traj_length, int32_t noise_mode, int32_t cand_offset, float* out_candidates, void* stream) {
  M3PC_REQUIRE(mu && std && out_candidates, "null argument");
  M3PC_REQUIRE(n_cand >= 1 && horizon >= 1 && horizon <= traj_length && traj_length <= M3PC_MAX_T && act_dim >= 1 && act_dim <= M3PC_MAX_ACT,
               "shape out of range");
  M3PC_REQUIRE(noise_mode == 0 || noise_mode == 1, "noise_mode must be 0 (tanh(mu + std eps)) or 1 (clamp(tanh(mu) + 0.09 eps))");
  m3pc::CandParams cp{};
  cp.mu = mu; cp.std = std; cp.eps = eps; cp.cand = out_candidates;
  cp.N = n_cand; cp.h = horizon; cp.A = act_dim; cp.T = traj_length;
  cp.noise_mode = noise_mode; cp.seed = seed; cp.cand_offset = cand_offset;
  return m3pc::launch_candidates(cp, reinterpret_cast<cudaStream_t>(stream));
}

int m3pc_twinq(m3pc_handle_t h, const float* states_pred, const float* candidates, int32_t n_cand, int32_t horizon, float* out_q, void* stream) {
  M3PC_REQUIRE(h != nullptr && h->finalized && states_pred && candidates && out_q, "bad argument");
  M3PC_REQUIRE(h->has_critic, "no critic parameters were loaded");
  M3PC_REQUIRE(n_cand >= 1 && n_cand <= h->cfg.max_batch && horizon >= 1 && horizon <= h->T, "shape out of range");
  return m3pc::critic(h, n_cand, horizon, reinterpret_cast<cudaStream_t>(stream), states_pred, candidates, out_q);
}

int m3pc_score_select(const float* rewards_pred, const float* returns_pred, const float* qvals, const float* candidates, const float* expq,
                      const float* norm_stats, float discount, float lmbda, float temperature, int32_t n_cand, int32_t horizon,
                      int32_t traj_length, int32_t act_dim, uint64_t seed, int32_t cand_offset, float* out_J, float* out_eval_action,
                      float* out_sample_action, float* out_partials, int32_t* out_indices, void* stream) {
  M3PC_REQUIRE(rewards_pred && candidates && norm_stats && out_J && out_eval_action && out_sample_action, "null argument");
  M3PC_REQUIRE((returns_pred != nullptr) != (qvals != nullptr), "exactly one of returns_pred (rtg_guiding) and qvals (critic guidance) must be given");
  M3PC_REQUIRE(n_cand >= 1 && horizon >= 1 && horizon <= traj_length && traj_length <= M3PC_MAX_T && act_dim >= 1 && act_dim <= M3PC_MAX_ACT,
               "shape out of range");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  m3pc::ScoreParams sp{};
  sp.rewards_pred = rewards_pred; sp.returns_pred = returns_pred; sp.qvals = qvals;
  sp.rw_mean = norm_stats[0]; sp.rw_std = norm_stats[1]; sp.rt_mean = norm_stats[2]; sp.rt_std = norm_stats[3];
  sp.discount = discount; sp.lmbda = lmbda;
  sp.N = n_cand; sp.h = horizon; sp.T = traj_length; sp.J = out_J;
  M3PC_TRY(m3pc::launch_score(sp, st));
  m3pc::SelectParams sl{};
  sl.n_env = 1; sl.J = out_J; sl.cand = candidates; sl.expq = expq;
  sl.N = n_cand; sl.h = horizon; sl.A = act_dim;
  sl.temperature = temperature; sl.seed = seed; sl.cand_offset = cand_offset;
  sl.eval_action = out_eval_action; sl.sample_action = out_sample_action; sl.partials = out_partials; sl.indices = out_indices;
  return m3pc::launch_select(sl, st);
}

int m3pc_last_device_ms(m3pc_handle_t h, float* ms) {
  M3PC_REQUIRE(h != nullptr && ms != nullptr, "null argument");
  M3PC_CHECK_CUDA(cudaEventSynchronize(h->ev1));
  M3PC_CHECK_CUDA(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return M3PC_OK;
}

int m3pc_set_profile(m3pc_handle_t h, int32_t on) {
  M3PC_REQUIRE(h != nullptr, "null handle");
  h->profile = on != 0;
  h->prof_used = 0;
  return M3PC_OK;
}

int m3pc_get_profile(m3pc_handle_t h, double* gemm_ms, double* gemm_flops, int32_t* gemm_launches) {
  M3PC_REQUIRE(h != nullptr && gemm_ms && gemm_flops && gemm_launches, "null argument");
  double ms = 0.0, fl = 0.0;
  for (size_t i = 0; i < h->prof_used; ++i) {
    float t = 0.f;
    M3PC_CHECK_CUDA(cudaEventSynchronize(h->prof_events[i].second));
    M3PC_CHECK_CUDA(cudaEventElapsedTime(&t, h->prof_events[i].first, h->prof_events[i].second));
    ms += t;
    fl += h->prof_flops[i];
  }
  *gemm_ms = ms;
  *gemm_flops = fl;
  *gemm_launches = static_cast<int32_t>(h->prof_used);
  return M3PC_OK;
}

int m3pc_last_launch_count(m3pc_handle_t h, int32_t* n) {
  M3PC_REQUIRE(h != nullptr && n != nullptr, "null argument");
  *n = h->last_launches;
  return M3PC_OK;
}

}  // extern "C"
