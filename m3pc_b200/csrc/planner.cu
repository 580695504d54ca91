// K6..K8: the M^3PC candidate loop, kept on the device (no host round-trip inside a plan).
//
//   candidates_kernel   K6  sample N action sequences from the pass-1 tanh-Gaussian (learner.py:285-287) or add fixed
//                           variance noise to its mean (learner.py:156-167); injected noise for parity, Philox otherwise.
//   critic_input_kernel K7  decode predicted states, normalise for the critic, concatenate the action (model.py:163-168).
//   critic_out_kernel   K7  last TwinQ layer + min(q1, q2) (model.py:170-171).
//   score_kernel        K8  TD(lambda) return per candidate, written as the reference's loop (learner.py:301-316).
//   select_kernel       K8  softmax over candidates, weighted-mean action, exponential-race sample == torch.multinomial
//                           (learner.py:318-325); emits the per-shard record merged by merge_kernel under sharding.
#include <algorithm>

#include "kernels.cuh"

namespace m3pc {
namespace {

// ---- Philox4x32-10 (counter-based: results do not depend on how candidates are sharded) -------------------
struct U4 { unsigned x, y, z, w; };
__device__ __forceinline__ U4 philox4x32(U4 c, unsigned k0, unsigned k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}
__device__ __forceinline__ float u01(unsigned u) { return (static_cast<float>(u >> 8) + 0.5f) * (1.0f / 16777216.0f); }  // (0,1)
__device__ __forceinline__ float philox_normal(unsigned long long seed, unsigned gid, unsigned elem, unsigned stream) {
  const U4 r = philox4x32(U4{gid, elem >> 1, stream, 0u}, static_cast<unsigned>(seed), static_cast<unsigned>(seed >> 32));
  const float rad = sqrtf(-2.0f * logf(u01(r.x)));
  const float ang = 6.283185307179586f * u01(r.y);
  return (elem & 1) ? rad * sinf(ang) : rad * cosf(ang);
}
__device__ __forceinline__ float philox_exp(unsigned long long seed, unsigned gid, unsigned stream) {
  const U4 r = philox4x32(U4{gid, 0u, stream, 1u}, static_cast<unsigned>(seed), static_cast<unsigned>(seed >> 32));
  return -logf(u01(r.x));
}

__global__ void candidates_kernel(const __grid_constant__ CandParams p) {
  PDL_PROLOGUE();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per = p.h * p.A;
  if (i >= p.N * per) return;
  const int n = i / per, e = i - n * per, j = e / p.A, a = e - j * p.A;
  const unsigned long long seed = p.seed_ptr ? *p.seed_ptr : p.seed;
  int gid = p.cand_offset + n;
  if (p.env_id != nullptr) {  // key by the caller's environment index
    const int n_env_c = p.n_per_env > 0 ? p.n_per_env : p.N, le = n / n_env_c;
    gid = p.cand_offset + p.env_id[le] * n_env_c + (n - le * n_env_c);
  }
  const float eps = p.eps ? p.eps[i] : philox_normal(seed, static_cast<unsigned>(gid), static_cast<unsigned>(e), 0u);
  const int t = p.T - p.h + j;
  const int ms = ((p.n_per_env > 0 ? n / p.n_per_env : 0) * p.T + t) * p.A + a;  // pass-1 distribution of the candidate's environment
  const float mu = p.mu[ms];
  float v;
  if (p.noise_mode == 0) {
    v = tanhf(__fadd_rn(mu, __fmul_rn(p.std[ms], eps)));
  } else {
    v = __fadd_rn(tanhf(mu), __fmul_rn(eps, 0.09f));
    v = fminf(fmaxf(v, -0.99999f), 0.99999f);
  }
  p.cand[i] = v;
}

__global__ void critic_input_kernel(const __grid_constant__ CriticInParams p) {
  PDL_PROLOGUE();
  const int w = p.ld;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.N * p.h * w) return;
  const int row = i / w, c = i - row * w;
  const int n = row / p.h, t = row - n * p.h;
  float v = 0.f;  // zero padding beyond obs + A
  if (c < p.obs) {
    const float y = p.states_pred[(static_cast<size_t>(n) * p.T + (p.T - p.h + t)) * p.obs + c];
    const float s = __fadd_rn(__fmul_rn(y, p.tok_std[c]), p.tok_mean[c]);  // tokenizer decode, continuous.py:90-92
    v = (s - p.obs_mean[c]) / p.obs_std[c];                                 // TwinQ.both, model.py:166
  } else if (c < p.obs + p.A) {
    v = p.cand[(static_cast<size_t>(n) * p.h + t) * p.A + (c - p.obs)];
  }
  if (p.out_bf16)
    reinterpret_cast<__nv_bfloat16*>(p.sa)[i] = __float2bfloat16_rn(v);
  else
    reinterpret_cast<float*>(p.sa)[i] = v;
}

__global__ void critic_out_kernel(const float* __restrict__ h1, const float* __restrict__ h2, const float* __restrict__ w1,
                                  const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                                  float* __restrict__ q, int rows, int H) {
  PDL_PROLOGUE();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float s1 = 0.f, s2 = 0.f;
  for (int c = lane; c < H; c += 32) {
    s1 = fmaf(h1[static_cast<size_t>(row) * H + c], __ldg(w1 + c), s1);
    s2 = fmaf(h2[static_cast<size_t>(row) * H + c], __ldg(w2 + c), s2);
  }
  s1 = warp_sum(s1) + __ldg(b1);
  s2 = warp_sum(s2) + __ldg(b2);
  if (lane == 0) q[row] = fminf(s1, s2);
}

// TD(lambda) return of candidate n, written as the reference's loop (learner.py:301-316)
__device__ __forceinline__ float score_one(const ScoreParams& p, int n) {
  const int T = p.T, h = p.h;
  float disc[M3PC_MAX_T], r[M3PC_MAX_T];
  float d = 1.0f;
  for (int i = 0; i < h; ++i) {  // torch.cumprod(discount * ones(t+1)) in fp32
    d = __fmul_rn(d, p.discount);
    disc[i] = d;
    // rewards are consumed for steps < h-1 only (the last step contributes its value term); later rows are never written
    r[i] = (i < h - 1) ? __fadd_rn(__fmul_rn(p.rewards_pred[static_cast<size_t>(n) * T + (T - h + i)], p.rw_std), p.rw_mean) : 0.f;
  }
  const double lam = static_cast<double>(p.lmbda);
  const float one_minus = static_cast<float>(1.0 - lam);
  float J = 0.f;
  double lam_t = 1.0;
  for (int t = 0; t < h; ++t) {
    float v;
    if (p.qvals != nullptr) {
      v = p.qvals[static_cast<size_t>(n) * h + t];
    } else {
      const float y = p.returns_pred[static_cast<size_t>(n) * T + (T - h + t)];
      v = __fmul_rn(__fadd_rn(__fmul_rn(y, p.rt_std), p.rt_mean), 1000.0f);  // learner.py:305
    }
    float s = 0.f;
    for (int j = 0; j < t; ++j) s = __fadd_rn(s, __fmul_rn(r[j], disc[j]));
    s = __fadd_rn(s, __fmul_rn(v, disc[t]));
    const float lt = static_cast<float>(lam_t);
    if (t < h - 1)
      J = __fadd_rn(J, __fmul_rn(__fmul_rn(s, one_minus), lt));
    else
      J = __fadd_rn(J, __fmul_rn(s, lt));
    lam_t *= lam;
  }
  return J;
}

__global__ void score_kernel(const __grid_constant__ ScoreParams p) {
  PDL_PROLOGUE();
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.N) return;
  p.J[n] = score_one(p, n);
}

// ---- block reductions (1024 threads, deterministic order) ------------------------------------------------
constexpr int SEL_THREADS = 1024;

__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = (lane < SEL_THREADS / 32) ? red[lane] : 0.f;
  t = warp_sum(t);
  return t;  // every thread holds the total
}
// argmax with lowest-index tie break; returns value, index broadcast to all threads
__device__ __forceinline__ void block_argmax(float& v, int& idx, float* redv, int* redi) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) { redv[warp] = v; redi[warp] = idx; }
  __syncthreads();
  v = (lane < SEL_THREADS / 32) ? redv[lane] : -INFINITY;
  idx = (lane < SEL_THREADS / 32) ? redi[lane] : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
  }
}

// log-sum-exp merge of per-shard records (SURVEY.md 8e), by ONE thread; `ld` reads a record float (plain or cache-volatile)
template <typename Ld>
__device__ __forceinline__ void merge_records(Ld ld, int n_shards, int A, float temperature, float* eval_action, float* sample_action, int* indices) {
  float m = -INFINITY;
  for (int g = 0; g < n_shards; ++g) m = fmaxf(m, ld(g, 0));
  float Z = 0.f, kbest = -INFINITY, jbest = -INFINITY;
  int kg = 0, ji = 0;
  for (int g = 0; g < n_shards; ++g) {
    const float sc = expf((ld(g, 0) - m) * temperature);
    Z += ld(g, 1) * sc;
    const float key = ld(g, 4) * sc;
    if (key > kbest) { kbest = key; kg = g; }
    if (ld(g, 2) > jbest) { jbest = ld(g, 2); ji = __float_as_int(ld(g, 3)); }
  }
  for (int a = 0; a < A; ++a) {
    float U = 0.f;
    for (int g = 0; g < n_shards; ++g) U += ld(g, 8 + a) * expf((ld(g, 0) - m) * temperature);
    eval_action[a] = U / Z;
    sample_action[a] = ld(kg, 8 + A + a);
  }
  if (indices) {
    indices[0] = ji;
    indices[1] = __float_as_int(ld(kg, 5));
  }
}

__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__global__ void __launch_bounds__(SEL_THREADS) select_kernel(const __grid_constant__ SelectParams p) {
  PDL_PROLOGUE();
  __shared__ float redv[32];
  __shared__ int redi[32];
  __shared__ float rec[M3PC_PARTIAL_FLOATS];  // this shard's record (exchange mode)
  __shared__ int xch_failed;
  const int tid = threadIdx.x;
  const bool exchange = p.xch.world > 0;
  const int stride_a0 = p.h * p.A;
  const unsigned long long seed = p.seed_ptr ? *p.seed_ptr : p.seed;
  // one block per environment: this block's slice of every per-candidate array
  const int env = blockIdx.x, row0 = env * p.N;
  const int out_env = p.env_id ? p.env_id[env] : env;  // the caller's row of this environment
  const int grow0 = out_env * p.N;                     // Philox id of its candidate 0 (before cand_offset)
  const float* Jv = p.J + row0;
  const float* __restrict__ candv = p.cand + static_cast<size_t>(row0) * stride_a0;
  const float* __restrict__ expq = p.expq ? p.expq + row0 : nullptr;
  float* eval_action = p.eval_action + out_env * p.A;
  float* sample_action = p.sample_action + out_env * p.A;
  // 0. scores of this environment's candidates, when the score pass rides in this launch (p.score.J == p.J)
  if (p.score.J != nullptr) {
    for (int n = tid; n < p.N; n += SEL_THREADS) p.score.J[row0 + n] = score_one(p.score, row0 + n);
    __syncthreads();  // block-wide visibility of the global stores above
  }
  // 1. max_n J_n (+ argmax)
  float m = -INFINITY;
  int mi = 0x7fffffff;
  for (int n = tid; n < p.N; n += SEL_THREADS) {
    const float j = Jv[n];
    if (j > m) { m = j; mi = n; }
  }
  block_argmax(m, mi, redv, redi);
  // 2. w_n = exp((J_n - m) * tau); Z = sum w_n; sample key = w_n / q_n  (== p_n / q_n up to the constant Z)
  float z = 0.f, kbest = -INFINITY;
  int ki = 0x7fffffff;
  for (int n = tid; n < p.N; n += SEL_THREADS) {
    const float w = expf(__fmul_rn(__fsub_rn(Jv[n], m), p.temperature));
    z += w;
    const float q = expq ? expq[n] : philox_exp(seed, static_cast<unsigned>(p.cand_offset + grow0 + n), 1u);
    const float key = w / q;
    if (key > kbest) { kbest = key; ki = n; }
  }
  const float Z = block_sum(z, redv);
  block_argmax(kbest, ki, redv, redi);
  // non-finite scores (every comparison false): the indices are still the 0x7fffffff sentinels.  Never index with them --
  // report candidate 0 and NaN actions, which the host can test for (the reference raises from torch.multinomial instead).
  const bool bad_k = ki == 0x7fffffff;
  if (mi == 0x7fffffff) mi = 0;
  if (bad_k) ki = 0;
  const float nanv = __int_as_float(0x7fc00000);
  // 3. U[a] = sum w_n a0[n, a]
  for (int a = 0; a < p.A; ++a) {
    float u = 0.f;
    for (int n = tid; n < p.N; n += SEL_THREADS) {
      const float w = expf(__fmul_rn(__fsub_rn(Jv[n], m), p.temperature));
      u = fmaf(w, candv[static_cast<size_t>(n) * stride_a0 + a], u);
    }
    const float U = block_sum(u, redv);
    if (tid == 0) {
      const float sa = bad_k ? nanv : candv[static_cast<size_t>(ki) * stride_a0 + a];
      if (!exchange) {
        eval_action[a] = U / Z;
        sample_action[a] = sa;
      }
      rec[8 + a] = U;
      rec[8 + p.A + a] = sa;
    }
  }
  if (tid == 0) {
    rec[0] = m;
    rec[1] = Z;
    rec[2] = m;
    rec[3] = __int_as_float(p.cand_offset + mi);
    rec[4] = kbest;
    rec[5] = __int_as_float(p.cand_offset + ki);
    rec[6] = static_cast<float>(p.N);
    rec[7] = 0.f;
    if (p.indices && !exchange) {
      p.indices[2 * out_env + 0] = p.cand_offset + mi;
      p.indices[2 * out_env + 1] = p.cand_offset + ki;
    }
    xch_failed = 0;
  }
  __syncthreads();
  const int n_rec = 8 + 2 * p.A;
  if (p.partials)
    for (int f = tid; f < n_rec; f += SEL_THREADS) p.partials[f] = rec[f];
  if (!exchange) return;

  // ---- all-gather of the records over peer memory + merge (one block: n_env == 1) ----
  const ExchangeParams& x = p.xch;
  const unsigned long long ep = *x.epoch + 1ull;  // epochs start at 1: the flags are zero-initialised
  const int slot = static_cast<int>(ep & 1ull);
  for (int i = tid; i < x.world * n_rec; i += SEL_THREADS) {
    const int g = i / n_rec, f = i - g * n_rec;
    float* dst = reinterpret_cast<float*>(x.peer[g]) + (static_cast<size_t>(slot) * XCH_MAX_RANKS + x.rank) * M3PC_PARTIAL_FLOATS + f;
    __stcg(dst, rec[f]);  // peer-mapped (NVLink) or local global memory
  }
  __threadfence_system();  // every thread's record stores are visible system-wide before the flag is
  __syncthreads();
  if (tid < x.world) {
    unsigned long long* pf = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(x.peer[tid]) + XCH_FLAG_OFFSET) + slot * XCH_MAX_RANKS + x.rank;
    st_release_sys_u64(pf, ep);
    const unsigned long long* mf = reinterpret_cast<const unsigned long long*>(reinterpret_cast<const char*>(x.peer[x.rank]) + XCH_FLAG_OFFSET) + slot * XCH_MAX_RANKS + tid;
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys_u64(mf) < ep) {
      if (global_timer_ns() - t0 > x.timeout_ns) {  // a peer never arrived: fail loudly instead of hanging the GPU
        xch_failed = 1;
        break;
      }
      __nanosleep(64);
    }
  }
  __syncthreads();
  if (tid == 0) {
    if (xch_failed) {
      *reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(x.peer[x.rank]) + XCH_ERR_OFFSET) = ep;
      for (int a = 0; a < p.A; ++a) eval_action[a] = sample_action[a] = nanv;
    } else {
      const float* base = reinterpret_cast<const float*>(x.peer[x.rank]) + static_cast<size_t>(slot) * XCH_MAX_RANKS * M3PC_PARTIAL_FLOATS;
      // cache-volatile loads: the lines were written by peers through NVLink, L1 may still hold the slot's previous contents
      merge_records([base](int g, int f) { return __ldcv(base + g * M3PC_PARTIAL_FLOATS + f); }, x.world, p.A, p.temperature, eval_action,
                    sample_action, p.indices);
    }
    *x.epoch = ep;
  }
}

// merge of records gathered by another transport (e.g. an NCCL all-gather of out_partials): m3pc_merge_partials
__global__ void merge_kernel(const float* __restrict__ partials, int n_shards, int A, float temperature, float* eval_action,
                             float* sample_action, int* indices) {
  PDL_PROLOGUE();
  if (threadIdx.x != 0) return;
  merge_records([partials](int g, int f) { return partials[g * M3PC_PARTIAL_FLOATS + f]; }, n_shards, A, temperature, eval_action, sample_action,
                indices);
}

__global__ void set_seed_kernel(unsigned long long* dst, unsigned long long seed) { *dst = seed; }

// C draws per environment: i = (e * C + c) * A + a.  C = 1 is the reference's single draw (zeroshot_omtm/learner.py:136-147).
__global__ void sampling_tail_kernel(const float* __restrict__ mu, const float* __restrict__ std, const float* __restrict__ eps, int T, int h,
                                     int A, int E, int C, float* eval_action, float* sample_action, unsigned long long seed,
                                     const unsigned long long* seed_ptr, const int* __restrict__ env_id, bool eps_at_env_id) {
  PDL_PROLOGUE();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= E * C * A) return;
  if (seed_ptr) seed = *seed_ptr;
  const int a = i % A, c = (i / A) % C, e = i / (A * C);
  const int oe = env_id ? env_id[e] : e;  // the caller's row of environment e
  const size_t src = (static_cast<size_t>(e) * T + (T - h)) * A + a;
  const float m = mu[src];
  const size_t ei = eps_at_env_id ? (static_cast<size_t>(oe) * C + c) * A + a : static_cast<size_t>(i);
  const float z = eps ? eps[ei] : philox_normal(seed, static_cast<unsigned>(oe), static_cast<unsigned>(c * A + a), 2u);
  if (c == 0) eval_action[oe * A + a] = tanhf(m);
  sample_action[(static_cast<size_t>(oe) * C + c) * A + a] = tanhf(__fadd_rn(m, __fmul_rn(std[src], z)));
}

__global__ void piid_fill_kernel(const float* __restrict__ win_states, const float* __restrict__ states_pred, const float* __restrict__ tok_mean,
                                 const float* __restrict__ tok_std, float* __restrict__ filled, int E, int T, int h, int obs) {
  PDL_PROLOGUE();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= E * T * obs) return;
  const int c = i % obs, t = (i / obs) % T;
  // zeroshot_omtm/learner.py:240-246: [T-h+2, T-1) and [0, T-h+1) come from the path-inference pass
  const bool from_pred = (t < T - h + 1) || (t >= T - h + 2 && t < T - 1);
  filled[i] = from_pred ? __fadd_rn(__fmul_rn(states_pred[i], tok_std[c]), tok_mean[c]) : win_states[i];
}

// ---- device-resident episode ring (row = [obs | act | reward]), one clock per slot: a slot list (and the horizons of its windows)
// travels as a kernel parameter ----
constexpr int RING_MAX_SLOTS = 256;  // per launch; the launchers split longer lists
struct RingSlots {
  int n;
  int slot[RING_MAX_SLOTS];
  unsigned char h[RING_MAX_SLOTS];
};

__global__ void ring_reset_kernel(float* __restrict__ ring, int L, int w, const __grid_constant__ RingSlots s) {
  PDL_PROLOGUE();
  const size_t per = static_cast<size_t>(L) * w;
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= per * s.n) return;
  const int k = static_cast<int>(i / per);
  ring[static_cast<size_t>(s.slot[k]) * per + (i - k * per)] = 0.f;
}

// listed slot k writes its observation (o row k) at step t[slot] and, when given, the action / reward of step t[slot] - 1
__global__ void ring_append_slots_kernel(float* __restrict__ ring, int L, int obs, int act, const int* __restrict__ tt, const __grid_constant__ RingSlots s,
                                         const float* __restrict__ o, const float* __restrict__ pa, const float* __restrict__ pr) {
  PDL_PROLOGUE();
  const int w = obs + act + 1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= s.n * w) return;
  const int k = i / w, c = i - k * w, e = s.slot[k];
  const int t = tt[e];
  if (t < 0 || t >= L) return;  // an idle slot (clock < 0) or a step outside the ring: nothing to record
  float* row_t = ring + (static_cast<size_t>(e) * L + t) * w;
  if (c < obs) {
    row_t[c] = o[k * obs + c];
  } else if (t > 0) {
    float* row_p = row_t - w;
    if (c < obs + act) {
      if (pa != nullptr) row_p[c] = pa[k * act + (c - obs)];
    } else if (pr != nullptr) {
      row_p[c] = pr[k];
    }
  }
}

// observation c of row first + r of listed slot k = rows[k, r, c]; the action and reward columns are left as they are
__global__ void ring_write_obs_kernel(float* __restrict__ ring, int L, int obs, int act, int first, int n_rows, const __grid_constant__ RingSlots s,
                                      const float* __restrict__ rows) {
  PDL_PROLOGUE();
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t per = static_cast<size_t>(n_rows) * obs;
  if (i >= per * s.n) return;
  const int k = static_cast<int>(i / per), r = static_cast<int>((i - k * per) / obs), c = static_cast<int>(i % obs);
  ring[(static_cast<size_t>(s.slot[k]) * L + first + r) * (obs + act + 1) + c] = rows[i];
}

// element c of time step t of window k: listed slot e = slots[k] at its step pl[e] with horizon h[k]
__global__ void ring_windows_slots_kernel(const float* __restrict__ ring, int L, int obs, int act, const int* __restrict__ pl, int T, int future_obs,
                                          const __grid_constant__ RingSlots s, const float* __restrict__ rtg_tok, float* __restrict__ ws,
                                          float* __restrict__ wa, float* __restrict__ wr, float* __restrict__ wt) {
  PDL_PROLOGUE();
  const int w = obs + act + 1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= s.n * T * w) return;
  const int c = i % w, t = (i / w) % T, k = i / (w * T), e = s.slot[k];
  const int p = pl[e], h = s.h[k];
  const int hl = T - h + 1, lo = p - hl + 1;  // learner.py:346-359
  int smart_T = T;                            // zeroshot_omtm/learner.py:77-79
  if (future_obs && p + h > 1000) smart_T = T - (p + h - 1000);
  const int step = lo + t;
  const bool in_ring = step >= 0 && step < L;
  const float* row = ring + (static_cast<size_t>(e) * L + (in_ring ? step : 0)) * w;
  if (c < obs) {
    const bool take = future_obs ? (t < smart_T || t < hl) : (t < hl);
    ws[(static_cast<size_t>(k) * T + t) * obs + c] = (take && in_ring) ? row[c] : 0.f;
  } else if (c < obs + act) {
    wa[(static_cast<size_t>(k) * T + t) * act + (c - obs)] = (t < hl && in_ring) ? row[c] : 0.f;
  } else {
    wr[k * T + t] = (t < hl && in_ring) ? row[c] : 0.f;
    wt[k * T + t] = rtg_tok[k];
  }
}

// ---- mixed-horizon plans: every horizon class's windows, noise rows and id table, gathered in one launch ----
__global__ void mix_gather_kernel(const __grid_constant__ MixGatherParams p) {
  PDL_PROLOGUE();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.y == 0) {  // windows: per step [states | actions | reward | return token]
    const int w = p.obs + p.A + 2;
    if (i >= p.E * p.T * w) return;
    const int s = i / (p.T * w), r = i - s * p.T * w, t = r / w, c = r - t * w;
    const size_t src = static_cast<size_t>(p.src[s]) * p.T + t, dst = static_cast<size_t>(s) * p.T + t;
    if (c < p.obs)
      p.gs[dst * p.obs + c] = p.ws[src * p.obs + c];
    else if (c < p.obs + p.A)
      p.ga[dst * p.A + (c - p.obs)] = p.wa[src * p.A + (c - p.obs)];
    else if (c == p.obs + p.A)
      p.gr[dst] = p.wr[src];
    else
      p.gt[dst] = p.wt[src];
  } else if (blockIdx.y == 1) {  // injected noise: the first h_e steps of each of environment e's rows
    const int per = p.eps_rows * p.eps_ld;
    if (p.eps == nullptr || i >= p.E * per) return;
    const int e = i / per, r = (i - e * per) / p.eps_ld, c = i - e * per - r * p.eps_ld, s = p.slot_of[e];
    const int wdt = (p.eps_off[s + 1] - p.eps_off[s]) / p.eps_rows;
    if (c < wdt) p.geps[p.eps_off[s] + r * wdt + c] = p.eps[i];
  } else {  // Exp(1) draws and the id table
    if (i < p.E) p.env_id[i] = p.src[i];
    if (p.expq == nullptr || i >= p.E * p.N) return;
    const int e = i / p.N;
    p.gexpq[p.slot_of[e] * p.N + (i - e * p.N)] = p.expq[i];
  }
}

}  // namespace

template <typename Fn>
int for_slot_chunks(const int* slots, const int* horizons, int n, int E, int T, Fn&& launch) {
  for (int k0 = 0; k0 < n; k0 += RING_MAX_SLOTS) {
    RingSlots s{};
    s.n = std::min(RING_MAX_SLOTS, n - k0);
    for (int k = 0; k < s.n; ++k) {
      M3PC_REQUIRE(slots[k0 + k] >= 0 && slots[k0 + k] < E, "ring: slot index out of range");
      if (horizons) {
        M3PC_REQUIRE(horizons[k0 + k] >= 1 && horizons[k0 + k] <= T, "ring: horizon out of range");
        s.h[k] = static_cast<unsigned char>(horizons[k0 + k]);
      }
      s.slot[k] = slots[k0 + k];
    }
    M3PC_TRY(launch(s, k0));
  }
  return M3PC_OK;
}

int launch_ring_reset(float* ring, int E, int L, int obs, int act, const int* slots, int n, cudaStream_t st) {
  M3PC_REQUIRE(ring && E >= 1 && L >= 1 && obs >= 1 && act >= 1 && n >= 0 && (n == 0 || slots), "ring_reset: bad shape");
  const int w = obs + act + 1;
  M3PC_REQUIRE(static_cast<long>(L) * w <= 0x7fffffffL / RING_MAX_SLOTS, "ring_reset: ring too long");
  return for_slot_chunks(slots, nullptr, n, E, 1, [&](const RingSlots& s, int) {
    M3PC_CHECK_CUDA(launch_k(ring_reset_kernel, dim3(ceil_div(s.n * L * w, 256)), dim3(256), 0, st, ring, L, w, s));
    M3PC_CHECK_LAUNCH();
    return M3PC_OK;
  });
}
int launch_ring_append_slots(float* ring, int E, int L, int obs, int act, const int* t, const int* slots, int n, const float* o, const float* pa,
                             const float* pr, cudaStream_t st) {
  M3PC_REQUIRE(ring && t && o && E >= 1 && L >= 1 && obs >= 1 && act >= 1 && n >= 0 && (n == 0 || slots), "ring_append_slots: bad shape");
  const int w = obs + act + 1;
  return for_slot_chunks(slots, nullptr, n, E, 1, [&](const RingSlots& s, int k0) {
    M3PC_CHECK_CUDA(launch_k(ring_append_slots_kernel, dim3(ceil_div(s.n * w, 128)), dim3(128), 0, st, ring, L, obs, act, t, s, o + static_cast<size_t>(k0) * obs,
                             pa ? pa + static_cast<size_t>(k0) * act : nullptr, pr ? pr + k0 : nullptr));
    M3PC_CHECK_LAUNCH();
    return M3PC_OK;
  });
}
int launch_ring_write_obs(float* ring, int E, int L, int obs, int act, const int* slots, int n, int first, int n_rows, const float* rows,
                          cudaStream_t st) {
  M3PC_REQUIRE(ring && E >= 1 && L >= 1 && obs >= 1 && act >= 1 && n >= 0 && (n == 0 || slots), "ring_write_obs: bad shape");
  M3PC_REQUIRE(first >= 0 && n_rows >= 0 && first + static_cast<long>(n_rows) <= L, "ring_write_obs: rows outside the ring");
  M3PC_REQUIRE(n_rows == 0 || n == 0 || rows, "ring_write_obs: null rows");
  if (n_rows == 0) return M3PC_OK;
  return for_slot_chunks(slots, nullptr, n, E, 1, [&](const RingSlots& s, int k0) {
    const size_t cnt = static_cast<size_t>(s.n) * n_rows * obs;
    M3PC_CHECK_CUDA(launch_k(ring_write_obs_kernel, dim3(static_cast<unsigned>((cnt + 255) / 256)), dim3(256), 0, st, ring, L, obs, act,
                             first, n_rows, s, rows + static_cast<size_t>(k0) * n_rows * obs));
    M3PC_CHECK_LAUNCH();
    return M3PC_OK;
  });
}
int launch_ring_windows_slots(const float* ring, int E, int L, int obs, int act, const int* pl, const int* slots, const int* horizons, int n,
                              int T, int future_obs, const float* rtg_tok, float* ws, float* wa, float* wr, float* wt, cudaStream_t st) {
  M3PC_REQUIRE(ring && pl && rtg_tok && ws && wa && wr && wt && horizons && E >= 1 && L >= 1 && n >= 0 && (n == 0 || slots) && T >= 1 &&
                   T <= M3PC_MAX_T,
               "ring_windows_slots: bad shape");
  const int w = obs + act + 1;
  return for_slot_chunks(slots, horizons, n, E, T, [&](const RingSlots& s, int k0) {
    const size_t o = static_cast<size_t>(k0) * T;
    M3PC_CHECK_CUDA(launch_k(ring_windows_slots_kernel, dim3(ceil_div(s.n * T * w, 256)), dim3(256), 0, st, ring, L, obs, act, pl, T, future_obs, s,
                             rtg_tok + k0, ws + o * obs, wa + o * act, wr + o, wt + o));
    M3PC_CHECK_LAUNCH();
    return M3PC_OK;
  });
}
int launch_mix_gather(const MixGatherParams& p, cudaStream_t st) {
  M3PC_REQUIRE(p.E >= 1 && p.E <= MIX_MAX_ENV, "mixed horizons: too many environments");
  const int n = std::max({p.E * p.T * (p.obs + p.A + 2), p.eps ? p.E * p.eps_rows * p.eps_ld : 0, p.E * p.N});
  M3PC_CHECK_CUDA(launch_k(mix_gather_kernel, dim3(ceil_div(n, 256), 3), dim3(256), 0, st, p));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}

int launch_candidates(const CandParams& p, cudaStream_t st) {
  const int n = p.N * p.h * p.A;
  M3PC_CHECK_CUDA(launch_k(candidates_kernel, dim3(ceil_div(n, 256)), dim3(256), 0, st, p));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}
int launch_critic_input(const CriticInParams& p, cudaStream_t st) {
  const int n = p.N * p.h * p.ld;
  M3PC_CHECK_CUDA(launch_k(critic_input_kernel, dim3(ceil_div(n, 256)), dim3(256), 0, st, p));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}
int launch_critic_out(const float* h1, const float* h2, const float* w1, const float* b1, const float* w2, const float* b2, float* q,
                      int rows, int H, cudaStream_t st) {
  M3PC_CHECK_CUDA(launch_k(critic_out_kernel, dim3(ceil_div(rows, 8)), dim3(256), 0, st, h1, h2, w1, b1, w2, b2, q, rows, H));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}
int launch_score(const ScoreParams& p, cudaStream_t st) {
  M3PC_REQUIRE(p.h >= 1 && p.h <= M3PC_MAX_T, "score: bad horizon");
  M3PC_CHECK_CUDA(launch_k(score_kernel, dim3(ceil_div(p.N, 128)), dim3(128), 0, st, p));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}
int launch_select(const SelectParams& p, cudaStream_t st) {
  M3PC_REQUIRE(p.A <= M3PC_MAX_ACT && p.N >= 1 && p.n_env >= 1, "select: bad shape");
  M3PC_REQUIRE(p.score.J == nullptr || (p.score.J == p.J && p.score.h >= 1 && p.score.h <= M3PC_MAX_T && p.score.N == p.N * p.n_env),
               "select: the fused score pass must write the scores this launch selects from");
  M3PC_REQUIRE(p.n_env == 1 || (p.partials == nullptr && p.xch.world == 0), "select: per-shard records are single-environment only");
  M3PC_REQUIRE(p.xch.world >= 0 && p.xch.world <= XCH_MAX_RANKS, "select: too many ranks");
  M3PC_CHECK_CUDA(launch_k(select_kernel, dim3(p.n_env), dim3(SEL_THREADS), 0, st, p));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}
int launch_merge(const float* partials, int n_shards, int A, float temperature, float* eval_action, float* sample_action, int* indices,
                 cudaStream_t st) {
  M3PC_CHECK_CUDA(launch_k(merge_kernel, dim3(1), dim3(32), 0, st, partials, n_shards, A, temperature, eval_action, sample_action, indices));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}
int launch_sampling_tail(const float* mu, const float* std, const float* eps, int T, int h, int A, int E, float* eval_action,
                         float* sample_action, unsigned long long seed, const unsigned long long* seed_ptr, cudaStream_t st, int C,
                         const int* env_id, bool eps_at_env_id) {
  M3PC_REQUIRE(C >= 1, "sampling tail: n_draws must be >= 1");
  M3PC_REQUIRE(env_id || !eps_at_env_id, "sampling tail: eps rows by environment id need the id table");
  M3PC_CHECK_CUDA(launch_k(sampling_tail_kernel, dim3(ceil_div(E * C * A, 128)), dim3(128), 0, st, mu, std, eps, T, h, A, E, C, eval_action, sample_action, seed, seed_ptr,
                           env_id, eps_at_env_id));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}
int launch_set_seed(unsigned long long* dst, unsigned long long seed, cudaStream_t st) {
  M3PC_CHECK_CUDA(launch_k(set_seed_kernel, dim3(1), dim3(1), 0, st, dst, seed));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}
int launch_piid_fill(const float* win_states, const float* states_pred, const float* tok_mean, const float* tok_std, float* filled, int E,
                     int T, int h, int obs, cudaStream_t st) {
  M3PC_CHECK_CUDA(launch_k(piid_fill_kernel, dim3(ceil_div(E * T * obs, 256)), dim3(256), 0, st, win_states, states_pred, tok_mean, tok_std, filled, E, T, h, obs));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}

}  // namespace m3pc
