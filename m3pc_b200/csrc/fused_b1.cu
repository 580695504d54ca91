// Fused B = 1 forward: the whole MTM encoder + restricted single-layer decoder for ONE batch row in ONE persistent
// cooperative kernel (grid = #SMs, software grid barrier between phases).
//
// Why: pass 1 of every M^3PC plan (Learner.rtg_guiding / critic_lambda_guiding, finetune_omtm/learner.py:278-284) and the
// zero-shot planners at E = 1 (zeroshot_omtm/learner.py:60-261) run omtm.forward at B = 1: 8..23 token rows through ~30
// dependent kernels of a few microseconds of work each, i.e. pure launch latency (190 us of an 810 us plan, profiles/r1a_*).
// Here the ~11 M weights are streamed exactly once by all SMs together; a phase is a skinny GEMM whose output columns are
// spread over every warp of the grid (activation rows staged in shared memory, weight rows read with 16-byte loads, fp32
// accumulation), and phases are separated by a ~1 us grid barrier instead of a kernel boundary.
//
// Numerics follow the multi-kernel bf16 path: fp32 residual stream and LayerNorm statistics, bf16 GEMM operands
// (LayerNorm outputs, attention outputs, GELU outputs), fp32 accumulation, fp32 softmax.
#include <algorithm>
#include <cstdlib>

#include "kernels.cuh"

namespace m3pc {
namespace {

constexpr int FB_THREADS = 256;
constexpr int FB_WARPS = FB_THREADS / 32;
constexpr int FB_APAD = 32;  // bf16 elements of row padding in a_s: rows g and g + 1 land on disjoint bank halves

// ---- grid barrier: bar[0] counts arrivals monotonically within a launch (barrier k completes at (k + 1) * G), bar[1] counts CTAs
// that have finished; the last one to finish resets both, so every launch starts from zero.  One release-add plus acquire-polls
// per CTA and barrier (no reset / generation round trip inside the barrier).
__device__ __forceinline__ void grid_sync(unsigned* bar, unsigned& target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    target += gridDim.x;
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(bar) : "memory");
    unsigned v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
    } while (v < target);
  }
  __syncthreads();
}
__device__ __forceinline__ void grid_finish(unsigned* bar) {
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(bar + 1, 1u) == gridDim.x - 1) {  // everyone is past the last barrier: nobody polls bar[0] any more
    atomicExch(bar, 0u);
    atomicExch(bar + 1, 0u);
  }
}

__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

// a_s[r][0:D] = bf16(LayerNorm(x[r]; gamma, beta)) for r < R, x fp32 (R, D) in global memory (written by other CTAs: L2 loads)
template <int NJ>
__device__ __forceinline__ void ln_rows_to_smem(const float* x, int R, const float* gamma, const float* beta, __nv_bfloat16* a_s, int lda) {
  constexpr int D = NJ * 128;
  constexpr int RB = NJ <= 4 ? 2 : 1;  // rows whose loads are in flight together (register budget)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int rb = warp; rb < R; rb += RB * FB_WARPS) {
    float4 v[RB][NJ];
#pragma unroll
    for (int i = 0; i < RB; ++i) {
      const int r = rb + i * FB_WARPS;
      if (r < R) {
#pragma unroll
        for (int j = 0; j < NJ; ++j) v[i][j] = ldcg4(x + static_cast<size_t>(r) * D + j * 128 + lane * 4);
      }
    }
#pragma unroll
    for (int i = 0; i < RB; ++i) {
      const int r = rb + i * FB_WARPS;
      if (r < R) {
        float4 o[NJ];
        warp_layernorm<NJ>(v[i], gamma, beta, lane, o);
#pragma unroll
        for (int j = 0; j < NJ; ++j) *reinterpret_cast<uint2*>(a_s + static_cast<size_t>(r) * lda + j * 128 + lane * 4) = f4_to_bf4(o[j]);
      }
    }
  }
}

// a_s[r][0:K] = A[r][0:K] (bf16, global, written by other CTAs)
__device__ __forceinline__ void copy_rows_to_smem(const __nv_bfloat16* A, int R, int K, __nv_bfloat16* a_s) {
  const int cpr = K / 8, chunks = R * cpr, lda = K + FB_APAD;
  const uint32_t base = smem_u32(a_s);
  for (int i = threadIdx.x; i < chunks; i += FB_THREADS) {  // cp.async.cg: L2 -> shared memory, every chunk in flight at once
    const int r = i / cpr, cc = i - r * cpr;
    cp_async16(base + 2u * static_cast<uint32_t>(r * lda + cc * 8), reinterpret_cast<const uint4*>(A) + i);
  }
  cp_async_commit();
  cp_async_wait_all();
}

// Skinny GEMM phase on tensor cores (mma.sync.m16n8k16, bf16 in, fp32 accumulate):
//   out(m, n) = sum_k a_s[m][k] * W[n][k]   for rows r0 <= m < r1 (at most 32 = two m16 tiles) and every column n < N.
// Work item = 8 output columns, handed out round-robin over the CTAs; the 8 warps of a CTA split K between them and combine their
// partial tiles through shared memory in a fixed order (deterministic).  The weight slab of an item is read exactly once, with
// 16-byte loads issued before anything else so that the L2 / HBM round trip overlaps the caller's activation prologue.
// K permutation: lane (g = lane / 4, q = lane % 4) loads the 8 consecutive k values k0 + 8q .. k0 + 8q + 7 of W row n0 + g and
// of A rows g / g + 8; the first mma consumes elements {0,1 | 2,3} of that run as its (k = 2q, 2q+1 | 2q+8, 2q+9) fragments, the
// second {4,5 | 6,7}.  A and B use the same permutation, so the dot products are unchanged.

struct WSlab {
  uint4 w[8];  // this lane's share of the item's weight slab: up to 8 k-steps of 32
};

// issue the weight loads of work item `item` (columns 8*item .. 8*item+7) for this warp's K slice
__device__ __forceinline__ void wslab_load(WSlab& ws, const __nv_bfloat16* __restrict__ W, int K, int item, int lane, int warp) {
  const int g = lane >> 2, q = lane & 3;
  const int kper = K / FB_WARPS;  // multiple of 32 (K is a multiple of 256)
  const __nv_bfloat16* wp = W + static_cast<size_t>(item * 8 + g) * K + warp * kper + q * 8;
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i * 32 < kper) ws.w[i] = __ldg(reinterpret_cast<const uint4*>(wp + i * 32));
}

template <class Epi>
__device__ __forceinline__ void rows_gemm(const __nv_bfloat16* a_s, int lda, int r0, int r1, int K, const __nv_bfloat16* __restrict__ W, int N,
                                          const float* __restrict__ bias, const float* res, int ldr, float* red, WSlab& ws, bool ws_loaded,
                                          Epi epi) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, q = lane & 3;
  const int G = gridDim.x, R = r1 - r0;
  const int kper = K / FB_WARPS;
  // reduction role of this thread: output (row = tr, column = tc) of the item's 32 x 8 tile
  const int tr = threadIdx.x >> 3, tc = threadIdx.x & 7;
  for (int item = blockIdx.x; item < N / 8; item += G) {
    if (!ws_loaded) wslab_load(ws, W, K, item, lane, warp);
    ws_loaded = false;
    const int n = item * 8 + tc;
    const float e_bias = bias != nullptr ? __ldg(bias + n) : 0.f;
    const float e_res = (res != nullptr && tr < R) ? __ldcg(res + static_cast<size_t>(r0 + tr) * ldr + n) : 0.f;
    float c[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    const __nv_bfloat16* ap = a_s + static_cast<size_t>(r0) * lda + warp * kper + q * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i * 32 < kper) {
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          const int ra = mt * 16 + g, rb = ra + 8;
          if (mt * 16 < R) {  // warp-uniform
            const uint4 lo = ra < R ? *reinterpret_cast<const uint4*>(ap + static_cast<size_t>(ra) * lda + i * 32) : make_uint4(0, 0, 0, 0);
            const uint4 hi = rb < R ? *reinterpret_cast<const uint4*>(ap + static_cast<size_t>(rb) * lda + i * 32) : make_uint4(0, 0, 0, 0);
            const uint32_t a0[4] = {lo.x, hi.x, lo.y, hi.y}, a1[4] = {lo.z, hi.z, lo.w, hi.w};
            mma_bf16_16816(c[mt], a0, ws.w[i].x, ws.w[i].y);
            mma_bf16_16816(c[mt], a1, ws.w[i].z, ws.w[i].w);
          }
        }
      }
    }
    // partial tiles -> shared memory: red[warp][row 0..31][col 0..7]
    __syncthreads();  // the previous item's reduction has been read
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      float* rp = red + (warp * 32 + mt * 16 + g) * 8 + 2 * q;
      *reinterpret_cast<float2*>(rp) = make_float2(c[mt][0], c[mt][1]);
      *reinterpret_cast<float2*>(rp + 64) = make_float2(c[mt][2], c[mt][3]);
    }
    __syncthreads();
    if (tr < R) {
      float v = 0.f;
#pragma unroll
      for (int w8 = 0; w8 < FB_WARPS; ++w8) v += red[(w8 * 32 + tr) * 8 + tc];
      epi(r0 + tr, n, v + e_bias, e_res);
    }
  }
}

// One (query row, head) pair per warp.  Scores: lane j owns key j (and j + 32): it dots the whole 128-wide head slice, so there is
// no per-key shuffle reduction and all of a lane's loads are independent.  P V: lane owns 4 of the 128 head dims.
// q / k / v are accessors returning a pointer to the bf16 head slice of a row; scores and softmax in fp32.
template <class QF, class KF, class VF>
__device__ __forceinline__ void attend_pair(QF qf, KF kf, VF vf, int n_kv, int lane, float4& out) {
  const float scale = 0.08838834764831845f;  // 1 / sqrt(128)
  const uint4* qp = reinterpret_cast<const uint4*>(qf());
  float sc[2] = {-INFINITY, -INFINITY};
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int j = lane + 32 * half;
    if (32 * half < n_kv) {  // warp-uniform
      const uint4* kp = reinterpret_cast<const uint4*>(kf(j < n_kv ? j : 0));
      uint4 kr[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) kr[i] = __ldcg(kp + i);
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float qv[8], kv[8];
        bf16x8_to_float(__ldcg(qp + i), qv);  // same address in every lane: one broadcast transaction
        bf16x8_to_float(kr[i], kv);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc = fmaf(qv[e], kv[e], acc);
      }
      if (j < n_kv) sc[half] = acc * scale;
    }
  }
  const float mx = warp_max(fmaxf(sc[0], sc[1]));
  const float e0 = sc[0] == -INFINITY ? 0.f : expf(sc[0] - mx), e1 = sc[1] == -INFINITY ? 0.f : expf(sc[1] - mx);
  const float inv = 1.0f / warp_sum(e0 + e1);
  out = make_float4(0.f, 0.f, 0.f, 0.f);
  constexpr int KB = 16;  // value rows whose loads are in flight together
  for (int j0 = 0; j0 < n_kv; j0 += KB) {
    uint2 vr[KB];
#pragma unroll
    for (int i = 0; i < KB; ++i)
      if (j0 + i < n_kv) vr[i] = __ldcg(reinterpret_cast<const uint2*>(vf(j0 + i)) + lane);
#pragma unroll
    for (int i = 0; i < KB; ++i) {
      const int j = j0 + i;
      if (j < n_kv) {
        const float pj = __shfl_sync(0xffffffffu, (j >> 5) ? e1 : e0, j & 31) * inv;
        const float4 v = bf4_to_f4(vr[i]);
        out.x = fmaf(pj, v.x, out.x); out.y = fmaf(pj, v.y, out.y); out.z = fmaf(pj, v.z, out.z); out.w = fmaf(pj, v.w, out.w);
      }
    }
  }
}

template <int NJ>
__global__ void __launch_bounds__(FB_THREADS, 1) fused_b1_kernel(const __grid_constant__ FusedB1Params p) {
  constexpr int D = NJ * 128, F = 4 * D, H = D / 128;
  constexpr int LD1 = D + FB_APAD, LD4 = F + FB_APAD;  // padded activation row strides in shared memory
  extern __shared__ __align__(16) uint8_t fb_smem[];
  float* red = reinterpret_cast<float*>(fb_smem);                               // split-K reduction tiles: 8 warps x 32 x 8 fp32
  __nv_bfloat16* a_s = reinterpret_cast<__nv_bfloat16*>(fb_smem + FB_WARPS * 32 * 8 * 4);  // activation rows of the current phase
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int G = gridDim.x;
  const int S = p.S;
  WSlab ws;
  unsigned bar_target = 0;
  PDL_PROLOGUE();  // launched without the PDL attribute (cooperative), but its successor may be pre-staged
  // weights of this CTA's first work item of the next GEMM phase: in flight while the activation prologue runs
  auto prefetch = [&](const __nv_bfloat16* W, int K, int N) {
    const bool mine = static_cast<int>(blockIdx.x) < N / 8;
    if (mine) wslab_load(ws, W, K, blockIdx.x, lane, warp);
    return mine;
  };

  // ================================================================= encoder
  for (int l = 0; l < p.n_enc; ++l) {
    const FusedLayer& w = p.enc[l];
    // ---- phase A: a = LN1(x) (layer 0: x = embedding, computed by every CTA; CTA 0 publishes it), QKV = a W_in^T + b ----
    bool pf = prefetch(w.in_w, D, 3 * D);
    if (l == 0) {
      for (int s = warp; s < S; s += FB_WARPS) {
        const EmbedTok& tk = p.tok[s];
        float4 acc[NJ], o[NJ];
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[j] = __ldg(reinterpret_cast<const float4*>(tk.cvec + j * 128 + lane * 4));
        for (int i0 = 0; i0 < tk.d; i0 += 32) {  // lane l fetches (and tokenises) feature i0 + l, then the warp shares them
          float xl = 0.f;
          if (i0 + lane < tk.d) {
            xl = __ldcg(tk.src + i0 + lane);
            if (tk.nmean != nullptr) xl = (xl - __ldg(tk.nmean + i0 + lane)) / __ldg(tk.nstd + i0 + lane);
          }
          const int cnt = min(32, tk.d - i0);
#pragma unroll 8
          for (int i = 0; i < cnt; ++i) {
            const float xi = __shfl_sync(0xffffffffu, xl, i);
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
              const float4 ww = __ldg(reinterpret_cast<const float4*>(tk.wt + static_cast<size_t>(i0 + i) * D + j * 128 + lane * 4));
              acc[j].x = fmaf(xi, ww.x, acc[j].x); acc[j].y = fmaf(xi, ww.y, acc[j].y);
              acc[j].z = fmaf(xi, ww.z, acc[j].z); acc[j].w = fmaf(xi, ww.w, acc[j].w);
            }
          }
        }
        warp_layernorm<NJ>(acc, w.n1_w, w.n1_b, lane, o);
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          *reinterpret_cast<uint2*>(a_s + static_cast<size_t>(s) * LD1 + j * 128 + lane * 4) = f4_to_bf4(o[j]);
          if (blockIdx.x == 0) *reinterpret_cast<float4*>(p.X + static_cast<size_t>(s) * D + j * 128 + lane * 4) = acc[j];
        }
      }
    } else {
      ln_rows_to_smem<NJ>(p.X, S, w.n1_w, w.n1_b, a_s, LD1);
    }
    __syncthreads();
    rows_gemm(a_s, LD1, 0, S, D, w.in_w, 3 * D, w.in_b, nullptr, 0, red, ws, pf, [&](int m, int n, float v, float) {
      p.QKV[static_cast<size_t>(m) * 3 * D + n] = __float2bfloat16_rn(v);
    });
    grid_sync(p.bar, bar_target);
    // ---- phase B: self-attention, one (row, head) pair per warp ----
    pf = prefetch(w.out_w, D, D);
    for (int pr = warp * G + blockIdx.x; pr < S * H; pr += FB_WARPS * G) {
      const int r = pr / H, h = pr - r * H;
      float4 o;
      attend_pair([&]() { return p.QKV + static_cast<size_t>(r) * 3 * D + h * 128; },
                  [&](int j) { return p.QKV + static_cast<size_t>(j) * 3 * D + D + h * 128; },
                  [&](int j) { return p.QKV + static_cast<size_t>(j) * 3 * D + 2 * D + h * 128; }, S, lane, o);
      *reinterpret_cast<uint2*>(p.ATT + static_cast<size_t>(r) * D + h * 128 + lane * 4) = f4_to_bf4(o);
    }
    grid_sync(p.bar, bar_target);
    // ---- phase C: x += att W_out^T + b ----
    copy_rows_to_smem(p.ATT, S, D, a_s);
    __syncthreads();
    rows_gemm(a_s, LD1, 0, S, D, w.out_w, D, w.out_b, p.X, D, red, ws, pf, [&](int m, int n, float v, float r) {
      p.X[static_cast<size_t>(m) * D + n] = r + v;
    });
    pf = prefetch(w.l1_w, D, F);
    grid_sync(p.bar, bar_target);
    // ---- phase D: hid = gelu(LN2(x) W1^T + b1) ----
    ln_rows_to_smem<NJ>(p.X, S, w.n2_w, w.n2_b, a_s, LD1);
    __syncthreads();
    rows_gemm(a_s, LD1, 0, S, D, w.l1_w, F, w.l1_b, nullptr, 0, red, ws, pf, [&](int m, int n, float v, float) {
      p.HID[static_cast<size_t>(m) * F + n] = __float2bfloat16_rn(gelu_erf_fast(v));
    });
    pf = prefetch(w.l2_w, F, D);
    grid_sync(p.bar, bar_target);
    // ---- phase E: x += hid W2^T + b2 ----
    copy_rows_to_smem(p.HID, S, F, a_s);
    __syncthreads();
    rows_gemm(a_s, LD4, 0, S, F, w.l2_w, D, w.l2_b, p.X, D, red, ws, pf, [&](int m, int n, float v, float r) {
      p.X[static_cast<size_t>(m) * D + n] = r + v;
    });
    grid_sync(p.bar, bar_target);
  }

  // ================================================================= decoder (single layer, needed rows only)
  const FusedLayer& w = p.dec;
  const int T4 = p.T4, NQ = p.n_need;
  // ---- phase F: enc = final encoder norm; decoder embedding of the kept tokens, per modality (mtm_model.py:646-661) ----
  ln_rows_to_smem<NJ>(p.X, S, p.enc_norm_w, p.enc_norm_b, a_s, LD1);
  __syncthreads();
  for (int k = 0; k < 4; ++k) {
    const int r0 = p.mod_row0[k], r1 = p.mod_row0[k + 1];
    if (r1 > r0)
      rows_gemm(a_s, LD1, r0, r1, D, p.dec_w[k], D, nullptr, nullptr, 0, red, ws, false, [&](int m, int n, float v, float) {
        p.Xd[static_cast<size_t>(m) * D + n] = v + __ldg(p.dec_cvec + static_cast<size_t>(p.enc_dectok[m]) * D + n);
      });
  }
  bool pf = prefetch(w.in_w, D, 3 * D);
  grid_sync(p.bar, bar_target);
  // ---- phase G: [Q | K | V] of the kept tokens = LN1(xd) W_in^T + b ----
  ln_rows_to_smem<NJ>(p.Xd, S, w.n1_w, w.n1_b, a_s, LD1);
  __syncthreads();
  rows_gemm(a_s, LD1, 0, S, D, w.in_w, 3 * D, w.in_b, nullptr, 0, red, ws, pf, [&](int m, int n, float v, float) {
    p.QKV[static_cast<size_t>(m) * 3 * D + n] = __float2bfloat16_rn(v);
  });
  grid_sync(p.bar, bar_target);
  // ---- phase H: needed queries x all 4T keys (mask-token rows from the batch-constant table); residual rows -> XS ----
  pf = prefetch(w.out_w, D, D);
  for (int pr = warp * G + blockIdx.x; pr < NQ * H; pr += FB_WARPS * G) {
    const int qi = pr / H, h = pr - qi * H;
    const int jq = p.need_tok[qi];
    const int sq = p.dec_src[jq];
    auto row_of = [&](int j, int part) -> const __nv_bfloat16* {
      const int s = p.dec_src[j];
      return (s < 0 ? p.const_qkv + static_cast<size_t>(j) * 3 * D : p.QKV + static_cast<size_t>(s) * 3 * D) + part * D + h * 128;
    };
    float4 o;
    attend_pair([&]() { return row_of(jq, 0); }, [&](int j) { return row_of(j, 1); }, [&](int j) { return row_of(j, 2); }, T4, lane, o);
    *reinterpret_cast<uint2*>(p.ATT + static_cast<size_t>(qi) * D + h * 128 + lane * 4) = f4_to_bf4(o);
    const float* res = sq < 0 ? p.dec_maskrow + static_cast<size_t>(jq) * D : p.Xd + static_cast<size_t>(sq) * D;
    *reinterpret_cast<float4*>(p.XS + static_cast<size_t>(qi) * D + h * 128 + lane * 4) = ldcg4(res + h * 128 + lane * 4);
  }
  grid_sync(p.bar, bar_target);
  // ---- phase I: xs += att W_out^T + b ----
  copy_rows_to_smem(p.ATT, NQ, D, a_s);
  __syncthreads();
  rows_gemm(a_s, LD1, 0, NQ, D, w.out_w, D, w.out_b, p.XS, D, red, ws, pf, [&](int m, int n, float v, float r) {
    p.XS[static_cast<size_t>(m) * D + n] = r + v;
  });
  pf = prefetch(w.l1_w, D, F);
  grid_sync(p.bar, bar_target);
  // ---- phase J: hid = gelu(LN2(xs) W1^T + b1) ----
  ln_rows_to_smem<NJ>(p.XS, NQ, w.n2_w, w.n2_b, a_s, LD1);
  __syncthreads();
  rows_gemm(a_s, LD1, 0, NQ, D, w.l1_w, F, w.l1_b, nullptr, 0, red, ws, pf, [&](int m, int n, float v, float) {
    p.HID[static_cast<size_t>(m) * F + n] = __float2bfloat16_rn(gelu_erf_fast(v));
  });
  pf = prefetch(w.l2_w, F, D);
  grid_sync(p.bar, bar_target);
  // ---- phase K: xs += hid W2^T + b2 ----
  copy_rows_to_smem(p.HID, NQ, F, a_s);
  __syncthreads();
  rows_gemm(a_s, LD4, 0, NQ, F, w.l2_w, D, w.l2_b, p.XS, D, red, ws, pf, [&](int m, int n, float v, float r) {
    p.XS[static_cast<size_t>(m) * D + n] = r + v;
  });
  grid_sync(p.bar, bar_target);
  // ---- phase L: y = final decoder norm, y2 = the consuming head's own LayerNorm of y (mtm_model.py:397-409, 428-433) ----
  for (int qi = warp * G + blockIdx.x; qi < NQ; qi += FB_WARPS * G) {
    float4 v[NJ], o[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) v[j] = ldcg4(p.XS + static_cast<size_t>(qi) * D + j * 128 + lane * 4);
    warp_layernorm<NJ>(v, p.fnorm_w, p.fnorm_b, lane, o);
#pragma unroll
    for (int j = 0; j < NJ; ++j) *reinterpret_cast<uint2*>(p.Y + static_cast<size_t>(qi) * D + j * 128 + lane * 4) = f4_to_bf4(o[j]);
    const int k = p.need_mod[qi];
    if (p.head_g[k] != nullptr) {
      float4 o2[NJ];
      warp_layernorm<NJ>(o, p.head_g[k], p.head_b[k], lane, o2);
#pragma unroll
      for (int j = 0; j < NJ; ++j) *reinterpret_cast<uint2*>(p.Y2 + static_cast<size_t>(qi) * D + j * 128 + lane * 4) = f4_to_bf4(o2[j]);
    } else if (p.out_mu != nullptr) {
      // actor head on the bf16-rounded final norm (DiagGaussianActor, mtm_model.py:313-321): mu, std = exp(-5 + 3.5 (tanh(.) + 1))
      float4 y[NJ];
#pragma unroll
      for (int j = 0; j < NJ; ++j) y[j] = bf4_to_f4(f4_to_bf4(o[j]));
      const int t_out = p.need_tok[qi] - k * (p.T4 / 4);
      for (int a0 = 0; a0 < p.act_dim; a0 += 4) {  // 4 outputs x 2 heads: 8 weight rows in flight
        float4 wm[4][NJ], wl[4][NJ];
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (a0 + i < p.act_dim) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
              wm[i][j] = __ldg(reinterpret_cast<const float4*>(p.mu_w + static_cast<size_t>(a0 + i) * D + j * 128 + lane * 4));
              wl[i][j] = __ldg(reinterpret_cast<const float4*>(p.ls_w + static_cast<size_t>(a0 + i) * D + j * 128 + lane * 4));
            }
          }
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (a0 + i < p.act_dim) {
            float sm = 0.f, sl = 0.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
              sm = fmaf(y[j].x, wm[i][j].x, sm); sm = fmaf(y[j].y, wm[i][j].y, sm); sm = fmaf(y[j].z, wm[i][j].z, sm); sm = fmaf(y[j].w, wm[i][j].w, sm);
              sl = fmaf(y[j].x, wl[i][j].x, sl); sl = fmaf(y[j].y, wl[i][j].y, sl); sl = fmaf(y[j].z, wl[i][j].z, sl); sl = fmaf(y[j].w, wl[i][j].w, sl);
            }
            sm = warp_sum(sm);
            sl = warp_sum(sl);
            if (lane == 0) {
              const size_t o_idx = static_cast<size_t>(t_out) * p.act_dim + a0 + i;
              p.out_mu[o_idx] = sm + __ldg(p.mu_b + a0 + i);
              p.out_std[o_idx] = expf(-5.0f + 3.5f * (tanhf(sl + __ldg(p.ls_b + a0 + i)) + 1.0f));
            }
          }
      }
    }
  }
  grid_finish(p.bar);
}

}  // namespace

size_t fused_b1_smem_bytes(int D, int S, int n_need) {
  return static_cast<size_t>(std::max(S, n_need)) * (4 * D + FB_APAD) * sizeof(__nv_bfloat16) + FB_WARPS * 32 * 8 * sizeof(float);
}

int launch_fused_b1(const FusedB1Params& p, int D, cudaStream_t st) {
  M3PC_REQUIRE(D == 512, "fused_b1: n_embd must be 512 (K slices of at most 8 x 32 per warp)");
  M3PC_REQUIRE(p.S >= 1 && p.S <= FB_MAX_ROWS && p.n_need >= 1 && p.n_need <= FB_MAX_ROWS && p.n_enc >= 1 && p.n_enc <= FB_MAX_LAYERS,
               "fused_b1: shape out of range");
  const size_t smem = fused_b1_smem_bytes(D, p.S, p.n_need);
  M3PC_REQUIRE(smem <= 200 * 1024, "fused_b1: activation panel does not fit shared memory");
  static PerDevice<size_t> smem_limit;  // the attribute and the SM count are per device, not per process
  auto kern = fused_b1_kernel<4>;
  const int num_sms = device_num_sms();
  M3PC_REQUIRE(num_sms > 0, "fused_b1: no device");
  M3PC_CHECK_CUDA(raise_smem_limit(kern, smem_limit, smem));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(num_sms);  // one CTA per SM: all CTAs are co-resident (cooperative launch), the grid barrier cannot deadlock
  cfg.blockDim = dim3(FB_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  M3PC_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}

}  // namespace m3pc
