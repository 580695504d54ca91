// Memory-bound fused kernels of the MTM forward (one warp per activation row, 128-bit accesses).
//
//   embed_kernel      K1: tokenizer normalise (omtm/tokenizers/continuous.py:74-79) + per-modality linear embedding +
//                     per-dim encoding + sincos positional embedding (mtm_model.py:546-557) + MAE gather of the kept
//                     tokens (mtm_model.py:534-544, 619-632) + the first block's LayerNorm, written token-major.
//   layernorm_kernel  LayerNorm / final-norm + head-norm chain (mtm_model.py:379-409, 428-433).
//   fill_rows_kernel  K4: batch-constant decoder rows (mask tokens after decoder_embed, mtm_model.py:646-696).
//   rowdot_kernel     K5: skinny output projections 512 -> d and the tanh-Gaussian actor head (mtm_model.py:313-321).
#include <algorithm>
#include <type_traits>

#include "kernels.cuh"

namespace m3pc {
namespace {

template <int NJ, typename AT>
__global__ void __launch_bounds__(256) embed_kernel(const __grid_constant__ EmbedParams p, float* __restrict__ x, AT* __restrict__ y,
                                                    const float* __restrict__ gamma, const float* __restrict__ beta) {
  PDL_PROLOGUE();
  constexpr int D = NJ * 128;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s = blockIdx.y;
  const EmbedTok& tk = p.tok[s];
  const int b_end = min(p.B, (static_cast<int>(blockIdx.x) + 1) * 64);
  // source row of batch row b: its own (bstride > 0), one shared by every row (bstride == 0: history tokens of a single
  // window), or one per group of bdiv global rows (the window of the row's environment).  A warp walks b upwards, so the
  // embedding + LayerNorm are recomputed only when the source row changes.
  long cur = -1;
  float4 acc[NJ], o[NJ];
  for (int b = blockIdx.x * 64 + warp; b < b_end; b += 8) {
    const long srow = tk.bdiv > 0 ? (p.b0 + b) / tk.bdiv : (tk.bstride == 0 ? 0 : b);
    if (srow != cur) {
      cur = srow;
      const float* src = tk.src + static_cast<size_t>(srow) * tk.bstride;
#pragma unroll
      for (int j = 0; j < NJ; ++j) acc[j] = __ldg(reinterpret_cast<const float4*>(tk.cvec + j * 128 + lane * 4));
      // the d input features of the row: one coalesced (and, where the tokenizer applies, normalised) load per 32 features,
      // broadcast with shuffles -- not d dependent scalar loads in the FMA chain
      for (int i0 = 0; i0 < tk.d; i0 += 32) {
        float xv = 0.f;
        if (i0 + lane < tk.d) {
          xv = __ldg(src + i0 + lane);
          if (tk.nmean != nullptr) xv = (xv - __ldg(tk.nmean + i0 + lane)) / __ldg(tk.nstd + i0 + lane);
        }
        const int n_i = min(32, tk.d - i0);
#pragma unroll 4
        for (int ii = 0; ii < n_i; ++ii) {
          const float xi = __shfl_sync(0xffffffffu, xv, ii);
          const int i = i0 + ii;
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(tk.wt + static_cast<size_t>(i) * D + j * 128 + lane * 4));
            acc[j].x = fmaf(xi, w.x, acc[j].x);
            acc[j].y = fmaf(xi, w.y, acc[j].y);
            acc[j].z = fmaf(xi, w.z, acc[j].z);
            acc[j].w = fmaf(xi, w.w, acc[j].w);
          }
        }
      }
      warp_layernorm<NJ>(acc, gamma, beta, lane, o);
    }
    const size_t row = static_cast<size_t>(s) * p.B + b;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      st4(x + row * D + j * 128 + lane * 4, acc[j]);
      st4(y + row * D + j * 128 + lane * 4, o[j]);
    }
  }
}

template <int NJ, typename AT>
__global__ void __launch_bounds__(256) layernorm_kernel(const __grid_constant__ LnParams p) {
  PDL_PROLOGUE();
  constexpr int D = NJ * 128;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= p.rows) return;
  float4 v[NJ], o[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) v[j] = ld4(p.x + static_cast<size_t>(row) * D + j * 128 + lane * 4);
  if (p.g1 != nullptr) {
    warp_layernorm<NJ>(v, p.g1, p.b1, lane, o);
    if (p.y1 != nullptr) {
      AT* y1 = reinterpret_cast<AT*>(p.y1);
#pragma unroll
      for (int j = 0; j < NJ; ++j) st4(y1 + static_cast<size_t>(row) * D + j * 128 + lane * 4, o[j]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < NJ; ++j) o[j] = v[j];
  }
  if (p.y2 != nullptr) {
    const int grp = p.tok_group[row / p.rows_per_group];
    const float* g2 = p.g2[grp];
    if (g2 != nullptr) {
      float4 o2[NJ];
      warp_layernorm<NJ>(o, g2, p.b2[grp], lane, o2);
      AT* y2 = reinterpret_cast<AT*>(p.y2);
#pragma unroll
      for (int j = 0; j < NJ; ++j) st4(y2 + static_cast<size_t>(row) * D + j * 128 + lane * 4, o2[j]);
    }
  }
}

template <int NJ>
__global__ void __launch_bounds__(256) fill_rows_kernel(const __grid_constant__ FillParams p, float* __restrict__ x) {
  PDL_PROLOGUE();
  constexpr int D = NJ * 128;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.y;
  const int bs = p.bstride[i];
  float4 v[NJ];
  if (bs == 0) {
#pragma unroll
    for (int j = 0; j < NJ; ++j) v[j] = __ldg(reinterpret_cast<const float4*>(p.row[i] + j * 128 + lane * 4));
  }
  const int b_end = min(p.B, (static_cast<int>(blockIdx.x) + 1) * 64);
  for (int b = blockIdx.x * 64 + warp; b < b_end; b += 8) {
    const size_t row = static_cast<size_t>(p.tok[i]) * p.B + b;
    if (bs != 0) {
#pragma unroll
      for (int j = 0; j < NJ; ++j) v[j] = *reinterpret_cast<const float4*>(p.row[i] + static_cast<size_t>(b) * bs + j * 128 + lane * 4);
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) st4(x + row * D + j * 128 + lane * 4, v[j]);
  }
}

// A warp owns R consecutive rows: every weight vector it loads is used for R dot products (at R = 1 the kernel re-read the
// whole (d_out, D) weight matrix through L1 for every row, which bounded it at ~10 % of the HBM rate its inputs need).
// Per row the arithmetic (per-lane FMA chain, then warp_sum) is the same for every R, so results do not depend on R.
// A launch carries up to ROWDOT_MAX_JOBS projections (the heads of the consumed modalities): blocks [block0[j], block0[j + 1]) work on job j.
template <int NJ, typename AT, int R>
__global__ void __launch_bounds__(256) rowdot_kernel(const __grid_constant__ RowDotGroup grp) {
  PDL_PROLOGUE();
  constexpr int D = NJ * 128;
  const int lane = threadIdx.x & 31;
  int job = 0;
#pragma unroll
  for (int j = 1; j < ROWDOT_MAX_JOBS; ++j)
    if (j < grp.n && static_cast<int>(blockIdx.x) >= grp.block0[j]) job = j;
  const RowDotParams& p = grp.p[job];
  const int n_rows = p.n_t * p.B;
  const int r0 = ((static_cast<int>(blockIdx.x) - grp.block0[job]) * 8 + (threadIdx.x >> 5)) * R;  // r = t * B + b
  if (r0 >= n_rows) return;
  float4 v[R][NJ];
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const int r = min(r0 + i, n_rows - 1);  // tail rows repeat the last row; they are not stored
    const AT* yrow = reinterpret_cast<const AT*>(p.y) + (static_cast<size_t>(p.tok0) * p.B + r) * D;
#pragma unroll
    for (int j = 0; j < NJ; ++j) v[i][j] = ld4(yrow + j * 128 + lane * 4);
  }
  for (int o0 = 0; o0 < p.d_out; o0 += 32) {
    float mine[R], mine2[R];
#pragma unroll
    for (int i = 0; i < R; ++i) mine[i] = mine2[i] = 0.f;
    const int o_end = min(p.d_out, o0 + 32);
#pragma unroll 2
    for (int o = o0; o < o_end; ++o) {
      float s[R];
#pragma unroll
      for (int i = 0; i < R; ++i) s[i] = 0.f;
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(p.w + static_cast<size_t>(o) * D + j * 128 + lane * 4));
#pragma unroll
        for (int i = 0; i < R; ++i) {
          s[i] = fmaf(v[i][j].x, w.x, s[i]); s[i] = fmaf(v[i][j].y, w.y, s[i]); s[i] = fmaf(v[i][j].z, w.z, s[i]); s[i] = fmaf(v[i][j].w, w.w, s[i]);
        }
      }
      const float bo = __ldg(p.b + o);
#pragma unroll
      for (int i = 0; i < R; ++i) {
        const float t = warp_sum(s[i]);
        if (lane == o - o0) mine[i] = t + bo;
      }
      if (p.w2 != nullptr) {
#pragma unroll
        for (int i = 0; i < R; ++i) s[i] = 0.f;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(p.w2 + static_cast<size_t>(o) * D + j * 128 + lane * 4));
#pragma unroll
          for (int i = 0; i < R; ++i) {
            s[i] = fmaf(v[i][j].x, w.x, s[i]); s[i] = fmaf(v[i][j].y, w.y, s[i]); s[i] = fmaf(v[i][j].z, w.z, s[i]); s[i] = fmaf(v[i][j].w, w.w, s[i]);
          }
        }
        const float bo2 = __ldg(p.b2 + o);
#pragma unroll
        for (int i = 0; i < R; ++i) {
          const float t = warp_sum(s[i]);
          if (lane == o - o0) mine2[i] = t + bo2;
        }
      }
    }
    if (o0 + lane < p.d_out) {
#pragma unroll
      for (int i = 0; i < R; ++i) {
        const int r = r0 + i;
        if (r >= n_rows) break;
        const int t = r / p.B, b = r - t * p.B;
        const size_t obase = (static_cast<size_t>(b) * p.T_out + (p.t_out0 + t)) * p.d_out;
        p.out[obase + o0 + lane] = mine[i];
        if (p.w2 != nullptr) {
          // log_std = -5 + 0.5 * (2 - (-5)) * (tanh(.) + 1); std = exp(log_std)     (mtm_model.py:313-321)
          const float ls = -5.0f + 3.5f * (tanhf(mine2[i]) + 1.0f);
          p.out2[obase + o0 + lane] = expf(ls);
        }
      }
    }
  }
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t n) {
  PDL_PROLOGUE();
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) out[i] = __float2bfloat16_rn(in[i]);
}

template <typename F>
int dispatch_d(int D, F&& f) {
  switch (D) {
    case 128: return f(std::integral_constant<int, 1>{});
    case 256: return f(std::integral_constant<int, 2>{});
    case 384: return f(std::integral_constant<int, 3>{});
    case 512: return f(std::integral_constant<int, 4>{});
    case 768: return f(std::integral_constant<int, 6>{});
    case 1024: return f(std::integral_constant<int, 8>{});
    default:
      set_error("unsupported n_embd " + std::to_string(D) + " (supported: 128, 256, 384, 512, 768, 1024)");
      return M3PC_ERR_INVALID;
  }
}

}  // namespace

int launch_embed(const EmbedParams& p, int D, float* x, void* y, bool y_bf16, const float* gamma, const float* beta, cudaStream_t st) {
  M3PC_REQUIRE(p.n_tok > 0 && p.n_tok <= MAX_TOK && p.B > 0, "embed: bad token table");
  dim3 grid(ceil_div(p.B, 64), p.n_tok);
  return dispatch_d(D, [&](auto nj) -> int {
    constexpr int NJ = decltype(nj)::value;
    if (y_bf16)
      M3PC_CHECK_CUDA(launch_k(embed_kernel<NJ, __nv_bfloat16>, dim3(grid), dim3(256), 0, st, p, x, reinterpret_cast<__nv_bfloat16*>(y), gamma, beta));
    else
      M3PC_CHECK_CUDA(launch_k(embed_kernel<NJ, float>, dim3(grid), dim3(256), 0, st, p, x, reinterpret_cast<float*>(y), gamma, beta));
    M3PC_CHECK_LAUNCH();
    return M3PC_OK;
  });
}

int launch_layernorm(const LnParams& p, int D, bool out_bf16, cudaStream_t st) {
  M3PC_REQUIRE(p.rows > 0, "layernorm: no rows");
  dim3 grid(ceil_div(p.rows, 8));
  return dispatch_d(D, [&](auto nj) -> int {
    constexpr int NJ = decltype(nj)::value;
    if (out_bf16)
      M3PC_CHECK_CUDA(launch_k(layernorm_kernel<NJ, __nv_bfloat16>, dim3(grid), dim3(256), 0, st, p));
    else
      M3PC_CHECK_CUDA(launch_k(layernorm_kernel<NJ, float>, dim3(grid), dim3(256), 0, st, p));
    M3PC_CHECK_LAUNCH();
    return M3PC_OK;
  });
}

int launch_fill_rows(const FillParams& p, int D, float* x, cudaStream_t st) {
  if (p.n == 0) return M3PC_OK;
  dim3 grid(ceil_div(p.B, 64), p.n);
  return dispatch_d(D, [&](auto nj) -> int {
    constexpr int NJ = decltype(nj)::value;
    M3PC_CHECK_CUDA(launch_k(fill_rows_kernel<NJ>, dim3(grid), dim3(256), 0, st, p, x));
    M3PC_CHECK_LAUNCH();
    return M3PC_OK;
  });
}

int launch_rowdot_group(const RowDotParams* jobs, int n, int D, bool y_bf16, cudaStream_t st) {
  M3PC_REQUIRE(n >= 0 && n <= ROWDOT_MAX_JOBS, "rowdot: too many projections in one launch");
  RowDotGroup g{};
  int max_rows = 0;
  for (int j = 0; j < n; ++j)
    if (jobs[j].n_t > 0) max_rows = std::max(max_rows, jobs[j].n_t * jobs[j].B);
  if (max_rows == 0) return M3PC_OK;
  const bool wide = max_rows >= 4096 && D <= 512;  // 4 rows per warp once there are enough rows to fill the SMs (register budget: D <= 512)
  int blocks = 0;
  for (int j = 0; j < n; ++j) {
    if (jobs[j].n_t <= 0) continue;
    g.p[g.n] = jobs[j];
    g.block0[g.n++] = blocks;
    blocks += ceil_div(jobs[j].n_t * jobs[j].B, 8 * (wide ? 4 : 1));
  }
  dim3 grid(blocks);
  return dispatch_d(D, [&](auto nj) -> int {
    constexpr int NJ = decltype(nj)::value;
    if constexpr (NJ <= 4) {
      if (wide) {
        if (y_bf16)
          M3PC_CHECK_CUDA(launch_k(rowdot_kernel<NJ, __nv_bfloat16, 4>, dim3(grid), dim3(256), 0, st, g));
        else
          M3PC_CHECK_CUDA(launch_k(rowdot_kernel<NJ, float, 4>, dim3(grid), dim3(256), 0, st, g));
        M3PC_CHECK_LAUNCH();
        return M3PC_OK;
      }
    }
    if (y_bf16)
      M3PC_CHECK_CUDA(launch_k(rowdot_kernel<NJ, __nv_bfloat16, 1>, dim3(grid), dim3(256), 0, st, g));
    else
      M3PC_CHECK_CUDA(launch_k(rowdot_kernel<NJ, float, 1>, dim3(grid), dim3(256), 0, st, g));
    M3PC_CHECK_LAUNCH();
    return M3PC_OK;
  });
}
int launch_rowdot(const RowDotParams& p, int D, bool y_bf16, cudaStream_t st) { return launch_rowdot_group(&p, 1, D, y_bf16, st); }

int launch_f32_to_bf16(const float* in, __nv_bfloat16* out, size_t n, cudaStream_t st) {
  if (n == 0) return M3PC_OK;
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  M3PC_CHECK_CUDA(launch_k(f32_to_bf16_kernel, dim3(blocks), dim3(256), 0, st, in, out, n));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}

}  // namespace m3pc
