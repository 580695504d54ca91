// Skinny bf16 GEMM for M <= 32 rows: C[M,N] = epilogue(A[M,K] * W[N,K]^T), fp32 accumulation on CUDA cores.
//
// The B = 1 passes of the planners (pass 1 of Learner.rtg_guiding / critic_lambda_guiding, learner.py:278-284; the
// zero-shot planners) have 8..17 token rows: a 128-row tcgen05 tile would be > 85 % padding and the kernel is pure
// latency.  Here every warp owns output columns: it streams the column's weight row once (coalesced 16-byte loads)
// and dots it with all M activation rows staged in shared memory, so all SMs pull weights from L2 concurrently.
// Same fused epilogues as the tensor-core kernel (bias, per-token table, GELU, ReLU, residual, bf16 / fp32 out).
#include "common.cuh"

namespace m3pc {
namespace {

constexpr int SK_THREADS = 256;      // 8 warps, one output column per warp
constexpr int SK_MAX_M = 32;
constexpr int SK_WREG = 8;           // 16-byte weight chunks a lane keeps in flight (covers K <= 2048 in one batch)

__global__ void __launch_bounds__(SK_THREADS) gemm_skinny_kernel(const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ W,
                                                                 void* __restrict__ C, int M, int N, int K, const float* __restrict__ bias,
                                                                 const float* __restrict__ table, int rows_per_group, int flags) {
  PDL_PROLOGUE();
  extern __shared__ __align__(16) uint8_t sk_smem[];
  __nv_bfloat16* As = reinterpret_cast<__nv_bfloat16*>(sk_smem);  // M x K
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = blockIdx.x * (SK_THREADS / 32) + warp;
  const int kchunks = K / 8;
  // issue this warp's first batch of weight loads before anything else: the whole row is in flight at once
  const uint4* wrow = reinterpret_cast<const uint4*>(W + static_cast<size_t>(min(n, N - 1)) * K);
  uint4 wreg[SK_WREG];
#pragma unroll
  for (int j = 0; j < SK_WREG; ++j) {
    const int c = lane + 32 * j;
    wreg[j] = (c < kchunks) ? __ldg(wrow + c) : make_uint4(0, 0, 0, 0);
  }
  // stage A (M*K bf16) with cp.async: every 16-byte chunk is in flight before the first one is waited for
  const int chunks = M * kchunks;
  const uint32_t as_base = smem_u32(As);
  for (int i = threadIdx.x; i < chunks; i += SK_THREADS) cp_async16(as_base + 16u * i, reinterpret_cast<const uint4*>(A) + i);
  cp_async_commit();
  // epilogue operands are independent of the accumulation: fetch them now as well
  const int erow = lane < M ? lane : 0;
  float e_bias = 0.f, e_table = 0.f, e_res = 0.f;
  if (n < N) {
    if (bias != nullptr) e_bias = __ldg(bias + n);
    if (table != nullptr) e_table = __ldg(table + static_cast<size_t>(erow / rows_per_group) * N + n);
    if (flags & EPI_RESIDUAL) e_res = reinterpret_cast<const float*>(C)[static_cast<size_t>(erow) * N + n];
  }
  cp_async_wait_all();
  __syncthreads();
  if (n >= N) return;
  const bool do_gelu = flags & EPI_GELU, do_relu = flags & EPI_RELU, do_res = flags & EPI_RESIDUAL;
  const bool out_f32 = do_res || (flags & EPI_OUT_F32);
  float acc[SK_MAX_M];
#pragma unroll
  for (int m = 0; m < SK_MAX_M; ++m) acc[m] = 0.f;
  for (int c0 = 0; c0 < kchunks; c0 += 32 * SK_WREG) {
    if (c0 > 0) {
#pragma unroll
      for (int j = 0; j < SK_WREG; ++j) {
        const int c = c0 + lane + 32 * j;
        wreg[j] = (c < kchunks) ? __ldg(wrow + c) : make_uint4(0, 0, 0, 0);
      }
    }
#pragma unroll
    for (int j = 0; j < SK_WREG; ++j) {
      const int c = c0 + lane + 32 * j;
      if (c0 + 32 * j >= kchunks) break;  // warp-uniform
      if (c < kchunks) {
        float wf[8];
        bf16x8_to_float(wreg[j], wf);
#pragma unroll
        for (int m = 0; m < SK_MAX_M; ++m) {  // fully unrolled so acc[] stays in registers
          if (m < M) {
            float af[8];
            bf16x8_to_float(*reinterpret_cast<const uint4*>(As + static_cast<size_t>(m) * K + c * 8), af);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[m] = fmaf(af[i], wf[i], acc[m]);
          }
        }
      }
    }
  }
  float mine = 0.f;
#pragma unroll
  for (int m = 0; m < SK_MAX_M; ++m) {
    if (m < M) {
      const float s = warp_sum(acc[m]);
      if (lane == m) mine = s;
    }
  }
  if (lane < M) {
    float v = mine + e_bias + e_table;
    if (do_gelu) v = gelu_erf_fast(v);
    if (do_relu) v = fmaxf(v, 0.f);
    if (out_f32) {
      if (do_res) v += e_res;
      reinterpret_cast<float*>(C)[static_cast<size_t>(lane) * N + n] = v;
    } else {
      reinterpret_cast<__nv_bfloat16*>(C)[static_cast<size_t>(lane) * N + n] = __float2bfloat16_rn(v);
    }
  }
}

}  // namespace

int gemm_bf16_skinny(const __nv_bfloat16* A, const __nv_bfloat16* W, void* C, int M, int N, int K, const GemmEpilogue& epi, cudaStream_t st) {
  M3PC_REQUIRE(M >= 1 && M <= SK_MAX_M && K % 8 == 0, "gemm_skinny: needs M <= 32 and K % 8 == 0");
  const size_t smem = static_cast<size_t>(M) * K * sizeof(__nv_bfloat16);
  M3PC_REQUIRE(smem <= 160 * 1024, "gemm_skinny: A panel does not fit shared memory");
  static PerDevice<size_t> smem_limit;
  M3PC_CHECK_CUDA(raise_smem_limit(gemm_skinny_kernel, smem_limit, smem));
  M3PC_CHECK_CUDA(launch_k(gemm_skinny_kernel, dim3(ceil_div(N, SK_THREADS / 32)), dim3(SK_THREADS), smem, st, A, W, C, M, N, K, epi.bias, epi.table,
                                                                          epi.rows_per_group > 0 ? epi.rows_per_group : 1, epi.flags));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}

}  // namespace m3pc
