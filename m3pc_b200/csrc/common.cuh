// Shared helpers for the m3pc sm_100a kernels: error plumbing, activation-type traits, warp reductions.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../include/m3pc.h"

namespace m3pc {

void set_error(const std::string& msg);

#define M3PC_CHECK_CUDA(expr)                                                                              \
  do {                                                                                                     \
    cudaError_t _e = (expr);                                                                               \
    if (_e != cudaSuccess) {                                                                               \
      ::m3pc::set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " (" + __FILE__ + ":" + \
                        std::to_string(__LINE__) + ")");                                                   \
      return M3PC_ERR_CUDA;                                                                                \
    }                                                                                                      \
  } while (0)

#define M3PC_REQUIRE(cond, msg)                                                                  \
  do {                                                                                           \
    if (!(cond)) {                                                                               \
      ::m3pc::set_error(std::string(msg) + " [" #cond "] (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
      return M3PC_ERR_INVALID;                                                                   \
    }                                                                                            \
  } while (0)

#define M3PC_TRY(expr)          \
  do {                          \
    int _rc = (expr);           \
    if (_rc != M3PC_OK) return _rc; \
  } while (0)

// Check the launch that was just issued (cheap: no sync) and count it (m3pc_last_launch_count).
extern thread_local int g_launch_count;
#define M3PC_CHECK_LAUNCH()                \
  do {                                     \
    ++::m3pc::g_launch_count;              \
    M3PC_CHECK_CUDA(cudaGetLastError());   \
  } while (0)

// epilogue flags (public ABI: m3pc_gemm_*)
constexpr int EPI_GELU = 1;
constexpr int EPI_RESIDUAL = 2;  // C (fp32) += result, in place
constexpr int EPI_RELU = 4;
// internal-only
constexpr int EPI_ROWTABLE = 8;  // add table[(row / rows_per_group) * N + col]
constexpr int EPI_OUT_F32 = 16;  // write fp32 even without residual

struct GemmEpilogue {
  const float* bias = nullptr;    // (N) or null
  const float* table = nullptr;   // (groups, N) or null; group = row / rows_per_group
  int rows_per_group = 1;
  int flags = 0;
};

// ---- activation element traits -------------------------------------------------------------------
template <typename T>
struct Act;
template <>
struct Act<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <>
struct Act<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

// 4 consecutive activations <-> float4
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
  uint2 u = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&u.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&u.y);
  float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
  __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&a);
  u.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// nn.GELU() (erf form), evaluated in fp32.
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// Branch-free GELU(erf) for the bf16 tensor-core epilogues: erf(a) = 1 - (1 + a1 a + ... + a6 a^6)^-16 for a >= 0
// (Abramowitz & Stegun 7.1.28, |error| <= 3e-7, far below the bf16 rounding of the result).  ~17 instructions, one MUFU,
// no divergence -- erff() costs 25-40 with a data-dependent branch, which made the FFN1 epilogue the bottleneck.
__device__ __forceinline__ float gelu_erf_fast(float x) {
  const float a = fminf(fabsf(x) * 0.70710678118654752440f, 6.0f);
  float t = fmaf(a, 0.0000430638f, 0.0002765672f);
  t = fmaf(a, t, 0.0001520143f);
  t = fmaf(a, t, 0.0092705272f);
  t = fmaf(a, t, 0.0422820123f);
  t = fmaf(a, t, 0.0705230784f);
  t = fmaf(a, t, 1.0f);
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(t));  // 1 ulp; the ^16 below keeps the result within 2e-6
  r *= r; r *= r; r *= r; r *= r;
  const float erf_abs = 1.0f - r;
  const float hx = 0.5f * x;
  return fmaf(fabsf(hx), erf_abs, hx);  // 0.5 x (1 + sign(x) erf|x|)
}

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// ---- per-device launch bookkeeping ---------------------------------------------------------------------------------------
// cudaFuncSetAttribute and the SM count belong to a DEVICE, not to the process: a second handle on another GPU of the same
// process must configure its own copy of every kernel.  Launchers keep `static PerDevice<...> configured;` and index it with
// current_device().
constexpr int kMaxDevices = 64;
inline int current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return (d < 0 || d >= kMaxDevices) ? 0 : d;
}
template <typename T>
struct PerDevice {
  T v[kMaxDevices] = {};
  T& here() { return v[current_device()]; }
};
int device_num_sms();  // multiprocessors of the current device (cached per device; engine.cu)

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------------
// Every kernel of a plan is launched with cudaLaunchAttributeProgrammaticStreamSerialization: it may be scheduled while
// its predecessor in the stream is still draining, runs its private prologue, and blocks in griddepcontrol.wait until the
// predecessor has completed and flushed its writes.  Rule: EVERY thread of EVERY kernel executes pdl_wait() before its first
// global-memory access and before it can exit (a grid that finished without waiting would release ITS dependents early).
// The trigger is issued right after the wait, so at most one dependent grid is pre-staged at a time.
extern int g_ln_unit_rows;  // gemm_ln.cu
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#define PDL_PROLOGUE() \
  do {                 \
    pdl_wait();        \
    pdl_trigger();     \
  } while (0)

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// ---- kernel launchers implemented across the .cu files -----------------------------------------------
// gemm_tcgen05.cu
int gemm_bf16_tcgen05(const __nv_bfloat16* A, const __nv_bfloat16* W, void* C, int M, int N, int K,
                      const GemmEpilogue& epi, cudaStream_t st);
int gemm_init_driver_api();
// gemm_ln.cu: X (M,512) fp32 <- R + A W^T + bias (R = X in place, the fp32 rows `R`, or table[row / rows_per_group]); Y (M,512) bf16 <- LayerNorm(X)
int gemm_ln_bf16(const __nv_bfloat16* A, const __nv_bfloat16* W, const float* bias, float* X, __nv_bfloat16* Y, const float* gamma,
                 const float* beta, const float* table, int rows_per_group, int M, int K, cudaStream_t st, const float* R = nullptr);
// several such problems in ONE launch (at most 4; same K, bias, gamma, beta): own A / W / X / Y / residual source each
struct LnJob {
  const __nv_bfloat16* A;
  const __nv_bfloat16* W;
  float* X;
  __nv_bfloat16* Y;
  const float* table;   // residual = table[row / rows_per_group], or null
  int rows_per_group;
  int M;
  const float* R;       // residual rows when they are not X itself (and table is null), or null
};
int gemm_ln_bf16_grouped(const LnJob* jobs, int n, const float* bias, const float* gamma, const float* beta, int K, cudaStream_t st);
// several independent bf16 GEMMs in one launch of the CTA-pair kernel (decoder embedding runs, K/V + Q, heads, twin critics)
struct GemmProblem {
  const __nv_bfloat16* A;
  const __nv_bfloat16* W;
  void* C;
  int M, N, K;
  GemmEpilogue epi;
};
int gemm_bf16_grouped(const GemmProblem* probs, int n, cudaStream_t st);
// gemm_skinny.cu: M <= 32 rows (B = 1 passes): a latency-optimised CUDA-core kernel, same epilogues
int gemm_bf16_skinny(const __nv_bfloat16* A, const __nv_bfloat16* W, void* C, int M, int N, int K, const GemmEpilogue& epi, cudaStream_t st);
// sgemm.cu
int gemm_fp32(const float* A, const float* W, float* C, int M, int N, int K, const GemmEpilogue& epi, cudaStream_t st);

}  // namespace m3pc
