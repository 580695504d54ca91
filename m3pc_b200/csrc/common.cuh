// Shared helpers for the m3pc sm_100a kernels: error plumbing, activation-type traits, warp reductions.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <cstdlib>
#include <string>
#include <utility>

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

// ---- bf16 packing (round to nearest even) ------------------------------------------------------------------------------------
// two floats -> packed bf16x2 (lo in the low half)
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
// four bf16 (8 bytes) <-> float4
__device__ __forceinline__ float4 bf4_to_f4(uint2 u) {
  const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&u.x), b = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
  const float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ uint2 f4_to_bf4(float4 v) { return make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w)); }
// eight bf16 (16 bytes) -> floats
__device__ __forceinline__ void bf16x8_to_float(const uint4& u, float (&f)[8]) {
  const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __bfloat1622float2(p[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}

// 4 consecutive activations <-> float4
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) { return bf4_to_f4(*reinterpret_cast<const uint2*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(__nv_bfloat16* p, float4 v) { *reinterpret_cast<uint2*>(p) = f4_to_bf4(v); }

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

// nn.LayerNorm epsilon (every norm of the model)
constexpr float kLnEps = 1e-5f;

// LayerNorm of one row of NJ * 128 columns held by a warp as lane-strided float4s: lane owns columns j*128 + lane*4 + {0..3}
template <int NJ>
__device__ __forceinline__ void warp_layernorm(const float4 (&v)[NJ], const float* __restrict__ gamma, const float* __restrict__ beta,
                                               int lane, float4 (&o)[NJ]) {
  constexpr float inv_d = 1.0f / (NJ * 128);
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < NJ; ++j) s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
  const float mean = warp_sum(s) * inv_d;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * inv_d + kLnEps);
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int c = j * 128 + lane * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
    o[j].x = (v[j].x - mean) * rstd * g.x + b.x;
    o[j].y = (v[j].y - mean) * rstd * g.y + b.y;
    o[j].z = (v[j].z - mean) * rstd * g.z + b.z;
    o[j].w = (v[j].w - mean) * rstd * g.w + b.w;
  }
}

// ---- shared memory staging and mma.sync ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
// 16-byte global -> shared copy through L2 only (cp.async.cg); a thread's copies land after cp_async_commit + cp_async_wait_all
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// d (16 x 8, fp32) += a (16 x 16, bf16, row fragment) * b (16 x 8, bf16, column fragment b0, b1): mma.sync.m16n8k16
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
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
// process must configure its own copy of every kernel.  Launchers keep `static PerDevice<...>` state and index it with
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

// Raise `kernel`'s dynamic shared-memory limit on the current device to `bytes` when `limit` (what was set so far) is below it:
// a launcher with a fixed size sets it once, one with a varying size only when the size grows.  `limit` is a static of the
// launcher, one per kernel instance: all instances of a kernel template have one function type, so a static in here would be
// shared between them.
template <typename... KArgs>
inline cudaError_t raise_smem_limit(void (*kernel)(KArgs...), PerDevice<size_t>& limit, size_t bytes) {
  if (bytes <= limit.here()) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
  if (e == cudaSuccess) limit.here() = bytes;
  return e;
}

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

// PDL launch of a grid whose CTAs form clusters of `cluster` CTAs along x (the cluster-dimension attribute comes first);
// cluster = 0 launches without the cluster attribute.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k_cluster(unsigned cluster, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                    Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (cluster > 0) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[n].val.programmaticStreamSerializationAllowed = 1;
  ++n;
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  return launch_k_cluster(0, kernel, grid, block, smem, st, std::forward<Args>(args)...);
}
#endif

// ---- kernel launchers implemented across the .cu files -----------------------------------------------
// Problems that share one launch of a grouped tensor-core kernel (gemm_bf16, gemm_ln_bf16_grouped): each launch carries their
// parameters in its kernel parameter space
constexpr int kMaxGroup = 4;
// gemm_tcgen05.cu
int gemm_init_driver_api();
// gemm_ln.cu: X (M,512) fp32 <- R + A W^T + bias (R = X in place, the fp32 rows `R`, or table[row / rows_per_group]); Y (M,512) bf16 <- LayerNorm(X)
// for 1 .. kMaxGroup such problems in ONE launch (same K, bias, gamma, beta): own A / W / X / Y / residual source each
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
// report: null, or int[2] that receives {rows per CTA-pair unit, CTA pairs} of the launch
int gemm_ln_bf16_grouped(const LnJob* jobs, int n, const float* bias, const float* gamma, const float* beta, int K, cudaStream_t st,
                         int* report = nullptr);
// n >= 1 independent bf16 GEMMs C = epilogue(A W^T); up to kMaxGroup of them share one launch of the CTA-pair kernel where it
// applies (decoder embedding runs, K/V + Q, heads, twin critics)
struct GemmProblem {
  const __nv_bfloat16* A;
  const __nv_bfloat16* W;
  void* C;
  int M, N, K;
  GemmEpilogue epi;
};
// report: null, or int[4 n] that receives {kind, a, b, launch} per problem: kind 0 = the skinny kernel; 1 = gemm_bf16_kernel with
// a = BN, b = CL; 2 = the CTA-pair kernel with a = strided, b = problems in its launch; launch = index of the launch within this call
int gemm_bf16(const GemmProblem* probs, int n, cudaStream_t st, int* report = nullptr);
// gemm_skinny.cu: M <= 32 rows (B = 1 passes): a latency-optimised CUDA-core kernel, same epilogues
int gemm_bf16_skinny(const __nv_bfloat16* A, const __nv_bfloat16* W, void* C, int M, int N, int K, const GemmEpilogue& epi, cudaStream_t st);
// sgemm.cu
int gemm_fp32(const float* A, const float* W, float* C, int M, int N, int K, const GemmEpilogue& epi, cudaStream_t st);
// gemm_tf32x3.cu: the same contract as gemm_fp32, on the tensor cores with the 3xTF32 split (small problems: gemm_fp32)
int gemm_tf32x3(const float* A, const float* W, float* C, int M, int N, int K, const GemmEpilogue& epi, cudaStream_t st);

}  // namespace m3pc
