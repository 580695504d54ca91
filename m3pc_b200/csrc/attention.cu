// K3: bidirectional multi-head attention for very short sequences (<= 64 tokens, head_dim 128).
//
// Reference call site: nn.MultiheadAttention inside nn.TransformerEncoderLayer (mtm_model.py:379-409):
// softmax(q k^T / sqrt(128)) v, no mask, eval mode.  Activations are token-major (row = token * B + b), so the
// (b, head) slice of a token is 128 contiguous values.  The score matrix never leaves the SM.
//
// Both kernels take the token-gather form (AttnParams): every query / key / value token carries its own source
// pointer and batch stride.  Plain self-attention is the special case where all tokens point into one qkv matrix;
// the planner's decoder uses the general case: queries only for the rows the planner consumes, keys / values split
// between per-candidate rows and batch-constant mask-token rows (bstride 0).
//
//   attention_mma_kernel  (bf16 mode)  one WARP per (batch row, head): Q, K, V staged in swizzled shared memory with
//       cp.async, Q K^T and P V on mma.sync.m16n8k16 (bf16 in, fp32 accumulate) -- these contractions are a few
//       hundred kFLOP per (b, head), far below what a tcgen05 tile (M = 128) could be filled with --, softmax in the
//       accumulator registers with quad shuffles.
//   attention_kernel      (fp32 mode)  one CTA per (b, head), fp32 everywhere (reference-grade path).
#include "kernels.cuh"

namespace m3pc {
namespace {

constexpr int HD = 128;       // head dim
constexpr int QS = HD + 1;    // padded row stride (floats) for conflict-free row-parallel reads
constexpr int ATT_THREADS = 128;

// element offset of batch row b in a token's source (AttnTok)
__device__ __forceinline__ size_t tok_off(const AttnTok& t, int b) {
  return static_cast<size_t>(t.bdiv > 0 ? b / t.bdiv : b) * t.bstride;
}

// ------------------------------------------------------------------------------------------------ fp32 path
__global__ void __launch_bounds__(ATT_THREADS) attention_kernel(const __grid_constant__ AttnParams p) {
  PDL_PROLOGUE();
  extern __shared__ float sm[];
  const int n_q = p.n_q, S = p.n_kv, B = p.B;
  float* Vs = sm;                 // S x HD (first: keeps its float4 stores 16-byte aligned)
  float* Qs = Vs + S * HD;        // n_q x QS
  float* Ks = Qs + n_q * QS;      // S x QS
  float* Ps = Ks + S * QS;        // n_q x (S + 1)
  const int b = blockIdx.x / p.n_head, h = blockIdx.x % p.n_head;
  const int tid = threadIdx.x;

  for (int idx = tid; idx < n_q * (HD / 4); idx += ATT_THREADS) {
    const int i = idx / (HD / 4), c = (idx % (HD / 4)) * 4;
    const float4 v = ld4(reinterpret_cast<const float*>(p.q[i].ptr) + tok_off(p.q[i], b) + h * HD + c);
    float* d = Qs + i * QS + c;
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
  }
  for (int idx = tid; idx < S * (HD / 4); idx += ATT_THREADS) {
    const int j = idx / (HD / 4), c = (idx % (HD / 4)) * 4;
    const float4 kv = ld4(reinterpret_cast<const float*>(p.k[j].ptr) + tok_off(p.k[j], b) + h * HD + c);
    float* d = Ks + j * QS + c;
    d[0] = kv.x; d[1] = kv.y; d[2] = kv.z; d[3] = kv.w;
    *reinterpret_cast<float4*>(Vs + j * HD + c) = ld4(reinterpret_cast<const float*>(p.v[j].ptr) + tok_off(p.v[j], b) + h * HD + c);
  }
  __syncthreads();

  const float scale = 0.08838834764831845f;  // 1/sqrt(128)
  for (int pidx = tid; pidx < n_q * S; pidx += ATT_THREADS) {
    const int i = pidx / S, j = pidx - i * S;
    const float* qi = Qs + i * QS;
    const float* kj = Ks + j * QS;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
    for (int d = 0; d < HD; d += 4) {
      a0 = fmaf(qi[d], kj[d], a0);
      a1 = fmaf(qi[d + 1], kj[d + 1], a1);
      a2 = fmaf(qi[d + 2], kj[d + 2], a2);
      a3 = fmaf(qi[d + 3], kj[d + 3], a3);
    }
    Ps[i * (S + 1) + j] = ((a0 + a1) + (a2 + a3)) * scale;
  }
  __syncthreads();

  const int lane = tid & 31, warp = tid >> 5;
  for (int i = warp; i < n_q; i += ATT_THREADS / 32) {
    float* pr = Ps + i * (S + 1);
    float m = -INFINITY;
    for (int j = lane; j < S; j += 32) m = fmaxf(m, pr[j]);
    m = warp_max(m);
    float s = 0.f;
    for (int j = lane; j < S; j += 32) {
      const float e = expf(pr[j] - m);
      pr[j] = e;
      s += e;
    }
    s = warp_sum(s);
    const float inv = 1.0f / s;
    for (int j = lane; j < S; j += 32) pr[j] *= inv;
  }
  __syncthreads();

  float* out = reinterpret_cast<float*>(p.out);
  const int D = p.n_head * HD;
  for (int i = 0; i < n_q; ++i) {
    const float* pr = Ps + i * (S + 1);
    float acc = 0.f;
    for (int j = 0; j < S; ++j) acc = fmaf(pr[j], Vs[j * HD + tid], acc);
    out[(static_cast<size_t>(i) * B + b) * D + h * HD + tid] = acc;
  }
}

// {kind, a, b, grid_x} of the launch into `info` when it is not null (the kernel-level entry reports which instance ran):
// kind 0 = attention_kernel, 1 = attention_mma_kernel<a, b>, 2 = attention_mma_shared_kernel<a, b>
void report_launch(int* info, int kind, int a, int b, int grid_x) {
  if (info == nullptr) return;
  info[0] = kind; info[1] = a; info[2] = b; info[3] = grid_x;
}

int launch_simple(const AttnParams& p, cudaStream_t st, int* info) {
  const size_t smem = (static_cast<size_t>(p.n_q) * QS + static_cast<size_t>(p.n_kv) * QS + static_cast<size_t>(p.n_kv) * HD +
                       static_cast<size_t>(p.n_q) * (p.n_kv + 1)) * sizeof(float);
  M3PC_REQUIRE(smem <= 200 * 1024, "attention: sequence too long for the shared-memory resident kernel");
  static PerDevice<size_t> smem_limit;
  M3PC_CHECK_CUDA(raise_smem_limit(attention_kernel, smem_limit, smem));
  M3PC_CHECK_CUDA(launch_k(attention_kernel, dim3(p.B * p.n_head), dim3(ATT_THREADS), smem, st, p));
  M3PC_CHECK_LAUNCH();
  report_launch(info, 0, 0, 0, p.B * p.n_head);
  return M3PC_OK;
}

// ------------------------------------------------------------------------------------------------ bf16 tensor-core path
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
// byte offset of 16-byte chunk `c` (0..15) of row `r` in a [rows][256 B] tile, XOR-swizzled so that the 8 rows an
// ldmatrix phase touches fall in 8 different 16-byte bank groups
__device__ __forceinline__ uint32_t swz(int r, int c) { return static_cast<uint32_t>(r * 256 + ((c ^ (r & 7)) << 4)); }

// Key tile jp (16 keys) of a warp's attention: the shared-memory addresses of the K and V buffers that hold it and its first row
// there.  Its keys are numbered key0 .. key0 + 15 and those numbered end or higher are pad rows, masked out of the softmax.
struct KvTile {
  uint32_t k, v;
  int row, key0, end;
};

extern __shared__ __align__(128) uint8_t smem_att[];  // dynamic shared memory of both tensor-core kernels

// Query tile mt (rows 16 mt .. 16 mt + 15) of the warp's Q rows, which start q_off bytes into smem_att (uQ: their shared-memory
// address), against NTK key tiles, kv(jp) -> KvTile: scores Q K^T on mma.sync (bf16 in, fp32 accumulate), softmax in the
// accumulator registers with quad shuffles, O = P V, and O staged as bf16 into the tile's own Q rows (dead once the scores are in
// registers), same swizzle.  kv is a lambda capturing by value, so jp stays a compile-time constant of the unrolled loops.
// Q is addressed as the shared-memory symbol plus an offset, not through a pointer argument, and the per-row kernel numbers its
// keys from 0 across tiles: with a pointer argument or per-tile key counts the compiler lays the kernels out differently (more
// registers, or a spill).
template <int NTK, class KvOf>
__device__ __forceinline__ void attend_q_tile(size_t q_off, uint32_t uQ, int mt, KvOf kv, int lane) {
  uint8_t* sQ = smem_att + q_off;
  const int g = lane >> 2, t = lane & 3;
  const float sl2 = 0.08838834764831845f * 1.4426950408889634f;  // 1/sqrt(128) * log2(e)
  // ---- scores = Q K^T : 16 x 16 NTK, fp32 accumulators ----
  float sc[2 * NTK][4];
#pragma unroll
  for (int j = 0; j < 2 * NTK; ++j) sc[j][0] = sc[j][1] = sc[j][2] = sc[j][3] = 0.f;
#pragma unroll
  for (int kk = 0; kk < HD / 16; ++kk) {
    uint32_t a[4];
    {
      const int r = mt * 16 + (lane & 7) + 8 * ((lane >> 3) & 1), c = 2 * kk + (lane >> 4);
      ldsm_x4(uQ + swz(r, c), a[0], a[1], a[2], a[3]);
    }
#pragma unroll
    for (int jp = 0; jp < NTK; ++jp) {  // two key tiles (16 keys) per ldmatrix.x4
      const KvTile tile = kv(jp);
      uint32_t b0, b1, b2, b3;
      const int r = tile.row + (lane & 7) + 8 * (lane >> 4), c = 2 * kk + ((lane >> 3) & 1);
      ldsm_x4(tile.k + swz(r, c), b0, b1, b2, b3);
      mma_bf16_16816(sc[2 * jp], a, b0, b1);
      mma_bf16_16816(sc[2 * jp + 1], a, b2, b3);
    }
  }
  // ---- softmax over keys (rows g and g+8 of the tile); pad keys of each key tile masked ----
  float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
  for (int j = 0; j < 2 * NTK; ++j) {
    const KvTile tile = kv(j >> 1);
    const int key = tile.key0 + 8 * (j & 1) + 2 * t;
    if (key >= tile.end) sc[j][0] = sc[j][2] = -INFINITY;
    if (key + 1 >= tile.end) sc[j][1] = sc[j][3] = -INFINITY;
    m0 = fmaxf(m0, fmaxf(sc[j][0], sc[j][1]));
    m1 = fmaxf(m1, fmaxf(sc[j][2], sc[j][3]));
  }
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int j = 0; j < 2 * NTK; ++j) {
    sc[j][0] = exp2f((sc[j][0] - m0) * sl2); sc[j][1] = exp2f((sc[j][1] - m0) * sl2);
    sc[j][2] = exp2f((sc[j][2] - m1) * sl2); sc[j][3] = exp2f((sc[j][3] - m1) * sl2);
    l0 += sc[j][0] + sc[j][1];
    l1 += sc[j][2] + sc[j][3];
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;

  // ---- O = P V : 16 x 128 ----
  float o[HD / 8][4];
#pragma unroll
  for (int n = 0; n < HD / 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
#pragma unroll
  for (int kk = 0; kk < NTK; ++kk) {  // 16 keys per step; the score tiles (2kk, 2kk+1) are exactly the A fragment
    uint32_t a[4];
    a[0] = pack_bf16(sc[2 * kk][0] * inv0, sc[2 * kk][1] * inv0);
    a[1] = pack_bf16(sc[2 * kk][2] * inv1, sc[2 * kk][3] * inv1);
    a[2] = pack_bf16(sc[2 * kk + 1][0] * inv0, sc[2 * kk + 1][1] * inv0);
    a[3] = pack_bf16(sc[2 * kk + 1][2] * inv1, sc[2 * kk + 1][3] * inv1);
    const KvTile tile = kv(kk);
#pragma unroll
    for (int np = 0; np < HD / 16; ++np) {  // two 8-wide dim tiles per ldmatrix.x4.trans
      uint32_t b0, b1, b2, b3;
      const int r = tile.row + (lane & 7) + 8 * ((lane >> 3) & 1), c = 2 * np + (lane >> 4);
      ldsm_x4_t(tile.v + swz(r, c), b0, b1, b2, b3);
      mma_bf16_16816(o[2 * np], a, b0, b1);
      mma_bf16_16816(o[2 * np + 1], a, b2, b3);
    }
  }
  // ---- stage O into the tile's (now dead) Q rows ----
  __syncwarp();
#pragma unroll
  for (int n = 0; n < HD / 8; ++n) {
    const int r0 = mt * 16 + g, r1 = r0 + 8;
    *reinterpret_cast<uint32_t*>(sQ + swz(r0, n) + 4 * t) = pack_bf16(o[n][0], o[n][1]);
    *reinterpret_cast<uint32_t*>(sQ + swz(r1, n) + 4 * t) = pack_bf16(o[n][2], o[n][3]);
  }
}

constexpr int MMA_WARPS = 4;  // (b, head) pairs per CTA

// NTQ = ceil(n_q / 16) query tiles, NTK = ceil(n_kv / 16) key tiles
template <int NTQ, int NTK>
__global__ void __launch_bounds__(MMA_WARPS * 32) attention_mma_kernel(const __grid_constant__ AttnParams p) {
  PDL_PROLOGUE();
  constexpr int QP = NTQ * 16, KP = NTK * 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pair = blockIdx.x * MMA_WARPS + warp;
  if (pair >= p.B * p.n_head) return;
  const int b = pair / p.n_head, h = pair - b * p.n_head;
  const int n_q = p.n_q, S = p.n_kv;
  uint8_t* sQ = smem_att + static_cast<size_t>(warp) * (QP + 2 * KP) * 256;
  uint8_t* sK = sQ + QP * 256;
  uint8_t* sV = sK + KP * 256;
  const uint32_t uQ = smem_u32(sQ), uK = smem_u32(sK), uV = smem_u32(sV);

  // ---- stage Q, K, V: 16 chunks of 16 bytes per row; pad rows are zeroed ----
  // A row's address is derived ONCE, by the lane whose index is the row (parameter loads, the group division, a 64-bit multiply),
  // and fetched with two shuffles by the lanes that copy its chunks -- not re-derived for each of its 16 chunks.
  constexpr int QSL = (QP + 31) / 32, KSL = (KP + 31) / 32;
  const char *qrow[QSL], *krow[KSL], *vrow[KSL];
#pragma unroll
  for (int sl = 0; sl < QSL; ++sl) {
    const int i = sl * 32 + lane;
    qrow[sl] = i < n_q ? reinterpret_cast<const char*>(p.q[i].ptr) + (tok_off(p.q[i], b) + h * HD) * 2 : nullptr;
  }
#pragma unroll
  for (int sl = 0; sl < KSL; ++sl) {
    const int i = sl * 32 + lane;
    krow[sl] = i < S ? reinterpret_cast<const char*>(p.k[i].ptr) + (tok_off(p.k[i], b) + h * HD) * 2 : nullptr;
    vrow[sl] = i < S ? reinterpret_cast<const char*>(p.v[i].ptr) + (tok_off(p.v[i], b) + h * HD) * 2 : nullptr;
  }
  auto shfl_ptr = [](const char* ptr, int src) -> const char* {
    const unsigned long long v = reinterpret_cast<unsigned long long>(ptr);
    const unsigned lo = __shfl_sync(0xffffffffu, static_cast<unsigned>(v), src), hi = __shfl_sync(0xffffffffu, static_cast<unsigned>(v >> 32), src);
    return reinterpret_cast<const char*>((static_cast<unsigned long long>(hi) << 32) | lo);
  };
  const int cchunk = lane & 15, rhalf = lane >> 4;
#pragma unroll
  for (int i = 0; i < QP / 2; ++i) {  // rows rhalf + 2 i: the slot of a row is a compile-time constant of i
    const int r = rhalf + 2 * i;
    const char* src = shfl_ptr(qrow[i >> 4], r & 31);
    if (r < n_q)
      cp_async16(uQ + swz(r, cchunk), src + cchunk * 16);
    else
      *reinterpret_cast<uint4*>(sQ + swz(r, cchunk)) = make_uint4(0, 0, 0, 0);
  }
#pragma unroll
  for (int i = 0; i < KP / 2; ++i) {
    const int r = rhalf + 2 * i;
    const uint32_t off = swz(r, cchunk);
    const char* ks = shfl_ptr(krow[i >> 4], r & 31);
    const char* vs = shfl_ptr(vrow[i >> 4], r & 31);
    if (r < S) {
      cp_async16(uK + off, ks + cchunk * 16);
      cp_async16(uV + off, vs + cchunk * 16);
    } else {
      *reinterpret_cast<uint4*>(sK + off) = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(sV + off) = make_uint4(0, 0, 0, 0);
    }
  }
  cp_async_commit();
  cp_async_wait_all();
  __syncwarp();

#pragma unroll 1
  for (int mt = 0; mt < NTQ; ++mt) attend_q_tile<NTK>(static_cast<size_t>(sQ - smem_att), uQ, mt, [=](int jp) { return KvTile{uK, uV, jp * 16, jp * 16, S}; }, lane);
  __syncwarp();
  // ---- coalesced copy-out: 16 lanes x 16 bytes per row ----
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(p.out);
  const int D = p.n_head * HD;
  for (int idx = lane; idx < n_q * 16; idx += 32) {
    const int r = idx >> 4, c = idx & 15;
    const uint4 v = *reinterpret_cast<const uint4*>(sQ + swz(r, c));
    *reinterpret_cast<uint4*>(out + (static_cast<size_t>(r) * p.B + b) * D + h * HD + c * 8) = v;
  }
}

// Variant for attention whose keys / values are mostly shared between batch rows: the planner's restricted decoder layer (19 of
// 32 keys are batch-constant mask-token rows at the shipped sizes) and the first encoder block of pass 2 (9 of 13 keys are the
// history tokens of the row's environment).  One CTA works on ONE head for SH_WARPS batch rows: the constant K / V tiles are staged once per CTA and
// shared by its warps; every warp stages only its own batch row's keys (one query tile).  Key order is [per-batch keys, constant
// keys] (softmax and P V are invariant to a common permutation of keys and values); each key tile is homogeneous.
constexpr int SH_WARPS = 8;
template <int NTB, int NTC>
__global__ void __launch_bounds__(SH_WARPS * 32) attention_mma_shared_kernel(const __grid_constant__ AttnParams p) {
  PDL_PROLOGUE();
  constexpr int NTK = NTB + NTC, BP = NTB * 16, CP = NTC * 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.y;
  const int n_q = p.n_q, n_b = p.n_kv_batch, n_c = p.n_kv - p.n_kv_batch;
  uint8_t* sKc = smem_att;             // CP x 256 B, shared by the CTA
  uint8_t* sVc = sKc + CP * 256;
  uint8_t* sQ = sVc + CP * 256 + static_cast<size_t>(warp) * (16 + 2 * BP) * 256;
  uint8_t* sKb = sQ + 16 * 256;
  uint8_t* sVb = sKb + BP * 256;
  const uint32_t uKc = smem_u32(sKc), uVc = smem_u32(sVc), uQ = smem_u32(sQ), uKb = smem_u32(sKb), uVb = smem_u32(sVb);

  // persistent over a contiguous range of 8-row blocks: the shared tiles are staged only when their source changes (never for
  // batch-constant rows, once per environment for per-group rows) and the CTA launch cost is paid once
  const int nblk = (p.B + SH_WARPS - 1) / SH_WARPS;
  const int bx_lo = static_cast<int>(static_cast<long long>(blockIdx.x) * nblk / gridDim.x);
  const int bx_hi = static_cast<int>(static_cast<long long>(blockIdx.x + 1) * nblk / gridDim.x);
  int cur_grp = -1;
  // Row descriptors, one per lane and slot: combined list [queries 0 .. n_q) | per-batch keys 0 .. n_b)] (n_q <= 16, n_b <= 32).
  // The copy loops below fetch a row's address with two shuffles instead of re-deriving it (parameter loads, a division and a
  // 64-bit multiply) for every 16-byte chunk -- the kernel was bound by exactly that integer work, not by memory
  // (profiles/r2j: 'wait' / 'short_scoreboard' stalls on the address arithmetic, 6 % on the cp.async wait).
  const char* rbase[2];
  long long rstride[2], vdelta[2];
  int rdiv[2];
#pragma unroll
  for (int sl = 0; sl < 2; ++sl) {
    const int i = sl * 32 + lane;
    rbase[sl] = nullptr; rstride[sl] = 0; vdelta[sl] = 0; rdiv[sl] = 0;
    if (i < n_q) {
      rbase[sl] = reinterpret_cast<const char*>(p.q[i].ptr) + h * HD * 2;
      rstride[sl] = static_cast<long long>(p.q[i].bstride) * 2;
      rdiv[sl] = p.q[i].bdiv;
    } else if (i < n_q + n_b) {
      const AttnTok& tk = p.k[i - n_q];
      rbase[sl] = reinterpret_cast<const char*>(tk.ptr) + h * HD * 2;
      rstride[sl] = static_cast<long long>(tk.bstride) * 2;
      rdiv[sl] = tk.bdiv;
      vdelta[sl] = reinterpret_cast<const char*>(p.v[i - n_q].ptr) - reinterpret_cast<const char*>(tk.ptr);
    }
  }
  // pad rows are zeroed ONCE: per-batch K / V pad rows are never written again; Q pad rows later hold finite leftovers of the
  // staged output, which only feed their own (discarded) score rows
  for (int idx = lane; idx < 16 * 16; idx += 32)
    if ((idx >> 4) >= n_q) *reinterpret_cast<uint4*>(sQ + swz(idx >> 4, idx & 15)) = make_uint4(0, 0, 0, 0);
  for (int idx = lane; idx < BP * 16; idx += 32)
    if ((idx >> 4) >= n_b) {
      *reinterpret_cast<uint4*>(sKb + swz(idx >> 4, idx & 15)) = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(sVb + swz(idx >> 4, idx & 15)) = make_uint4(0, 0, 0, 0);
    }
  __syncwarp();
  const int cchunk = lane & 15, rhalf = lane >> 4;
  const int D_out = p.n_head * HD;
  auto row_ptr = [&](const char* const (&rp)[2], int i) -> const char* {  // address of combined row i for this iteration's batch row
    unsigned long long v = reinterpret_cast<unsigned long long>(rp[0]);
    unsigned lo = __shfl_sync(0xffffffffu, static_cast<unsigned>(v), i & 31), hi = __shfl_sync(0xffffffffu, static_cast<unsigned>(v >> 32), i & 31);
    if (NTB > 1) {  // rows 32 .. 47 live in slot 1
      const unsigned long long w = reinterpret_cast<unsigned long long>(rp[1]);
      const unsigned lo1 = __shfl_sync(0xffffffffu, static_cast<unsigned>(w), i & 31), hi1 = __shfl_sync(0xffffffffu, static_cast<unsigned>(w >> 32), i & 31);
      if (i >= 32) { lo = lo1; hi = hi1; }
    }
    return reinterpret_cast<const char*>((static_cast<unsigned long long>(hi) << 32) | lo);
  };
#pragma unroll 1
  for (int bx = bx_lo; bx < bx_hi; ++bx) {
    const int b_raw = bx * SH_WARPS + warp;
    const bool live = b_raw < p.B;
    const int b = live ? b_raw : p.B - 1;  // idle warps shadow the last row (they must reach the barriers) and store nothing
    // keys / values shared by the CTA's batch rows: batch-constant rows (bstride 0) or one row per group of bdiv batch rows
    // (bdiv is a multiple of SH_WARPS, so the 8 rows of a block belong to one group)
    const int b_cta = min(bx * SH_WARPS, p.B - 1);
    const int grp_id = p.k[n_b].bdiv > 0 ? b_cta / p.k[n_b].bdiv : 0;
    const bool restage = grp_id != cur_grp;
    if (restage) {
      if (cur_grp != -1) __syncthreads();  // every warp has finished reading the previous tiles
      cur_grp = grp_id;
      for (int idx = threadIdx.x; idx < CP * 16; idx += SH_WARPS * 32) {
        const int r = idx >> 4, c = idx & 15;
        const uint32_t off = swz(r, c);
        if (r < n_c) {
          const AttnTok& tk = p.k[n_b + r];
          const AttnTok& tv = p.v[n_b + r];
          cp_async16(uKc + off, reinterpret_cast<const __nv_bfloat16*>(tk.ptr) + (tk.bdiv > 0 ? tok_off(tk, b_cta) : 0) + h * HD + c * 8);
          cp_async16(uVc + off, reinterpret_cast<const __nv_bfloat16*>(tv.ptr) + (tv.bdiv > 0 ? tok_off(tv, b_cta) : 0) + h * HD + c * 8);
        } else {
          *reinterpret_cast<uint4*>(sKc + off) = make_uint4(0, 0, 0, 0);
          *reinterpret_cast<uint4*>(sVc + off) = make_uint4(0, 0, 0, 0);
        }
      }
    }
    const char* rp[2];  // this iteration's address of the lane's rows
    long long vd[2];
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) {
      rp[sl] = rbase[sl] + static_cast<long long>(rdiv[sl] > 0 ? b / rdiv[sl] : b) * rstride[sl];
      vd[sl] = vdelta[sl];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {  // queries of this warp's batch row: rows rhalf + 2 i, the lane's 16-byte chunk of each
      const int r = rhalf + 2 * i;
      const char* src = row_ptr(rp, r);
      if (r < n_q) cp_async16(uQ + swz(r, cchunk), src + cchunk * 16);
    }
#pragma unroll
    for (int i = 0; i < BP / 2; ++i) {  // per-batch keys / values
      const int r = rhalf + 2 * i, ri = n_q + r;
      const char* src = row_ptr(rp, ri);
      long long dv = __shfl_sync(0xffffffffu, vd[0], ri & 31);
      if (NTB > 1) {
        const long long dv1 = __shfl_sync(0xffffffffu, vd[1], ri & 31);
        if (ri >= 32) dv = dv1;
      }
      if (r < n_b) {
        const uint32_t off = swz(r, cchunk);
        cp_async16(uKb + off, src + cchunk * 16);
        cp_async16(uVb + off, src + dv + cchunk * 16);
      }
    }
    cp_async_commit();
    cp_async_wait_all();
    if (restage) __syncthreads(); else __syncwarp();

    // per-batch key tiles first, then the shared ones
    attend_q_tile<NTK>(static_cast<size_t>(sQ - smem_att), uQ, 0, [=](int jp) {
      return jp < NTB ? KvTile{uKb, uVb, jp * 16, 0, n_b - 16 * jp} : KvTile{uKc, uVc, (jp - NTB) * 16, 0, n_c - 16 * (jp - NTB)};
    }, lane);
    __syncwarp();
    if (live) {
      char* orow = reinterpret_cast<char*>(p.out) + ((static_cast<size_t>(rhalf) * p.B + b) * D_out + h * HD) * 2 + cchunk * 16;
      const size_t ostep = static_cast<size_t>(2) * p.B * D_out * 2;  // two query rows further
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = rhalf + 2 * i;
        if (r < n_q) *reinterpret_cast<uint4*>(orow + i * ostep) = *reinterpret_cast<const uint4*>(sQ + swz(r, cchunk));
      }
    }
    __syncwarp();  // the copy-out has read this warp's tiles before the next block's loads overwrite them
  }  // bx
}

template <int NTB, int NTC>
int launch_mma_shared(const AttnParams& p, cudaStream_t st, int* info) {
  constexpr int smem = 2 * NTC * 16 * 256 + SH_WARPS * (16 + 2 * NTB * 16) * 256;
  static PerDevice<size_t> smem_limit;
  M3PC_CHECK_CUDA(raise_smem_limit(attention_mma_shared_kernel<NTB, NTC>, smem_limit, smem));
  const int nblk = ceil_div(p.B, SH_WARPS);
  const int per_sm = std::max(1, (227 * 1024) / (smem + 1024));
  // one wave of resident CTAs, each walking a range of row blocks -- once there are enough blocks for the ranges to balance
  // (>= 4 per CTA); smaller problems keep one block per CTA
  const int wave = std::max(1, ceil_div(per_sm * device_num_sms(), p.n_head));
  const int gx = nblk >= 4 * wave ? wave : nblk;
  M3PC_CHECK_CUDA(launch_k(attention_mma_shared_kernel<NTB, NTC>, dim3(gx, p.n_head), dim3(SH_WARPS * 32), smem, st, p));
  M3PC_CHECK_LAUNCH();
  report_launch(info, 2, NTB, NTC, gx);
  return M3PC_OK;
}

template <int NTQ, int NTK>
int launch_mma(const AttnParams& p, cudaStream_t st, int* info) {
  constexpr int smem = MMA_WARPS * (NTQ + 2 * NTK) * 16 * 256;
  static PerDevice<size_t> smem_limit;
  M3PC_CHECK_CUDA(raise_smem_limit(attention_mma_kernel<NTQ, NTK>, smem_limit, smem));
  const int gx = ceil_div(p.B * p.n_head, MMA_WARPS);
  M3PC_CHECK_CUDA(launch_k(attention_mma_kernel<NTQ, NTK>, dim3(gx), dim3(MMA_WARPS * 32), smem, st, p));
  M3PC_CHECK_LAUNCH();
  report_launch(info, 1, NTQ, NTK, gx);
  return M3PC_OK;
}

template <int NTK>
int dispatch_q(const AttnParams& p, cudaStream_t st, int* info) {
  switch ((p.n_q + 15) / 16) {
    case 1: return launch_mma<1, NTK>(p, st, info);
    case 2: return launch_mma<2, NTK>(p, st, info);
    case 3: return launch_mma<3, NTK>(p, st, info);
    default: return launch_mma<4, NTK>(p, st, info);
  }
}

}  // namespace

int launch_attention_gather(const AttnParams& p, bool bf16, cudaStream_t st, int* launched) {
  M3PC_REQUIRE(p.B > 0 && p.n_q > 0 && p.n_kv > 0 && p.n_q <= MAX_TOK && p.n_kv <= MAX_TOK && p.n_head > 0, "attention: bad shape (<= 64 tokens)");
  if (!bf16) return launch_simple(p, st, launched);
  if (p.n_kv_batch > 0 && p.n_q <= 16 && p.B >= 64) {  // batch keys first, constant keys after (see AttnParams)
    const int n_c = p.n_kv - p.n_kv_batch, ntb = (p.n_kv_batch + 15) / 16, ntc = (n_c + 15) / 16;
    // The constant keys must all have one form: batch-constant, or per-group with one common bdiv (a multiple of SH_WARPS, so
    // the 8 rows of a block share a group).  The kernel decides when to restage the shared tiles from the first constant key.
    const int cdiv = n_c > 0 ? p.k[p.n_kv_batch].bdiv : 0;
    bool ok = n_c >= 8 && ntb <= 2 && ntc <= 3 && cdiv % SH_WARPS == 0;
    for (int j = 0; j < p.n_kv && ok; ++j)
      ok = j < p.n_kv_batch ? (p.k[j].bstride == p.v[j].bstride && p.k[j].bdiv == p.v[j].bdiv)  // K and V of a token move together
                            : (p.k[j].bdiv == cdiv && p.v[j].bdiv == cdiv && (cdiv > 0 || (p.k[j].bstride == 0 && p.v[j].bstride == 0)));
    if (ok) {
      switch (ntb * 10 + ntc) {
        case 11: return launch_mma_shared<1, 1>(p, st, launched);
        case 12: return launch_mma_shared<1, 2>(p, st, launched);
        case 13: return launch_mma_shared<1, 3>(p, st, launched);
        case 21: return launch_mma_shared<2, 1>(p, st, launched);
        case 22: return launch_mma_shared<2, 2>(p, st, launched);
        default: return launch_mma_shared<2, 3>(p, st, launched);
      }
    }
  }
  switch ((p.n_kv + 15) / 16) {
    case 1: return dispatch_q<1>(p, st, launched);
    case 2: return dispatch_q<2>(p, st, launched);
    case 3: return dispatch_q<3>(p, st, launched);
    default: return dispatch_q<4>(p, st, launched);
  }
}

int launch_attention(const void* qkv, void* out, int B, int S, int n_head, bool bf16, cudaStream_t st) {
  M3PC_REQUIRE(B > 0 && S > 0 && S <= MAX_TOK && n_head > 0, "attention: bad shape (S must be <= 64)");
  const int D = n_head * HD;
  const size_t es = bf16 ? 2 : 4;
  AttnParams p{};
  p.n_q = p.n_kv = S;
  p.B = B;
  p.n_head = n_head;
  p.out = out;
  for (int s = 0; s < S; ++s) {
    const char* row = reinterpret_cast<const char*>(qkv) + static_cast<size_t>(s) * B * 3 * D * es;
    p.q[s] = AttnTok{row, 3 * D};
    p.k[s] = AttnTok{row + D * es, 3 * D};
    p.v[s] = AttnTok{row + 2 * D * es, 3 * D};
  }
  return launch_attention_gather(p, bf16, st);
}

}  // namespace m3pc
