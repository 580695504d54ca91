// fp32-grade GEMM on the sm_100a tensor cores (M3PC_PREC_TF32X3): C[M,N] = epilogue(A[M,K] * W[N,K]^T), A, W and C fp32,
// with the 3xTF32 split of both operands:
//   x_hi = x rounded to the nearest tf32 value, x_lo = x - x_hi (exact in fp32) rounded to the nearest tf32 value (both are exact
//          tf32 values, so it does not matter whether the tensor core truncates or rounds its inputs; |x_lo| <= 2^-11 |x|),
//   C    = A_lo W_hi + A_hi W_lo + A_hi W_hi   (three tcgen05.mma kind::tf32 per k-step, small terms first; A_lo W_lo, below
//                                               2^-22 of the product, is dropped).
// The sum over K is NOT left to the tensor memory accumulator: its additions lose accuracy at every MMA, an error that grows
// with K (measured on a B200 with the whole K in one TMEM accumulator: 3.6 .. 7.5x the fp32 FFMA error, 1e-5 relative at
// K = 2048; after this kernel's promotion 0.3 .. 0.6x, DESIGN.md section 4).  Every KB_PER_ACC k-blocks of 32 get an accumulator
// of their own (two alternate in TMEM, so the MMAs of one run while the epilogue warps drain the other), and the epilogue warps add
// these partial sums in fp32 registers, rounding to nearest.
// The operands are the fp32 activations and the fp32 weight arena as they are: the split happens in shared memory.
//
// The CTA-pair structure of the bf16 kernel (gemm_tcgen05.cu, TcPipeline): a cluster of two CTAs owns a 256 x 256 output tile,
// each CTA loads its 128 rows of A and its 128 of the 256 W rows per k-block of 32 fp32 (one 128-byte SWIZZLE_128B row, the same
// byte geometry as 64 bf16: descriptors and the +32 bytes per MMA k-step carry over; one kind::tf32 MMA takes K = 8).  The
// pipeline's unit is one accumulator: KB_PER_ACC k-blocks of one tile.
//   warp 0       TMA producer (both CTAs): A and W k-blocks into this CTA's ring stage, completion on its own `full` barrier.
//   warp 1       MMA issuer (leader CTA): waits on the stage's `split` barrier, issues 3 x 4 MMAs (M = 256, N = 256, K = 8)
//                per k-block into the unit's accumulator.
//   warps 2..3   split (both CTAs): rewrite the landed tiles in place to hi and write lo into the stage's second half, then
//                fence.proxy.async and arrive on the leader's `split` barrier (counting the split warps of both CTAs).
//   warps 4..19  epilogue (both CTAs): 32 TMEM lanes x 64 columns each: bias + row table, plus the tile's accumulators summed
//                in registers (64 running sums within the 96 registers a thread of 20 warps has), then GELU(erf, erff) / ReLU in
//                fp32 and a TMA store -- or, for the residual, a TMA reduce-add into C (one rounding, as load-add-store).
// Shared memory per stage: A hi + lo and W hi + lo, 4 x 16 KB; three stages and the epilogue's staging boxes fit in 227 KB.
//
// Problems with at most kTf32x3SmallRows rows (pass 1 of a plan at B = 1 .. 3 environments: a CTA pair would get half a row tile
// and most of the grid would idle), whose N is not a multiple of 256, or whose K is not a multiple of 4 (the TMA row stride must
// be a multiple of 16 bytes: the critic's first layer) run on the CUDA-core fp32 kernel (sgemm.cu), the same accuracy class.
#include <cuda.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace m3pc {

namespace {

constexpr int kTf32x3SmallRows = 128;
constexpr int TK = 32;  // fp32 k per k-block: 128 bytes
constexpr int TF32_K = 8;
constexpr int KB_PER_ACC = 2;  // k-blocks summed in one tensor-memory accumulator before the fp32 register promotion
constexpr int STAGES = 3;
constexpr int BN = 256;
constexpr int NUM_SPLIT_WARPS = 2;
constexpr int NUM_EPI_WARPS = 16;
constexpr int THREADS = 32 * (2 + NUM_SPLIT_WARPS + NUM_EPI_WARPS);

using Pipe = TcPipeline<STAGES, 2, BN, 2, 2>;

struct Layout {
  static constexpr int kTile = BM * TK * 4;       // 16 KB: 128 rows of one k-block
  static constexpr int kStageBytes = 4 * kTile;   // A hi | A lo | W hi | W lo
  static constexpr int kStoreBufBytes = 32 * 64;  // one staged chunk: 32 rows x 16 fp32, SWIZZLE_64B
  static constexpr int kStoreOffset = STAGES * kStageBytes;
  static constexpr int kBarOffset = kStoreOffset + NUM_EPI_WARPS * kStoreBufBytes;
  static constexpr int kSplitBarOffset = kBarOffset + 128;
  static constexpr int kLoopOffset = kSplitBarOffset + 8 * STAGES;  // the epilogue's loop bounds: the pair's tile bound, accumulators a tile
  static constexpr int kTotal = kLoopOffset + 8 + 1024;             // + alignment slack
  static_assert(Pipe::kBarBytes <= 128, "pipeline barriers");
};
static_assert(Layout::kTotal <= 227 * 1024, "shared memory budget exceeded");

struct Tf32Problem {
  CUtensorMap ta, tw, tc;
  const float* bias;
  const float* table;
  int rows_per_group, flags;
  int M, n_tiles, num_kb;
  int unit0;
};
struct Tf32Params {
  Tf32Problem p[1];
  int n, n_units;
};

// 8 columns of this warp's 32 TMEM lanes (the epilogue's running sums leave no room for wider loads at 96 registers)
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}

__device__ __forceinline__ int ld_shared_volatile(uint32_t addr) {
  int v;
  asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// one 16 KB tile in place -> hi, and lo into `lo` (elementwise: the swizzled layout is the same in both)
__device__ __forceinline__ void split_tile(uint8_t* tile, uint8_t* lo, int t) {
  float4* h4 = reinterpret_cast<float4*>(tile);
  float4* l4 = reinterpret_cast<float4*>(lo);
#pragma unroll 4
  for (int i = 0; i < Layout::kTile / 16 / (32 * NUM_SPLIT_WARPS); ++i) {
    const int idx = i * 32 * NUM_SPLIT_WARPS + t;
    const float4 x = h4[idx];
    const float4 h = make_float4(to_tf32(x.x), to_tf32(x.y), to_tf32(x.z), to_tf32(x.w));
    h4[idx] = h;
    l4[idx] = make_float4(to_tf32(x.x - h.x), to_tf32(x.y - h.y), to_tf32(x.z - h.z), to_tf32(x.w - h.w));
  }
}

__global__ void __launch_bounds__(THREADS, 1) gemm_tf32x3_kernel(const __grid_constant__ Tf32Params gp) {
  using L = Layout;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const Tf32Problem& P = gp.p[0];
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  // this pair's tiles [t_lo, t_hi) -- contiguous, so a pair mostly stays on one row block -- as units g = tile * num_kb + k-block
  // (32-bit: at most 74 pairs x a few thousand tiles; the 64-bit division costs the registers the epilogue sums need)
  const int t_lo = static_cast<int>(static_cast<unsigned>(pair) * static_cast<unsigned>(gp.n_units) / static_cast<unsigned>(n_pairs));
  const int t_hi = static_cast<int>(static_cast<unsigned>(pair + 1) * static_cast<unsigned>(gp.n_units) / static_cast<unsigned>(n_pairs));
  const int nkb = P.num_kb, nacc = (nkb + KB_PER_ACC - 1) / KB_PER_ACC;  // k-blocks, accumulators per tile
  const int g_lo = t_lo * nacc, g_hi = t_hi * nacc;
  uint64_t* split_bar = reinterpret_cast<uint64_t*>(smem + L::kSplitBarOffset);

  auto pipe = Pipe::setup(smem + L::kBarOffset, NUM_EPI_WARPS, [&] {
    prefetch_tmap(&P.ta);
    prefetch_tmap(&P.tw);
    prefetch_tmap(&P.tc);
    for (int s = 0; s < STAGES; ++s) mbar_init(&split_bar[s], 2 * NUM_SPLIT_WARPS);
    reinterpret_cast<int*>(smem + L::kLoopOffset)[0] = t_hi;
    reinterpret_cast<int*>(smem + L::kLoopOffset)[1] = nacc;
  });
  pipe.ready = split_bar;

  if (warp == 0) {
    if (lane == 0) {
      // ---- TMA producer (both CTAs): this CTA's 128 A rows and 128 W rows, completion on its own barrier ----
      int m0 = 0, n0 = 0, kb0 = 0, cnt = 0;
      pipe.produce(g_lo, g_hi, 1, [&](int g) -> const int& {
        const int t = g / nacc, mp = t / P.n_tiles, nt = t - mp * P.n_tiles;
        m0 = (mp * 2 + static_cast<int>(crank)) * BM;
        n0 = nt * BN + static_cast<int>(crank) * 128;
        kb0 = (g - t * nacc) * KB_PER_ACC;
        cnt = min(KB_PER_ACC, nkb - kb0);
        return cnt;
      }, [&](int kb, int s) {
        uint8_t* dst = smem + s * L::kStageBytes;
        mbar_arrive_expect_tx(&pipe.full[s], 2u * L::kTile);
        tma_load_2d(dst, &P.ta, &pipe.full[s], (kb0 + kb) * TK, m0);
        tma_load_2d(dst + 2 * L::kTile, &P.tw, &pipe.full[s], (kb0 + kb) * TK, n0);
      });
    }
  } else if (warp == 1) {
    if (lane == 0 && crank == 0) {
      // ---- MMA issuer (leader only): per k-step A_lo W_hi, A_hi W_lo, A_hi W_hi; the first MMA of a k-block overwrites ----
      constexpr uint32_t idesc = make_idesc_tf32(2 * BM, BN);
      int cnt = 0;
      pipe.issue(g_lo, g_hi, 1, [&](int g) -> const int& {
        cnt = min(KB_PER_ACC, nkb - (g % nacc) * KB_PER_ACC);
        return cnt;
      }, [&](uint32_t tmem_d, int kb, int s) {
        const uint32_t a_hi = smem_u32(smem + s * L::kStageBytes), a_lo = a_hi + L::kTile;
        const uint32_t w_hi = a_hi + 2 * L::kTile, w_lo = a_hi + 3 * L::kTile;
#pragma unroll
        for (int k = 0; k < TK / TF32_K; ++k) {
          const uint32_t o = k * TF32_K * 4;
          umma_tf32_2sm(tmem_d, make_smem_desc(a_lo + o), make_smem_desc(w_hi + o), idesc, (kb | k) != 0 ? 1u : 0u);
          umma_tf32_2sm(tmem_d, make_smem_desc(a_hi + o), make_smem_desc(w_lo + o), idesc, 1u);
          umma_tf32_2sm(tmem_d, make_smem_desc(a_hi + o), make_smem_desc(w_hi + o), idesc, 1u);
        }
      });
    }
  } else if (warp < 2 + NUM_SPLIT_WARPS) {
    // ---- split warps (both CTAs) ----
    const int t = threadIdx.x - 64;
    const uint32_t split_leader = mapa_u32(smem_u32(split_bar), 0);
    int s = 0;
    uint32_t ph = 0;
    for (int kb = t_lo * nkb; kb < t_hi * nkb; ++kb) {
      mbar_wait(&pipe.full[s], ph);
      uint8_t* st = smem + s * L::kStageBytes;
      split_tile(st, st + L::kTile, t);
      split_tile(st + 2 * L::kTile, st + 3 * L::kTile, t);
      fence_proxy_async();  // the generic-proxy writes -> visible to the MMAs (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_release(split_leader + 8u * static_cast<uint32_t>(s));
      if (++s == STAGES) { s = 0; ph ^= 1; }
    }
  } else {
    // ---- epilogue warps (both CTAs): 32 rows (TMEM lane quarter) x 64 columns of this CTA's 128 x 256 tile each ----
    const int ew = warp - 2 - NUM_SPLIT_WARPS;
    const int quarter = warp & 3;  // TMEM lanes [32*quarter, +32) are the ones this warp may read
    const int cgrp = ew >> 2;      // which 64 of the tile's 256 columns
    uint8_t* buf = smem + L::kStoreOffset + ew * L::kStoreBufBytes;
    const uint32_t sw = static_cast<uint32_t>((lane >> 1) & 3);  // SWIZZLE_64B: 16-byte chunk j of row r lives at j ^ ((r >> 1) & 3)
    const bool do_gelu = P.flags & EPI_GELU, do_relu = P.flags & EPI_RELU, do_res = P.flags & EPI_RESIDUAL;
    const int M = P.M, N = P.n_tiles * BN;
    uint32_t it = 0;
    // the loop bounds and the CTA rank are re-read where they are used: kept in registers across a tile they would push the 64
    // running sums over the 96-register budget of 20 warps
    const uint32_t loop_bounds = smem_u32(smem + L::kLoopOffset);
    for (int t = t_lo; t < ld_shared_volatile(loop_bounds); ++t) {
      const int mp = t / P.n_tiles, nt = t - mp * P.n_tiles;
      const int row0 = (mp * 2 + static_cast<int>(cluster_ctarank())) * BM + quarter * 32;
      const int colw = nt * BN + cgrp * 64;
      const int row = row0 + lane;
      // the sums start from bias + row table (loaded while the tile's first k-block is still in the tensor pipe)
      float sum[64];
#pragma unroll
      for (int j = 0; j < 64; j += 4) {
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (P.bias != nullptr) b4 = __ldg(reinterpret_cast<const float4*>(P.bias + colw + j));
        if (P.table != nullptr && row < M) {
          const float4 t4 = __ldg(reinterpret_cast<const float4*>(P.table + static_cast<size_t>(row / P.rows_per_group) * N + colw + j));
          b4.x += t4.x; b4.y += t4.y; b4.z += t4.z; b4.w += t4.w;
        }
        sum[j] = b4.x; sum[j + 1] = b4.y; sum[j + 2] = b4.z; sum[j + 3] = b4.w;
      }
      for (int g = 0; g < ld_shared_volatile(loop_bounds + 4); ++g, ++it) {
        const uint32_t a = pipe.acc_wait(it);
        const uint32_t tacc = pipe.tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + a * BN + static_cast<uint32_t>(cgrp * 64);
#pragma unroll
        for (int c = 0; c < 64; c += 8) {
          uint32_t r[8];
          tmem_ld8(tacc + static_cast<uint32_t>(c), r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) sum[c + j] += __uint_as_float(r[j]);
        }
        pipe.acc_release(a);  // every TMEM read of this accumulator has landed in registers
      }
      if (row0 >= M) continue;  // rows beyond M: nothing to store
#pragma unroll
      for (int c = 0; c < 64; c += 16) {
        const int col0 = colw + c;
        float* v = sum + c;  // the activation runs in place on the sums
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if (do_gelu) v[j] = gelu_erf(v[j]);
          if (do_relu) v[j] = fmaxf(v[j], 0.0f);
        }
        if (lane == 0) bulk_wait_read<0>();  // the staging box of the previous chunk has been read by the TMA
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(buf + lane * 64 + ((static_cast<uint32_t>(j) ^ sw) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        fence_proxy_async();  // my generic-proxy writes -> visible to the TMA (async proxy)
        __syncwarp();
        if (lane == 0) {
          if (do_res) tma_reduce_add_2d(&P.tc, buf, col0, row0); else tma_store_2d(&P.tc, buf, col0, row0);
          bulk_commit();
        }
      }
    }
    if (lane == 0) bulk_wait_read<0>();  // shared memory may be released once the stores have been READ; the writes complete with the grid
  }
  pipe.teardown();  // no CTA may exit while its peer can still read its shared memory or arrive on its barriers
}

}  // namespace

int gemm_tf32x3(const float* A, const float* W, float* C, int M, int N, int K, const GemmEpilogue& epi, cudaStream_t st) {
  M3PC_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_tf32x3: empty problem");
  M3PC_REQUIRE(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(C)) & 15) == 0,
               "gemm_tf32x3: operands must be 16-byte aligned");
  M3PC_REQUIRE(((reinterpret_cast<uintptr_t>(epi.bias) | reinterpret_cast<uintptr_t>(epi.table)) & 15) == 0,
               "gemm_tf32x3: bias and row table must be 16-byte aligned (the epilogue reads them as float4)");
  if (M <= kTf32x3SmallRows || N % BN != 0 || K % 4 != 0) return gemm_fp32(A, W, C, M, N, K, epi, st);
  M3PC_TRY(gemm_init_driver_api());
  static PerDevice<size_t> smem_limit;
  Tf32Params gp{};
  gp.n = 1;
  Tf32Problem& P = gp.p[0];
  M3PC_TRY(make_tmap_f32(&P.ta, A, static_cast<uint64_t>(M), static_cast<uint64_t>(K), BM));
  M3PC_TRY(make_tmap_f32(&P.tw, W, static_cast<uint64_t>(N), static_cast<uint64_t>(K), 128));
  M3PC_TRY(make_tmap_out(&P.tc, C, static_cast<uint64_t>(M), static_cast<uint64_t>(N), true));
  P.bias = epi.bias;
  P.table = epi.table;
  P.rows_per_group = epi.rows_per_group > 0 ? epi.rows_per_group : 1;
  P.flags = epi.flags;
  P.M = M;
  P.n_tiles = N / BN;
  P.num_kb = ceil_div(K, TK);  // a K tail is zero-filled by the TMA
  return launch_pair(gemm_tf32x3_kernel, smem_limit, Layout::kTotal, THREADS, gp,
                     [](const Tf32Problem& q) { return q.n_tiles * ceil_div(q.M, 2 * BM); }, [](int) {}, st);
}

}  // namespace m3pc
