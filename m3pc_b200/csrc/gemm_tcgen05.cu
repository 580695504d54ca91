// bf16 GEMM for sm_100a: C[M,N] = epilogue(A[M,K] * W[N,K]^T), fp32 accumulation in TMEM.
//
// This is the dense-contraction kernel of the MTM encoder/decoder blocks (reference call sites:
// nn.TransformerEncoderLayer QKV / out-proj / linear1 / linear2 at omtm/models/mtm_model.py:379-409,
// decoder_embed_dict at :646-661, output_head_dict[*].1 at :428-433).
//
// Persistent, warp-specialised, one CTA per SM (grid = min(tiles, #SM)); each CTA walks output tiles
// (128 x BN, n fastest so concurrently running CTAs share A panels and the whole weight in L2):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D loads of the A (128 x 64) and W (BN x 64) k-blocks into a
//               STAGES-deep shared-memory ring (SWIZZLE_128B), completion on `full` mbarriers.
//   warp 1      allocates TMEM (2 accumulators of BN fp32 columns), then one lane issues tcgen05.mma
//               (kind::f16, bf16 x bf16 -> fp32, M=128, N=BN, K=16 per instruction) from smem descriptors;
//               tcgen05.commit releases ring slots (`empty`) and publishes the accumulator (`acc_full`).
//   warps 2..9  epilogue, overlapped with the next tile's main loop through the second accumulator: tcgen05.ld
//               (each warp its own 32-lane TMEM quarter and half of the columns), transpose through a padded
//               smem tile so that global accesses are full 128-byte lines, fused bias / per-token table /
//               GELU(erf) / ReLU / residual add, 16-byte stores; `acc_empty` hands the accumulator back.
// Clusters: with CL > 1, CL CTAs of a thread-block cluster work on CL consecutive m-tiles of the same n-tile in lockstep;
// each loads 1/CL of the W k-block and TMA-multicasts it to all of them, so a W tile crosses the L2 -> SM fabric once per
// cluster instead of once per CTA (the GEMMs of this model are bound by that traffic, not by the tensor pipe: K is only
// 512..2048).  Ring slots are released cluster-wide: every CTA's tcgen05.commit multicast-arrives on all `empty` barriers.
// Both operands are K-major, which is the layout the activations (row-major (rows, K)) and nn.Linear weights
// ((out, in) row-major) already have -- no transposes anywhere.  Rows beyond M are zero-filled by TMA and masked
// in the epilogue, so M is arbitrary (ragged candidate counts, B = 1).
#include <cuda.h>

#include <cmath>

#include "common.cuh"
#include "tcgen05.cuh"

namespace m3pc {

namespace {

constexpr int NUM_EPI_WARPS = 8;
constexpr int GEMM_THREADS = 32 * (2 + NUM_EPI_WARPS);
constexpr int XPOSE_LD = 36;  // floats per staged row: 128-bit accesses are bank-conflict free both row- and column-wise

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode_tiled = nullptr;

struct EpiParams {
  const float* bias;
  const float* table;
  int rows_per_group;
  int flags;
};

template <int BN, int STAGES>
struct SmemLayout {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kXposeOffset = STAGES * kStageBytes;
  static constexpr int kXposeBytesPerWarp = 32 * XPOSE_LD * 4;
  static constexpr int kBarOffset = kXposeOffset + NUM_EPI_WARPS * kXposeBytesPerWarp;
  static constexpr int kTotal = kBarOffset + 256 + 1024;  // barriers + alignment slack
};

__device__ __forceinline__ float apply_act(float v, bool do_gelu, bool do_relu) {
  if (do_gelu) v = gelu_erf_fast(v);
  if (do_relu) v = fmaxf(v, 0.0f);
  return v;
}

// One epilogue warp's share of a 128 x BN accumulator tile: TMEM lanes [32*quarter, +32) (= rows), columns
// [half*BN/2, +BN/2), in chunks of 32 columns: tcgen05.ld -> padded smem transpose -> fused epilogue -> 16-byte coalesced stores.
template <int BN>
__device__ __forceinline__ void epilogue_tile(uint32_t tmem_acc, float* xp, void* C, int M, int N, int m0, int n0, int quarter, int half,
                                              int lane, const EpiParams& ep) {
  const bool do_gelu = ep.flags & EPI_GELU, do_relu = ep.flags & EPI_RELU, do_res = ep.flags & EPI_RESIDUAL;
  const bool out_f32 = do_res || (ep.flags & EPI_OUT_F32);
  const int row_base = m0 + quarter * 32;
#pragma unroll 1
  for (int c = 0; c < BN / 2; c += 32) {
    const int col_in_tile = half * (BN / 2) + c;
    const int col0 = n0 + col_in_tile;
    // residual rows are independent of the accumulator: issue all 8 coalesced loads first so their DRAM/L2 latency
    // overlaps the TMEM load and the transpose (lane -> 4 consecutive columns, 8 lanes per row, 4 rows per pass)
    float4 res[8];
    if (do_res) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int row = row_base + 4 * i + (lane >> 3);
        res[i] = (row < M) ? *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(C) + static_cast<size_t>(row) * N + col0 + 4 * (lane & 7))
                           : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    uint32_t r[32];
    tmem_ld32(tmem_acc + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(col_in_tile), r);
    tmem_ld_wait();
    // row-per-lane -> staging tile (lane = row)
#pragma unroll
    for (int j = 0; j < 8; ++j)
      *reinterpret_cast<uint4*>(xp + lane * XPOSE_LD + 4 * j) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
    __syncwarp();
    if (out_f32) {
      // lane -> 4 consecutive columns, 8 lanes per row, 4 rows per pass
      const int cc = 4 * (lane & 7);
      float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ep.bias != nullptr) b4 = __ldg(reinterpret_cast<const float4*>(ep.bias + col0 + cc));
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rr = 4 * i + (lane >> 3);
        const int row = row_base + rr;
        float4 v = *reinterpret_cast<const float4*>(xp + rr * XPOSE_LD + cc);
        if (row < M) {
          v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
          if (ep.table != nullptr) {
            const float4 t4 = __ldg(reinterpret_cast<const float4*>(ep.table + static_cast<size_t>(row / ep.rows_per_group) * N + col0 + cc));
            v.x += t4.x; v.y += t4.y; v.z += t4.z; v.w += t4.w;
          }
          v.x = apply_act(v.x, do_gelu, do_relu); v.y = apply_act(v.y, do_gelu, do_relu);
          v.z = apply_act(v.z, do_gelu, do_relu); v.w = apply_act(v.w, do_gelu, do_relu);
          float* cp = reinterpret_cast<float*>(C) + static_cast<size_t>(row) * N + col0 + cc;
          if (do_res) { v.x += res[i].x; v.y += res[i].y; v.z += res[i].z; v.w += res[i].w; }
          *reinterpret_cast<float4*>(cp) = v;
        }
      }
    } else {
      // lane -> 8 consecutive columns, 4 lanes per row, 8 rows per pass
      const int cc = 8 * (lane & 3);
      float bb[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (ep.bias != nullptr) {
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(ep.bias + col0 + cc));
        const float4 b1 = __ldg(reinterpret_cast<const float4*>(ep.bias + col0 + cc + 4));
        bb[0] = b0.x; bb[1] = b0.y; bb[2] = b0.z; bb[3] = b0.w; bb[4] = b1.x; bb[5] = b1.y; bb[6] = b1.z; bb[7] = b1.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rr = 8 * i + (lane >> 2);
        const int row = row_base + rr;
        const float4 v0 = *reinterpret_cast<const float4*>(xp + rr * XPOSE_LD + cc);
        const float4 v1 = *reinterpret_cast<const float4*>(xp + rr * XPOSE_LD + cc + 4);
        if (row < M) {
          float v[8] = {v0.x + bb[0], v0.y + bb[1], v0.z + bb[2], v0.w + bb[3], v1.x + bb[4], v1.y + bb[5], v1.z + bb[6], v1.w + bb[7]};
          if (ep.table != nullptr) {
            const float* tr = ep.table + static_cast<size_t>(row / ep.rows_per_group) * N + col0 + cc;
            const float4 t0 = __ldg(reinterpret_cast<const float4*>(tr));
            const float4 t1 = __ldg(reinterpret_cast<const float4*>(tr + 4));
            v[0] += t0.x; v[1] += t0.y; v[2] += t0.z; v[3] += t0.w; v[4] += t1.x; v[5] += t1.y; v[6] += t1.z; v[7] += t1.w;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = apply_act(v[j], do_gelu, do_relu);
          *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(C) + static_cast<size_t>(row) * N + col0 + cc) =
              make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
        }
      }
    }
    __syncwarp();  // staging tile is reused by the next chunk
  }
}

template <int BN, int STAGES, int CL>
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_a,
                                                                    const __grid_constant__ CUtensorMap tmap_w,
                                                                    void* __restrict__ C, int M, int N, int K, EpiParams ep) {
  using L = SmemLayout<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb = K / BK;
  const int n_tiles = N / BN;
  // work unit = CL consecutive m-tiles x one n-tile; the CTAs of a cluster walk the same unit sequence in lockstep
  const int total_tiles = n_tiles * (((M + BM - 1) / BM + CL - 1) / CL);
  const uint32_t crank = CL > 1 ? cluster_ctarank() : 0u;
  const int unit0 = blockIdx.x / CL, unit_step = gridDim.x / CL;

  const auto pipe = TcPipeline<STAGES, 2, BN, 1, CL>::setup(smem + L::kBarOffset, NUM_EPI_WARPS, [&] {
    prefetch_tmap(&tmap_a);
    prefetch_tmap(&tmap_w);
  });

  if (warp == 0) {
    if (lane == 0) {
      int m0 = 0, n0 = 0;
      pipe.produce(unit0, total_tiles, unit_step, [&](int tile) {
        m0 = ((tile / n_tiles) * CL + static_cast<int>(crank)) * BM;
        n0 = (tile % n_tiles) * BN;
        return num_kb;
      }, [&](int kb, int s) {
        mbar_arrive_expect_tx(&pipe.full[s], L::kStageBytes);
        uint8_t* sa = smem + s * L::kStageBytes;
        tma_load_2d(sa, &tmap_a, &pipe.full[s], kb * BK, m0);
        if (CL == 1) {
          tma_load_2d(sa + L::kABytes, &tmap_w, &pipe.full[s], kb * BK, n0);
        } else {  // my 1/CL slice of the W k-block, delivered to every CTA of the cluster
          constexpr int kSliceRows = BN / CL;
          tma_load_2d_mc(sa + L::kABytes + crank * (kSliceRows * BK * 2), &tmap_w, &pipe.full[s], kb * BK,
                         n0 + static_cast<int>(crank) * kSliceRows, static_cast<uint16_t>((1u << CL) - 1u));
        }
      });
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BN);
      pipe.issue(unit0, total_tiles, unit_step, [&](int) { return num_kb; }, [&](uint32_t tmem_d, int kb, int s) {
        const uint32_t a_addr = smem_u32(smem + s * L::kStageBytes);
        const uint32_t b_addr = a_addr + L::kABytes;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          // advance inside the 128-byte swizzle atom: +32 bytes per K=16 step
          umma_bf16(tmem_d, make_smem_desc(a_addr + k * UMMA_K * 2), make_smem_desc(b_addr + k * UMMA_K * 2), idesc,
                    (kb | k) != 0 ? 1u : 0u);
        }
      });
    }
  } else {
    // ---- epilogue warps: TMEM -> registers -> smem transpose -> coalesced global ----
    const int ew = warp - 2;
    const int quarter = warp & 3;       // TMEM lanes [32*quarter, 32*quarter+32) are the ones this warp may read
    const int half = ew >> 2;           // which half of the BN columns
    float* xp = reinterpret_cast<float*>(smem + L::kXposeOffset + ew * L::kXposeBytesPerWarp);
    uint32_t it = 0;
    for (int tile = unit0; tile < total_tiles; tile += unit_step, ++it) {
      const int m0 = ((tile / n_tiles) * CL + static_cast<int>(crank)) * BM, n0 = (tile % n_tiles) * BN;
      const uint32_t a = pipe.acc_wait(it);
      epilogue_tile<BN>(pipe.tmem_base + a * BN, xp, C, M, N, m0, n0, quarter, half, lane, ep);
      pipe.acc_release(a);
    }
  }
  pipe.teardown();
}


// ======================================================================================================================
// CTA-pair kernel (cta_group::2) -- the production path for M > 128, N % 256 == 0.
// A cluster of two CTAs owns a 256 x 256 output tile: one tcgen05.mma of the leader multiplies the pair's 256 x 16 A slab
// with a 256-wide W slab of which each CTA holds (and loads) only half, so a CTA stages 32 KB per k-block instead of 48 KB.
// Epilogue (measured to be what bounds these K = 512 .. 2048 GEMMs, profiles/r1b_*): each of the 8 epilogue warps drains its
// 32-lane x 128-column share of the accumulator in 32-column chunks -- tcgen05.ld (lane = row) -> bias / row table /
// activation in registers -> 16-byte shared-memory stores into a hardware-swizzled staging box (conflict free) -> one TMA
// bulk tensor store per chunk, double buffered.  The residual epilogue never loads C: the staged tile is added to the fp32
// residual stream in L2 by a TMA reduce-add (cp.reduce.async.bulk.tensor .add), one rounding, same result as load-add-store.
// The bias of the tile's columns is staged in shared memory once per tile, before the accumulator is waited for.
constexpr int NUM_EPI_WARPS_2SM = 16;  // 4 per TMEM lane quarter: enough warps per scheduler to hide TMEM / fence / store latencies
constexpr int GEMM_THREADS_2SM = 32 * (2 + NUM_EPI_WARPS_2SM);

template <int STAGES>
struct Smem2 {
  static constexpr int kABlk = BM * BK * 2;   // this CTA's 128 rows of one A k-block
  static constexpr int kBBlk = 128 * BK * 2;  // this CTA's 128 of the 256 W rows of one k-block
  static constexpr int kStageBytes = kABlk + kBBlk;
  static constexpr int kStoreBufBytes = 32 * 64;  // one staged chunk: 32 rows x 64 bytes (16 fp32 or 32 bf16 columns), SWIZZLE_64B
  static constexpr int kStoreOffset = STAGES * kStageBytes;
  static constexpr int kBiasOffset = kStoreOffset + NUM_EPI_WARPS_2SM * 2 * kStoreBufBytes;
  static constexpr int kBarOffset = kBiasOffset + NUM_EPI_WARPS_2SM * 64 * 4;
  static constexpr int kTotal = kBarOffset + 256 + 1024;
};

// Grouped launches: up to kMaxGroup independent problems (own operands, output, epilogue, shapes) share one launch; the pair's
// unit range simply runs across problem boundaries, so several small GEMMs of the decoder / heads / critic cost one kernel
// boundary instead of one each.
struct alignas(64) GroupProblem {
  CUtensorMap ta, tw, tc;
  const float* bias;
  const float* table;
  int rows_per_group, flags;
  int M, n_tiles;  // rows; N / 256
  int num_kb;      // k-blocks (K / 64)
  int unit0;       // first unit of this problem in the launch-wide unit order
};
struct GroupParams {
  GroupProblem p[kMaxGroup];
  int n, n_units;
  int strided;  // 1: pair p works on units p, p + n_pairs, ... (see launch_2sm) instead of one contiguous range
};
struct UnitCoord { int g, mp, nt; };
__device__ __forceinline__ UnitCoord decode_unit(const GroupParams& gp, int u) {
  UnitCoord c;
  c.g = problem_of(gp, u);
  const GroupProblem& P = gp.p[c.g];
  // unsigned: a unit index is never negative, and the signed division's sign fix-up costs registers the epilogue warps need
  // for their per-unit state (with it, ptxas spills that state to local memory)
  const unsigned lu = static_cast<unsigned>(u - P.unit0), nt = static_cast<unsigned>(P.n_tiles);
  c.mp = static_cast<int>(lu / nt);
  c.nt = static_cast<int>(lu - static_cast<unsigned>(c.mp) * nt);
  return c;
}

// Epilogue values of CW columns of one row: accumulator words r + bias (staged in shared memory at sbias) + row table, then GELU
// and ReLU as the flags ask.
template <int CW>
__device__ __forceinline__ void epilogue_values(const uint32_t (&r)[32], const float* sbias, const EpiParams& ep, int row, int M, int N,
                                                int col0, bool do_gelu, bool do_relu, float (&v)[CW]) {
#pragma unroll
  for (int j = 0; j < CW / 4; ++j) {
    const float4 b4 = *reinterpret_cast<const float4*>(sbias + 4 * j);
    v[4 * j + 0] = __uint_as_float(r[4 * j + 0]) + b4.x;
    v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + b4.y;
    v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + b4.z;
    v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + b4.w;
  }
  if (ep.table != nullptr && row < M) {
    const float* tr = ep.table + static_cast<size_t>(row / ep.rows_per_group) * N + col0;
#pragma unroll
    for (int j = 0; j < CW / 4; ++j) {
      const float4 t4 = __ldg(reinterpret_cast<const float4*>(tr + 4 * j));
      v[4 * j + 0] += t4.x; v[4 * j + 1] += t4.y; v[4 * j + 2] += t4.z; v[4 * j + 3] += t4.w;
    }
  }
  if (do_gelu) {
#pragma unroll
    for (int j = 0; j < CW; ++j) v[j] = gelu_erf_tanh(v[j]);
  }
  if (do_relu) {
#pragma unroll
    for (int j = 0; j < CW; ++j) v[j] = fmaxf(v[j], 0.0f);
  }
}

template <int STAGES>
__global__ void __launch_bounds__(GEMM_THREADS_2SM, 1) gemm_bf16_2sm_kernel(const __grid_constant__ GroupParams gp) {
  constexpr int BN = 256;
  using L = Smem2<STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int n_units = gp.n_units;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  // units are ordered m-major and split contiguously: a pair mostly stays on one row block, whose A slab stays hot in L2
  // strided (N = 512 problems with a long K): neighbouring pairs take the two column tiles of the SAME row block at the same
  // time, so its A slab is fetched from HBM once and the second reader hits L2 (contiguous ranges re-read it ~150 MB later)
  const int u_step = gp.strided ? n_pairs : 1;
  const int u_lo = gp.strided ? pair : static_cast<int>(static_cast<long long>(pair) * n_units / n_pairs);
  const int u_hi = gp.strided ? n_units : static_cast<int>(static_cast<long long>(pair + 1) * n_units / n_pairs);

  // 2 accumulators of 256 fp32 columns = all of TMEM; the leader's acc_empty counts both CTAs' epilogue warps
  const auto pipe = TcPipeline<STAGES, 2, BN, 2, 2>::setup(smem + L::kBarOffset, NUM_EPI_WARPS_2SM, [&] {
    for (int g = 0; g < gp.n; ++g) {
      prefetch_tmap(&gp.p[g].ta);
      prefetch_tmap(&gp.p[g].tw);
      prefetch_tmap(&gp.p[g].tc);
    }
  });

  if (warp == 0) {
    if (lane == 0) {
      // ---- TMA producer (both CTAs): own half of every operand slab, completion signalled on the LEADER's barrier ----
      const uint32_t full_leader = mapa_u32(smem_u32(&pipe.full[0]), 0);
      const GroupProblem* P = nullptr;
      int m0 = 0, n0 = 0;
      pipe.produce(u_lo, u_hi, u_step, [&](int u) -> const int& {
        const UnitCoord uc = decode_unit(gp, u);
        P = &gp.p[uc.g];
        m0 = (uc.mp * 2 + static_cast<int>(crank)) * BM;
        n0 = uc.nt * BN + static_cast<int>(crank) * 128;
        return P->num_kb;
      }, [&](int kb, int s) {
        if (leader) mbar_arrive_expect_tx(&pipe.full[s], 2u * L::kStageBytes);
        uint8_t* dst = smem + s * L::kStageBytes;
        const uint32_t bar = full_leader + 8u * static_cast<uint32_t>(s);
        tma_load_2d_2sm(dst, &P->ta, bar, kb * BK, m0);
        tma_load_2d_2sm(dst + L::kABlk, &P->tw, bar, kb * BK, n0);
      });
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      // ---- MMA issuer (leader only) ----
      constexpr uint32_t idesc = make_idesc_mn(2 * BM, BN);
      pipe.issue(u_lo, u_hi, u_step, [&](int u) { return gp.p[decode_unit(gp, u).g].num_kb; }, [&](uint32_t tmem_d, int kb, int s) {
        const uint32_t a_addr = smem_u32(smem + s * L::kStageBytes);
        const uint32_t b_addr = a_addr + L::kABlk;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k)
          umma_bf16_2sm(tmem_d, make_smem_desc(a_addr + k * UMMA_K * 2), make_smem_desc(b_addr + k * UMMA_K * 2), idesc, (kb | k) != 0 ? 1u : 0u);
      });
    }
  } else {
    // ---- epilogue warps (both CTAs): 32 rows (TMEM lane quarter) x 64 columns of this CTA's 128 x 256 tile each ----
    const int ew = warp - 2;
    const int quarter = warp & 3;  // TMEM lanes [32*quarter, +32) are the ones this warp may read
    const int cgrp = ew >> 2;      // which 64 of the tile's 256 columns
    uint8_t* sbuf = smem + L::kStoreOffset + ew * 2 * L::kStoreBufBytes;
    float* sbias = reinterpret_cast<float*>(smem + L::kBiasOffset) + ew * 64;
    const uint32_t sw = static_cast<uint32_t>((lane >> 1) & 3);  // SWIZZLE_64B: 16-byte chunk j of row r lives at j ^ ((r >> 1) & 3)
    uint32_t it = 0;
    uint32_t nstore = 0;  // chunks staged so far (selects the staging buffer)
    for (int u = u_lo; u < u_hi; u += u_step, ++it) {
      const UnitCoord uc = decode_unit(gp, u);
      const GroupProblem& P = gp.p[uc.g];
      const CUtensorMap* tmap_c = &P.tc;
      const int M = P.M, N = P.n_tiles * BN;
      EpiParams ep{P.bias, P.table, P.rows_per_group, P.flags};
      const bool do_gelu = ep.flags & EPI_GELU, do_relu = ep.flags & EPI_RELU, do_res = ep.flags & EPI_RESIDUAL;
      const bool out_f32 = do_res || (ep.flags & EPI_OUT_F32);
      const int cw = out_f32 ? 16 : 32;  // columns per staged chunk (64 bytes of output)
      const int row0 = (uc.mp * 2 + static_cast<int>(crank)) * BM + quarter * 32;
      const int colw = uc.nt * BN + cgrp * 64;  // first column of this warp's share
      // bias of my 64 columns -> shared memory (the previous tile's reads are done: same warp, program order)
      {
        float2 b2 = make_float2(0.f, 0.f);
        if (ep.bias != nullptr) b2 = __ldg(reinterpret_cast<const float2*>(ep.bias + colw + 2 * lane));
        *reinterpret_cast<float2*>(sbias + 2 * lane) = b2;
        __syncwarp();
      }
      const uint32_t a = pipe.acc_wait(it);
      const bool live = row0 < M;
      const int row = row0 + lane;
      const uint32_t tacc = pipe.tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + a * BN + static_cast<uint32_t>(cgrp * 64);
      if (live) {
#pragma unroll 1
        for (int c = 0; c < 64; c += cw) {
          const int col0 = colw + c;
          uint32_t r[32];
          if (out_f32) tmem_ld16(tacc + static_cast<uint32_t>(c), r); else tmem_ld32(tacc + static_cast<uint32_t>(c), r);
          // the staging buffer about to be overwritten was handed to the TMA two chunks ago: wait until it has been read
          uint8_t* buf = sbuf + (nstore & 1) * L::kStoreBufBytes;
          if (lane == 0) bulk_wait_read<1>();
          __syncwarp();
          tmem_ld_wait();
          if (c + cw == 64) pipe.acc_release(a);  // every TMEM read of this tile has landed in registers
          if (out_f32) {
            float v[16];
            epilogue_values<16>(r, sbias + c, ep, row, M, N, col0, do_gelu, do_relu, v);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<float4*>(buf + lane * 64 + ((static_cast<uint32_t>(j) ^ sw) << 4)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          } else {
            float v[32];
            epilogue_values<32>(r, sbias + c, ep, row, M, N, col0, do_gelu, do_relu, v);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              *reinterpret_cast<uint4*>(buf + lane * 64 + ((static_cast<uint32_t>(j) ^ sw) << 4)) =
                  make_uint4(pack_bf16(v[8 * j + 0], v[8 * j + 1]), pack_bf16(v[8 * j + 2], v[8 * j + 3]), pack_bf16(v[8 * j + 4], v[8 * j + 5]),
                             pack_bf16(v[8 * j + 6], v[8 * j + 7]));
            }
          }
          fence_proxy_async();  // my generic-proxy writes -> visible to the TMA (async proxy)
          __syncwarp();
          if (lane == 0) {
            if (do_res) tma_reduce_add_2d(tmap_c, buf, col0, row0); else tma_store_2d(tmap_c, buf, col0, row0);
            bulk_commit();
          }
          ++nstore;
        }
      } else {  // nothing to store (rows beyond M): just release the accumulator
        pipe.acc_release(a);
      }
    }
    if (lane == 0) bulk_wait_read<0>();  // shared memory may be released once the stores have been READ; the writes complete with the grid
  }
  pipe.teardown();  // no CTA may exit while its peer can still read its shared memory or arrive on its barriers
}

}  // namespace
namespace {
int make_tmap_operand(CUtensorMap* map, CUtensorMapDataType type, uint32_t elem_bytes, const void* ptr, uint64_t rows, uint64_t cols,
                      uint32_t box_rows) {
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * elem_bytes};
  cuuint32_t box[2] = {128u / elem_bytes, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode_tiled(map, type, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)) + " (rows=" +
              std::to_string(rows) + ", cols=" + std::to_string(cols) + ")");
    return M3PC_ERR_CUDA;
  }
  return M3PC_OK;
}
}  // namespace
int make_tmap(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  return make_tmap_operand(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ptr, rows, cols, box_rows);
}
int make_tmap_f32(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  return make_tmap_operand(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, ptr, rows, cols, box_rows);
}
namespace {

template <int BN, int STAGES, int CL>
int launch(const GemmProblem& q, cudaStream_t st, int* report) {
  using L = SmemLayout<BN, STAGES>;
  static_assert(L::kTotal <= 227 * 1024, "shared memory budget exceeded");
  static PerDevice<size_t> smem_limit;
  M3PC_CHECK_CUDA(raise_smem_limit(gemm_bf16_kernel<BN, STAGES, CL>, smem_limit, L::kTotal));
  CUtensorMap ta, tw;
  M3PC_TRY(make_tmap(&ta, q.A, static_cast<uint64_t>(q.M), static_cast<uint64_t>(q.K), BM));
  M3PC_TRY(make_tmap(&tw, q.W, static_cast<uint64_t>(q.N), static_cast<uint64_t>(q.K), BN / CL));
  const EpiParams ep{q.epi.bias, q.epi.table, q.epi.rows_per_group > 0 ? q.epi.rows_per_group : 1, q.epi.flags};
  const int units = (q.N / BN) * ceil_div(ceil_div(q.M, BM), CL);
  const int clusters = std::min(units, device_num_sms() / CL);
  M3PC_CHECK_CUDA(launch_k_cluster(CL, gemm_bf16_kernel<BN, STAGES, CL>, dim3(clusters * CL), dim3(GEMM_THREADS), L::kTotal, st, ta, tw, q.C,
                                   q.M, q.N, q.K, ep));
  M3PC_CHECK_LAUNCH();
  if (report != nullptr) { report[0] = 1; report[1] = BN; report[2] = CL; }
  return M3PC_OK;
}


// output tensor map: boxes of 32 rows x 64 bytes (16 fp32 / 32 bf16 columns), SWIZZLE_64B
}  // namespace
int make_tmap_out(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, bool f32) {
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * (f32 ? 4u : 2u)};
  cuuint32_t box[2] = {f32 ? 16u : 32u, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode_tiled(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ptr, gdim, gstride, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                              CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (output) failed with CUresult " + std::to_string(static_cast<int>(r)));
    return M3PC_ERR_CUDA;
  }
  return M3PC_OK;
}
namespace {

// One launch of the CTA-pair kernel over `n` problems (n <= kMaxGroup; every N a multiple of 256).
template <int STAGES>
int launch_2sm(const GemmProblem* probs, int n, cudaStream_t st, int* report) {
  using L = Smem2<STAGES>;
  static_assert(L::kTotal <= 227 * 1024, "shared memory budget exceeded");
  static_assert(sizeof(GroupParams) <= 4000, "kernel parameter space");
  static PerDevice<size_t> smem_limit;
  GroupParams gp{};
  gp.n = n;
  for (int g = 0; g < n; ++g) {
    const GemmProblem& q = probs[g];
    GroupProblem& P = gp.p[g];
    const bool out_f32 = (q.epi.flags & (EPI_RESIDUAL | EPI_OUT_F32)) != 0;
    M3PC_TRY(make_tmap(&P.ta, q.A, static_cast<uint64_t>(q.M), static_cast<uint64_t>(q.K), BM));
    M3PC_TRY(make_tmap(&P.tw, q.W, static_cast<uint64_t>(q.N), static_cast<uint64_t>(q.K), 128));
    M3PC_TRY(make_tmap_out(&P.tc, q.C, static_cast<uint64_t>(q.M), static_cast<uint64_t>(q.N), out_f32));
    P.bias = q.epi.bias;
    P.table = q.epi.table;
    P.rows_per_group = q.epi.rows_per_group > 0 ? q.epi.rows_per_group : 1;
    P.flags = q.epi.flags;
    P.M = q.M;
    P.n_tiles = q.N / 256;
    P.num_kb = q.K / BK;
  }
  M3PC_TRY(launch_pair(gemm_bf16_2sm_kernel<STAGES>, smem_limit, L::kTotal, GEMM_THREADS_2SM, gp,
                       [](const GroupProblem& P) { return P.n_tiles * ceil_div(P.M, 2 * BM); },
                       [&](int pairs) {
                         gp.strided = n == 1 && gp.p[0].n_tiles == 2 && probs[0].K >= 1024 && pairs % 2 == 0 && gp.n_units >= 2 * pairs;
                       }, st));
  for (int g = 0; report != nullptr && g < n; ++g) {
    report[4 * g] = 2; report[4 * g + 1] = gp.strided; report[4 * g + 2] = n;
  }
  return M3PC_OK;
}

// Modelled time of one configuration: the slower of the tensor pipe (rounds of the persistent grid x MMA cycles per tile)
// and the L2 -> SM operand stream (measured ~10.5 TB/s on B200 for this access pattern, profiles/README.md).
double model_time(int M, int N, int K, int bn, int cl) {
  const int m_tiles = ceil_div(M, BM);
  const int units = (N / bn) * ceil_div(m_tiles, cl);
  const int clusters = std::min(units, device_num_sms() / cl);
  const double rounds = std::ceil(static_cast<double>(units) / clusters);
  const double kb = K / BK;
  const double t_mma = rounds * kb * 4.0 * (bn / 2.0) / 1.7e9 + 2.0e-6;                          // 64 / 128 cycles per K=16 step
  const double bytes = static_cast<double>(units) * cl * kb * (BM * BK * 2.0 + bn * BK * 2.0 / cl);  // per CTA: own A + 1/cl of W
  return std::max(t_mma, bytes / 10.5e12);
}

// One problem in a launch of its own: the skinny kernel for a few rows, the CTA-pair kernel wherever a pair has two row tiles to
// work on and N splits into 256-wide tiles, else the single-CTA kernel.
int gemm_bf16_one(const GemmProblem& q, cudaStream_t st, int* report) {
  if (q.M <= 32 && static_cast<size_t>(q.M) * q.K * 2 <= 160 * 1024) {
    if (report != nullptr) { report[0] = 0; report[1] = 0; report[2] = 0; }
    return gemm_bf16_skinny(q.A, q.W, q.C, q.M, q.N, q.K, q.epi, st);
  }
  if (q.N % 256 == 0 && q.M > BM) return launch_2sm<4>(&q, 1, st, report);
  // pick tile width and cluster size by the modelled time (ties: wider tile, larger cluster = less L2 traffic)
  struct Cand { int bn, cl; } cands[] = {{256, 2}, {256, 1}, {128, 2}, {128, 1}};
  int best = -1;
  double best_t = 1e30;
  for (int i = 0; i < 4; ++i) {
    if (q.N % cands[i].bn != 0) continue;
    const double t = model_time(q.M, q.N, q.K, cands[i].bn, cands[i].cl);
    if (t < best_t * 0.98) { best_t = t; best = i; }
  }
  switch (best) {
    case 0: return launch<256, 3, 2>(q, st, report);
    case 1: return launch<256, 3, 1>(q, st, report);
    case 2: return launch<128, 4, 2>(q, st, report);
    default: return launch<128, 4, 1>(q, st, report);
  }
}

}  // namespace

int gemm_init_driver_api() {
  if (g_encode_tiled != nullptr) return M3PC_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  M3PC_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (qres != cudaDriverEntryPointSuccess || fn == nullptr) {
    set_error("cuTensorMapEncodeTiled not available from the CUDA driver");
    return M3PC_ERR_CUDA;
  }
  g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
  return M3PC_OK;
}

// Problems are taken kMaxGroup at a time.  Several problems whose N all split into 256-wide tiles share one CTA-pair launch (small
// ones included) once one of them gives a pair two row tiles to work on (see GroupParams); otherwise each problem gets its own.
// Every argument is checked before the first CUDA call: a bias or table the epilogues read with vector loads must be 16-byte aligned.
int gemm_bf16(const GemmProblem* probs, int n, cudaStream_t st, int* report) {
  M3PC_REQUIRE(n >= 1, "gemm_bf16: no problems");
  for (int g = 0; g < n; ++g) {
    const GemmProblem& q = probs[g];
    const GemmEpilogue& ep = q.epi;
    M3PC_REQUIRE(q.M > 0 && q.N > 0 && q.K > 0, "gemm_bf16: empty problem");
    M3PC_REQUIRE(q.K % BK == 0, "gemm_bf16: K must be a multiple of 64");
    M3PC_REQUIRE(q.N % 128 == 0, "gemm_bf16: N must be a multiple of 128");
    M3PC_REQUIRE(((reinterpret_cast<uintptr_t>(q.A) | reinterpret_cast<uintptr_t>(q.W) | reinterpret_cast<uintptr_t>(q.C)) & 15) == 0,
                 "gemm_bf16: operands must be 16-byte aligned");
    M3PC_REQUIRE((ep.flags & ~(EPI_GELU | EPI_RESIDUAL | EPI_RELU | EPI_ROWTABLE | EPI_OUT_F32)) == 0, "gemm_bf16: unknown flag");
    M3PC_REQUIRE((ep.table != nullptr) == ((ep.flags & EPI_ROWTABLE) != 0), "gemm_bf16: a table goes with EPI_ROWTABLE and only with it");
    M3PC_REQUIRE((ep.flags & (EPI_ROWTABLE | EPI_RESIDUAL)) != (EPI_ROWTABLE | EPI_RESIDUAL),
                 "gemm_bf16: a row table and the in-place residual exclude each other");
    M3PC_REQUIRE(ep.rows_per_group >= 1, "gemm_bf16: rows_per_group must be at least 1");
    M3PC_REQUIRE(((reinterpret_cast<uintptr_t>(ep.bias) | reinterpret_cast<uintptr_t>(ep.table)) & 15) == 0,
                 "gemm_bf16: bias and table must be 16-byte aligned");
  }
  M3PC_TRY(gemm_init_driver_api());
  int launches = 0;
  for (int i0 = 0; i0 < n; i0 += kMaxGroup) {
    const GemmProblem* group = probs + i0;
    int* rep = report != nullptr ? report + 4 * i0 : nullptr;
    const int m = std::min(kMaxGroup, n - i0);
    bool pair = m > 1;
    int max_m = 0;
    for (int g = 0; g < m; ++g) {
      pair = pair && group[g].N % 256 == 0;
      max_m = std::max(max_m, group[g].M);
    }
    if (pair && max_m > BM) {
      M3PC_TRY(launch_2sm<4>(group, m, st, rep));
      for (int g = 0; rep != nullptr && g < m; ++g) rep[4 * g + 3] = launches;
      ++launches;
    } else {
      for (int g = 0; g < m; ++g, ++launches) {
        M3PC_TRY(gemm_bf16_one(group[g], st, rep != nullptr ? rep + 4 * g : nullptr));
        if (rep != nullptr) rep[4 * g + 3] = launches;
      }
    }
  }
  return M3PC_OK;
}

}  // namespace m3pc
