// Tensor-core GEMM with a fused residual + LayerNorm epilogue (N = n_embd = 512):
//
//     X[M,512] (fp32)  <-  R + A[M,K] W[512,K]^T + bias          R = X (in place), other fp32 rows, or table[row / rows_per_group]
//     Y[M,512] (bf16)  <-  LayerNorm(X; gamma, beta)             eps 1e-5, statistics in fp32
//
// Reference call sites: the out-projection / linear2 of nn.TransformerEncoderLayer followed by the next pre-LN norm
// (mtm_model.py:379-409; norm_first: x = x + sa(norm1(x)); x = x + ff(norm2(x))).  The unfused path writes X through a TMA
// reduce-add (read-modify-write of 4 KB per row) and a separate LayerNorm kernel reads it again; here a CTA pair owns ALL 512
// columns of its rows, so the epilogue sees whole rows: it loads the residual tile through the TMA, adds, stores X, keeps the
// updated rows in TMEM (tcgen05.st), exchanges the row statistics between the warps that share a row, and writes the
// normalised bf16 operand of the next GEMM.  6 KB of HBM traffic per row and one launch instead of 8 KB and two.
//
// Two unit sizes (template parameter ROWS, chosen per launch in gemm_ln_bf16_grouped):
//   ROWS = 256  M = 256 MMAs; the unit's accumulator is the pair's whole tensor memory (128 lanes x 512 columns per CTA), so the
//               epilogue of a unit and the MMAs of the next take turns.  Least operand traffic per FLOP: right for long K.
//   ROWS = 128  M = 128 MMAs (cta_group::2).  Each CTA's 64 x N slice of D is stored as 128 lanes x N/2 columns (lanes 0-63:
//               columns [0, N/2); lanes 64-127: columns [N/2, N) -- the "2x2" datapath layout), so a 128-row x 512-column unit
//               takes 256 TMEM columns per CTA and TWO fit: the epilogue of unit u runs under the MMAs of unit u + 1.  Same tensor
//               pipe rate; W is streamed once per 128 rows instead of once per 256.  Right for K = 512, where the launch is
//               bound by the epilogue's 6 KB per row, and for launches too small to fill whole rounds of 256-row units.
// Per-element arithmetic (k order of the accumulation, fp32 epilogue) is the same in both: results are bit-identical.
// Tried and dropped (profiles/r2g_gemm_ln_variants.txt): pulling a unit's residual tile into L2 ahead of its epilogue
// (cp.async.bulk.prefetch.tensor by the producer warp, 8 k-blocks before the unit's last MMA) -- 147 vs 125 us (K = 512) and
// 252 vs 236 us (K = 2048) at 106 496 rows: the prefetched lines compete with the operand stream and are fetched twice.
//
// Structure (per CTA of the pair, 18 warps): warp 0 lane 0 = TMA producer (A: own ROWS / 2 rows; W: own 128 rows of each
// 256-row half), warp 1 lane 0 of the leader = MMA issuer (two tcgen05.mma cta_group::2 M = ROWS, N = 256, K = 16 per k-step,
// one per column half), warps 2..17 = epilogue (TMEM lane quarter q = warp % 4, group g = (warp - 2) / 4):
//   ROWS = 256  rows q * 32 + lane of the CTA's 128, columns g * 128 .. + 128 (a row is shared by 4 warps)
//   ROWS = 128  rows (q & 1) * 32 + lane of the CTA's 64, columns h * 256 + s * 128 + c0 .. + 64 with s = q >> 1 (lane half),
//               h = g >> 1 (which N = 256 MMA), c0 = (g & 1) * 64 (a row is shared by 8 warps)
#include "common.cuh"
#include "tcgen05.cuh"

namespace m3pc {

// rows per CTA-pair unit of the fused kernel: 0 = chosen per launch (gemm_ln_bf16_grouped), or 128 / 256 forced; m3pc_set_option
// "gemm_ln_unit_rows"
int g_ln_unit_rows = 0;

namespace {

constexpr int LN_N = 512;
constexpr int LN_EPI_WARPS = 16;
constexpr int LN_THREADS = 32 * (2 + LN_EPI_WARPS);

// One problem of a launch: X[M,512] <- R + A W^T + bias, Y <- LayerNorm(X).  Several problems share a launch (same K, bias, gamma,
// beta; own operands, outputs and residual source): the fixed cost of a launch -- barrier set-up, tensor-memory allocation,
// cluster sync, pipeline fill and drain, ~10 us -- is paid once for e.g. the table part and the per-candidate part of the first
// encoder block's out-projection, the decoder-embedding runs of the kept tokens, or the residual sources of the restricted decoder.
struct LnProblem {
  CUtensorMap ta, tw, tx, ty;
  CUtensorMap tr;      // residual source (fp32, same box shape as tx): X itself, or other rows (restricted decoder: the residual-stream
                       // rows of a kept token, read in place while the result goes to the compact needed-row block)
  const float* table;  // null: residual through tr
  int rows_per_group;
  int M;
  int unit0;           // first unit of this problem in the launch's unit order
};

struct LnGemmParams {
  LnProblem p[kMaxGroup];
  const float* bias;
  const float* gamma;
  const float* beta;
  int n, num_kb, n_units;
};
static_assert(sizeof(LnGemmParams) <= 4000, "kernel parameter space");

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

template <int ROWS, int STAGES, int NBOX>
struct SmemLn {
  static constexpr int kABlk = (ROWS / 2) * BK * 2;  // this CTA's ROWS / 2 rows of one A k-block
  static constexpr int kBBlk = 128 * BK * 2;         // 16 KB: this CTA's 128 rows of one 256-row half of W
  static constexpr int kStageBytes = kABlk + 2 * kBBlk;
  static constexpr int kBoxBytes = 32 * 64;
  static constexpr int kStoreOffset = STAGES * kStageBytes;
  static constexpr int kConstOffset = kStoreOffset + LN_EPI_WARPS * NBOX * kBoxBytes;
  static constexpr int kStatsOffset = kConstOffset + 3 * LN_N * 4;  // float2 [ROWS / 2 rows][8 column groups]
  static constexpr int kBarOffset = kStatsOffset + (ROWS / 2) * 8 * 8;
  static constexpr int kTotal = kBarOffset + 1024 + 1024;
};

template <int ROWS, int STAGES, int NBOX>
__global__ void __launch_bounds__(LN_THREADS, 1) gemm_ln_2sm_kernel(const __grid_constant__ LnGemmParams P) {
  static_assert(ROWS == 128 || ROWS == 256, "unit rows");
  using L = SmemLn<ROWS, STAGES, NBOX>;
  constexpr int NACC = ROWS == 128 ? 2 : 1;         // accumulators in tensor memory
  constexpr uint32_t ACC_COLS = LN_N / NACC;        // TMEM columns of one accumulator
  constexpr int NSHARE = ROWS == 128 ? 8 : 4;       // warps that share a row
  constexpr int WCOLS = LN_N / NSHARE;              // output columns per warp
  // Row statistics are accumulated in a CANONICAL order that does not depend on ROWS, so both unit sizes produce identical bits: each
  // group ("slice") of 64 consecutive columns gets its sum and its sum of squared deviations from its own mean, built from its four
  // 16-column chunks in ascending order (Chan et al.'s pairwise update), and the row's variance adds the eight slices' deviations in
  // column order around the row mean.  Centred sums, which m3pc_layernorm and nn.LayerNorm use as well, keep the variance accurate for
  // rows whose mean is large against their spread, where E[x^2] - mean^2 cancels catastrophically in fp32.
  constexpr int NSLICE = 8;
  using Pipe = TcPipeline<STAGES, NACC, ACC_COLS, 2, 2>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* res_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset + Pipe::kBarBytes);  // [LN_EPI_WARPS][NBOX]: residual box landed
  float* sconst = reinterpret_cast<float*>(smem + L::kConstOffset);
  float2* sstats = reinterpret_cast<float2*>(smem + L::kStatsOffset);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

  for (int i = threadIdx.x; i < LN_N; i += LN_THREADS) {
    sconst[i] = P.bias != nullptr ? __ldg(P.bias + i) : 0.f;
    sconst[LN_N + i] = __ldg(P.gamma + i);
    sconst[2 * LN_N + i] = __ldg(P.beta + i);
  }
  // all 512 TMEM columns: two accumulators of 256 columns (one 128-row x 512-column unit each) or one of 512
  const Pipe pipe = Pipe::setup(smem + L::kBarOffset, LN_EPI_WARPS, [&] {
    for (int g = 0; g < P.n; ++g) {
      prefetch_tmap(&P.p[g].ta);
      prefetch_tmap(&P.p[g].tw);
      prefetch_tmap(&P.p[g].tx);
      prefetch_tmap(&P.p[g].ty);
      prefetch_tmap(&P.p[g].tr);
    }
    for (int i = 0; i < NBOX * LN_EPI_WARPS; ++i) mbar_init(&res_bar[i], 1);
  });

  if (warp == 0) {
    if (lane == 0) {
      // ---- TMA producer (both CTAs): own 64 rows of A, own 128 rows of each 256-row half of W ----
      const uint32_t full_leader = mapa_u32(smem_u32(&pipe.full[0]), 0);
      const LnProblem* Q = nullptr;
      int m0 = 0;
      pipe.produce(pair, P.n_units, n_pairs, [&](int u) -> const int& {
        Q = &P.p[problem_of(P, u)];
        m0 = ((u - Q->unit0) * 2 + static_cast<int>(crank)) * (ROWS / 2);
        return P.num_kb;
      }, [&](int kb, int s) {
        if (leader) mbar_arrive_expect_tx(&pipe.full[s], 2u * L::kStageBytes);
        uint8_t* dst = smem + s * L::kStageBytes;
        const uint32_t bar = full_leader + 8u * static_cast<uint32_t>(s);
        tma_load_2d_2sm(dst, &Q->ta, bar, kb * BK, m0);
        tma_load_2d_2sm(dst + L::kABlk, &Q->tw, bar, kb * BK, static_cast<int>(crank) * 128);
        tma_load_2d_2sm(dst + L::kABlk + L::kBBlk, &Q->tw, bar, kb * BK, 256 + static_cast<int>(crank) * 128);
      });
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      // ---- MMA issuer (leader only): M = ROWS across the pair, both N = 256 halves per k-step, accumulators alternate ----
      constexpr uint32_t idesc = make_idesc_mn(ROWS, 256);
      pipe.issue(pair, P.n_units, n_pairs, [&](int) -> const int& { return P.num_kb; }, [&](uint32_t d0, int kb, int s) {
        const uint32_t a_addr = smem_u32(smem + s * L::kStageBytes);
        const uint32_t b0_addr = a_addr + L::kABlk, b1_addr = b0_addr + L::kBBlk;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint32_t acc = (kb | k) != 0 ? 1u : 0u;
          const uint64_t da = make_smem_desc(a_addr + k * UMMA_K * 2);
          umma_bf16_2sm(d0, da, make_smem_desc(b0_addr + k * UMMA_K * 2), idesc, acc);
          umma_bf16_2sm(d0 + ACC_COLS / 2, da, make_smem_desc(b1_addr + k * UMMA_K * 2), idesc, acc);
        }
      });
    }
  } else {
    // ---- epilogue warps (both CTAs): 32 rows x WCOLS columns each ----
    const int ew = warp - 2;
    const int q = warp & 3;
    const int grp = ew >> 2;
    // ROWS = 128 ("2x2" layout): lanes [0, 64) hold columns [0, 128) of each N = 256 MMA and lanes [64, 128) columns [128, 256), so
    // quarter q covers rows (q & 1) * 32 .. and the lane half q >> 1 selects the column half; ROWS = 256: lane = row
    const int rowq = ROWS == 128 ? (q & 1) : q;         // which block of 32 rows of this CTA
    const int lanehalf = ROWS == 128 ? (q >> 1) : 0;
    const int colw = ROWS == 128 ? (grp >> 1) * 256 + lanehalf * 128 + (grp & 1) * 64 : grp * 128;   // first output column of this warp
    const uint32_t tcol = static_cast<uint32_t>(ROWS == 128 ? (grp >> 1) * 128 + (grp & 1) * 64 : grp * 128);  // its TMEM column inside an accumulator
    const int slice = colw / 64;                                                           // first 64-column group of this warp
    uint8_t* sbuf = smem + L::kStoreOffset + ew * NBOX * L::kBoxBytes;
    uint64_t* rbar = res_bar + NBOX * ew;
    uint32_t rph = 0;  // bit b: parity of rbar[b]
    const uint32_t sw = static_cast<uint32_t>((lane >> 1) & 3);  // SWIZZLE_64B: 16-byte chunk j of row r lives at j ^ ((r >> 1) & 3)
    const float* sbias = sconst;
    const float* sgamma = sconst + LN_N;
    const float* sbeta = sconst + 2 * LN_N;
    constexpr int NB1 = WCOLS / 16;             // residual / X boxes per warp per unit (16 fp32 columns each)
    constexpr int NB2 = WCOLS / 32;             // Y boxes (32 bf16 columns each)
    constexpr int NPRE = NBOX < NB1 ? NBOX : NB1;  // boxes requested before the accumulator is waited for
    uint32_t it = 0;
    // Box buffers are used strictly round-robin (buffer = ns % NBOX for the ns-th bulk group this warp commits), which is what makes
    // "wait until at most NBOX - 1 groups are still being read" the condition for reusing one.  With the residual coming through the
    // TMA every unit starts from a drained state (ns = 0, all buffers free).
    uint32_t ns = 0;
    for (int u = pair; u < P.n_units; u += n_pairs, ++it) {
      const LnProblem& Q = P.p[problem_of(P, u)];
      const bool from_x = Q.table == nullptr;
      const int row0 = ((u - Q.unit0) * 2 + static_cast<int>(crank)) * (ROWS / 2) + rowq * 32;
      const int row = row0 + lane;
      const bool live = row0 < Q.M;
      // residual boxes travel to shared memory while the MMAs of this unit (and the epilogue of the previous one) still run
      if (from_x) ns = 0;
      if (from_x && live && lane == 0) {
        bulk_wait_read<0>();  // every buffer's last store has been read
#pragma unroll
        for (int b = 0; b < NPRE; ++b) {
          mbar_arrive_expect_tx(&rbar[b], L::kBoxBytes);
          tma_load_2d(sbuf + b * L::kBoxBytes, &Q.tr, &rbar[b], colw + b * 16, row0);
        }
      }
      const uint32_t buf = pipe.acc_wait(it);
      const uint32_t tacc = pipe.tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * ACC_COLS + tcol;
      float s1 = 0.f, s2 = 0.f;
      if (live) {
        // ---- pass 1: x = acc + bias + residual -> X (TMA store) and back into TMEM; row sums ----
#pragma unroll 1
        for (int ci = 0; ci < NB1; ++ci) {
          const int col0 = colw + ci * 16;
          const int b = static_cast<int>(ns % NBOX);
          uint8_t* bx = sbuf + b * L::kBoxBytes;
          uint32_t r[32];
          tmem_ld16(tacc + static_cast<uint32_t>(ci * 16), r);
          if (from_x) {
            mbar_wait(&rbar[b], (rph >> b) & 1u);
            rph ^= 1u << b;
          } else {
            if (lane == 0) bulk_wait_read<NBOX - 1>();  // the store issued from this buffer NBOX boxes ago has been read
            __syncwarp();
          }
          tmem_ld_wait();
          float v[16];
          const float* trow = (from_x || Q.table == nullptr) ? nullptr : Q.table + static_cast<size_t>(min(row, Q.M - 1) / Q.rows_per_group) * LN_N + col0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float4* slot = reinterpret_cast<float4*>(bx + lane * 64 + ((static_cast<uint32_t>(j) ^ sw) << 4));
            const float4 res = from_x ? *slot : (trow != nullptr ? __ldg(reinterpret_cast<const float4*>(trow + 4 * j)) : make_float4(0.f, 0.f, 0.f, 0.f));
            const float4 b4 = *reinterpret_cast<const float4*>(sbias + col0 + 4 * j);
            v[4 * j + 0] = __uint_as_float(r[4 * j + 0]) + b4.x + res.x;
            v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + b4.y + res.y;
            v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + b4.z + res.z;
            v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + b4.w + res.w;
            *slot = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
          {
            float c1 = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) c1 += v[j];
            const float cm = c1 * (1.0f / 16);
            float c2 = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) c2 = fmaf(v[j] - cm, v[j] - cm, c2);
            // merge this chunk (16 columns, mean cm) into the k = ci & 3 chunks of the slice so far (16 k columns, sum s1):
            // M2 += c2 + d^2 * 16 k / (k + 1), d = cm - s1 / (16 k); constants selected instead of divided
            const int k = ci & 3;
            const float inv_n = k == 1 ? 1.0f / 16 : (k == 2 ? 1.0f / 32 : 1.0f / 48);
            const float wgt = k == 1 ? 8.0f : (k == 2 ? 32.0f / 3 : 12.0f);
            const float d = cm - s1 * inv_n;
            s2 += k == 0 ? c2 : fmaf(d * d, wgt, c2);
            s1 += c1;
          }
          if ((ci & 3) == 3) {  // a 64-column group is complete
            sstats[(rowq * 32 + lane) * NSLICE + slice + (ci >> 2)] = make_float2(s1, s2);
            s1 = s2 = 0.f;
          }
          tmem_st16(tacc + static_cast<uint32_t>(ci * 16), v);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&Q.tx, bx, col0, row0);
            bulk_commit();
            if (from_x && ci + NBOX < NB1) {  // this buffer is needed again for a later residual box of the unit
              bulk_wait_read<0>();
              mbar_arrive_expect_tx(&rbar[b], L::kBoxBytes);
              tma_load_2d(bx, &Q.tr, &rbar[b], col0 + NBOX * 16, row0);
            }
          }
          ++ns;
        }
        tmem_st_wait();
      }
      // ---- row statistics across the NSHARE warps that share these 32 rows ----
      if (!live) {
#pragma unroll
        for (int g = 0; g < WCOLS / 64; ++g) sstats[(rowq * 32 + lane) * NSLICE + slice + g] = make_float2(0.f, 0.f);
      }
      named_bar_sync(1 + rowq, 32 * NSHARE);
      float mean, rstd;
      {
        const float2* rs = sstats + (rowq * 32 + lane) * NSLICE;
        float t1 = 0.f;
#pragma unroll
        for (int g = 0; g < NSLICE; ++g) t1 += rs[g].x;
        mean = t1 * (1.0f / LN_N);
        float t2 = 0.f;
#pragma unroll
        for (int g = 0; g < NSLICE; ++g) {
          const float d = rs[g].x * (1.0f / 64) - mean;
          t2 += rs[g].y + 64.0f * d * d;
        }
        rstd = rsqrtf(t2 * (1.0f / LN_N) + kLnEps);
      }
      named_bar_sync(1 + rowq, 32 * NSHARE);  // everybody has read the statistics: the next unit may overwrite them
      if (live) {
        // ---- pass 2: y = (x - mean) * rstd * gamma + beta -> bf16 -> Y ----
#pragma unroll 1
        for (int ci = 0; ci < NB2; ++ci) {
          const int col0 = colw + ci * 32;
          uint8_t* bx = sbuf + (ns % NBOX) * L::kBoxBytes;
          uint32_t r[32];
          tmem_ld32(tacc + static_cast<uint32_t>(ci * 32), r);
          if (lane == 0) bulk_wait_read<NBOX - 1>();
          __syncwarp();
          tmem_ld_wait();
          if (ci == NB2 - 1) pipe.acc_release(buf);  // the accumulator has been drained: the MMA warp may reuse it
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float y[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int c = col0 + 8 * j + e;
              y[e] = (__uint_as_float(r[8 * j + e]) - mean) * rstd * sgamma[c] + sbeta[c];
            }
            *reinterpret_cast<uint4*>(bx + lane * 64 + ((static_cast<uint32_t>(j) ^ sw) << 4)) =
                make_uint4(pack_bf16(y[0], y[1]), pack_bf16(y[2], y[3]), pack_bf16(y[4], y[5]), pack_bf16(y[6], y[7]));
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&Q.ty, bx, col0, row0);
            bulk_commit();
          }
          ++ns;
        }
      } else {
        pipe.acc_release(buf);
      }
    }
    if (lane == 0) bulk_wait_read<0>();  // shared memory may be released once the stores have been read; the writes complete with the grid
  }

  pipe.teardown();
}

template <int ROWS, int STAGES, int NBOX>
int launch_ln(LnGemmParams& P, cudaStream_t st, int* report) {
  using L = SmemLn<ROWS, STAGES, NBOX>;
  static_assert(L::kTotal <= 227 * 1024, "shared memory budget exceeded");
  static_assert(L::kStoreOffset % 1024 == 0, "operand stages must keep 1024-byte alignment");
  static PerDevice<size_t> smem_limit;
  return launch_pair(gemm_ln_2sm_kernel<ROWS, STAGES, NBOX>, smem_limit, L::kTotal, LN_THREADS, P,
                     [](const LnProblem& Q) { return ceil_div(Q.M, ROWS); }, [&](int pairs) {
                       if (report != nullptr) { report[0] = ROWS; report[1] = pairs; }
                     }, st);
}

}  // namespace

// X (M, 512) fp32 in place (or other fp32 rows / table rows as the residual), Y (M, 512) bf16 = LayerNorm(X).  K % 64 == 0.
// Up to kMaxGroup problems per launch (shared K, bias, gamma, beta).
// Unit size (rows per CTA pair; bit-identical results, tests/test_gpu_parity.py::test_gemm_ln_unit_sizes_are_bit_identical):
//   K <= 512   128-row units: the launch is bound by its epilogue traffic (6 KB per row), which then runs under the next unit's MMAs
//              (measured at 106 496 rows: 125 us vs 135 us with 256-row units; profiles/r2g_gemm_ln_variants.txt)
//   K  > 512   256-row units feed the tensor pipe with 1/3 less operand traffic per FLOP (238 vs 264 us) -- unless the launch is so
//              small that whole 256-row units quantise badly on the 74 CTA pairs (26 624 rows: 104 units = 2 rounds, vs 3 half rounds)
int gemm_ln_bf16_grouped(const LnJob* jobs, int n, const float* bias, const float* gamma, const float* beta, int K, cudaStream_t st,
                         int* report) {
  M3PC_REQUIRE(n >= 1 && n <= kMaxGroup, "gemm_ln: 1 .. kMaxGroup problems per launch");
  M3PC_REQUIRE(K > 0 && K % BK == 0, "gemm_ln: K must be a positive multiple of 64");
  M3PC_REQUIRE(gamma && beta, "gemm_ln: null operand");
  for (int g = 0; g < n; ++g) {
    const LnJob& j = jobs[g];
    M3PC_REQUIRE(j.M > 0 && j.A && j.W && j.X && j.Y, "gemm_ln: null operand or empty problem");
    M3PC_REQUIRE(((reinterpret_cast<uintptr_t>(j.A) | reinterpret_cast<uintptr_t>(j.W) | reinterpret_cast<uintptr_t>(j.X) | reinterpret_cast<uintptr_t>(j.Y)) & 15) == 0,
                 "gemm_ln: operands must be 16-byte aligned");
    M3PC_REQUIRE(j.R == nullptr || j.table == nullptr, "gemm_ln: a residual source excludes a table");
    // the epilogue reads table rows with 16-byte loads
    M3PC_REQUIRE(((reinterpret_cast<uintptr_t>(j.R) | reinterpret_cast<uintptr_t>(j.table)) & 15) == 0, "gemm_ln: R and table must be 16-byte aligned");
    M3PC_REQUIRE(j.rows_per_group >= 1, "gemm_ln: rows_per_group must be at least 1");
  }
  M3PC_TRY(gemm_init_driver_api());
  int rows = g_ln_unit_rows;
  if (rows != 128 && rows != 256) {
    const int pairs = std::max(1, device_num_sms() / 2);
    int u256 = 0, u128 = 0;
    for (int g = 0; g < n; ++g) {
      u256 += ceil_div(jobs[g].M, 256);
      u128 += ceil_div(jobs[g].M, 128);
    }
    const double rounds256 = ceil_div(u256, pairs), rounds128 = 0.5 * ceil_div(u128, pairs);
    rows = (K <= 512 || rounds128 + 0.25 < rounds256) ? 128 : 256;
  }
  LnGemmParams P{};
  P.n = n;
  for (int g = 0; g < n; ++g) {
    const LnJob& j = jobs[g];
    LnProblem& Q = P.p[g];
    M3PC_TRY(make_tmap(&Q.ta, j.A, static_cast<uint64_t>(j.M), static_cast<uint64_t>(K), rows / 2));
    M3PC_TRY(make_tmap(&Q.tw, j.W, static_cast<uint64_t>(LN_N), static_cast<uint64_t>(K), 128));
    M3PC_TRY(make_tmap_out(&Q.tx, j.X, static_cast<uint64_t>(j.M), LN_N, true));
    M3PC_TRY(make_tmap_out(&Q.tr, const_cast<float*>(j.R != nullptr ? j.R : j.X), static_cast<uint64_t>(j.M), LN_N, true));
    M3PC_TRY(make_tmap_out(&Q.ty, j.Y, static_cast<uint64_t>(j.M), LN_N, false));
    Q.table = j.table;
    Q.rows_per_group = j.rows_per_group;
    Q.M = j.M;
  }
  P.bias = bias; P.gamma = gamma; P.beta = beta;
  P.num_kb = K / BK;
  return rows == 128 ? launch_ln<128, 3, 2>(P, st, report) : launch_ln<256, 3, 2>(P, st, report);
}

}  // namespace m3pc
