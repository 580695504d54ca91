// tcgen05 / TMA / mbarrier PTX wrappers shared by the sm_100a tensor-core kernels (gemm_tcgen05.cu, gemm_ln.cu, gemm_tf32x3.cu).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace m3pc {

constexpr int BM = 128;     // rows of one CTA's MMA tile (TMEM lanes)
constexpr int BK = 64;      // 64 bf16 = 128 bytes = one SWIZZLE_128B atom row
constexpr int UMMA_K = 16;  // K of one tcgen05.mma (kind::f16)

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(addr),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4, [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1),
//   [32,46) stride byte offset >> 4 (8 rows * 128 B = 1024), [46,48) version = 1, [61,64) layout = 2 (SW128).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// kind::f16 instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=bf16, both K-major.
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(BM >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }


// ---- cta_group::2 (CTA pair) variants --------------------------------------------------------------------------------
// shared::cta address -> shared::cluster address of the same location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// TMA load into this CTA's shared memory whose completion is signalled on an mbarrier of either CTA of the pair
// (`bar_cluster_addr` is a shared::cluster address, normally the leader's barrier)
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
// D[tmem, 256 x N split over the pair: 128 lanes in each CTA] (+)= A[256 x 16: 128 rows from each CTA's smem] * B[N x 16: N/2 rows
// from each CTA's smem]^T; issued by one thread of the leader CTA, descriptors are the leader's (same offsets in the peer).
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all prior MMAs of this thread have completed) on the barrier at the same offset in both CTAs of the pair
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(static_cast<uint16_t>(3))
               : "memory");
}
__host__ __device__ constexpr uint32_t make_idesc_mn(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): c_format [4,6) = F32 (1), a_format [7,10) = b_format [10,13) =
// TF32 (2 in UMMA::F16F32Format), both K-major, N >> 3 at bit 17, M >> 4 at bit 24.
__host__ __device__ constexpr uint32_t make_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
// as umma_bf16_2sm, kind::tf32: K = 8 fp32 (32 bytes) per instruction
__device__ __forceinline__ void umma_tf32_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on a barrier of another CTA of the cluster, releasing this thread's prior writes at cluster scope
__device__ __forceinline__ void mbar_arrive_remote_release(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// arrive on a barrier of the pair's leader CTA (CUTLASS ClusterBarrier::arrive form: no cluster-scope release fence -- the
// only thing ordered through it are TMEM reads, which tcgen05.wait::ld + tcgen05.fence::before_thread_sync already cover)
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

// GELU(erf) for the bf16 epilogues in 8 instructions (one MUFU): 0.5 x (1 + tanh(x (c0 + c1 x^2 + c2 x^4))) with x^2 capped at 16;
// coefficients fitted to the erf form (max |error| 2.5e-5 with an exact tanh; tanh.approx adds <= 2^-11 relative on tanh),
// an order of magnitude below the bf16 rounding of the stored result.  The fp32 precision mode uses erff().
__device__ __forceinline__ float gelu_erf_tanh(float x) {
  const float x2 = fminf(x * x, 16.0f);
  float q = fmaf(x2, -0.00035151679f, 0.037005646f);
  q = fmaf(x2, q, 0.79750788f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * q));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}

// ---- the pipeline every tensor-core GEMM kernel runs -----------------------------------------------------------------------------
// Warp 0 (one thread) streams the operands of each k-block through a STAGES-deep shared-memory ring (`full`: the stage's bytes have
// landed; `empty`: the MMAs that read it have completed).  Warp 1 (one thread; the leader CTA's with a CTA pair) issues the MMAs of
// a unit into one of NACC accumulators of ACC_COLS TMEM columns (`acc_full`: complete; `acc_empty`: every epilogue warp has read it),
// so with NACC = 2 the epilogue of one unit runs under the MMAs of the next.  Every role walks the same units u_lo, u_lo + u_step,
// ... < u_hi in order, which keeps their stage and accumulator indices in step.  The MMAs of a stage wait on `ready`, which is `full`
// unless the kernel points it at barriers of its own (a stage that is transformed in shared memory before the MMAs read it).  CG is
// the MMAs' cta_group (2: a CTA pair shares each MMA and its accumulator) and CL the CTAs of a cluster (CG = 1: CL CTAs multicast
// their operands to each other).
template <int STAGES, int NACC, int ACC_COLS, int CG, int CL>
struct TcPipeline {
  static_assert(CG == 1 || CL == 2, "a CTA pair is a cluster of two");
  static constexpr uint32_t kTmemCols = NACC * ACC_COLS;
  static constexpr int kBarBytes = 8 * (2 * STAGES + 2 * NACC + 1);  // the barriers and the TMEM address slot
  uint64_t* full;
  uint64_t* empty;
  uint64_t* acc_full;
  uint64_t* acc_empty;
  uint64_t* ready;
  uint32_t acc_empty_leader;  // CG = 2: shared::cluster address of the leader's acc_empty
  uint32_t tmem_base;

  // Set-up, run by every thread of the CTA, with the kBarBytes of barriers at `bars`.  Thread 0 initialises them -- an accumulator
  // is handed back by the `epi_warps` epilogue warps of each CTA of the MMA -- and runs init() (tensor-map prefetches, barriers of
  // the kernel's own); warp 1 allocates the tensor memory.  Ends with PDL_PROLOGUE: everything before it is private to the CTA (or
  // pair), operands of the previous kernel are touched only after it.
  template <typename Init>
  static __device__ __forceinline__ TcPipeline setup(uint8_t* bars, uint32_t epi_warps, Init&& init) {
    TcPipeline p;
    p.full = reinterpret_cast<uint64_t*>(bars);
    p.empty = p.full + STAGES;
    p.acc_full = p.empty + STAGES;
    p.acc_empty = p.acc_full + NACC;
    p.ready = p.full;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p.acc_empty + NACC);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(&p.full[s], 1);
        mbar_init(&p.empty[s], CG == 2 ? 1 : CL);  // one tcgen05.commit arrival from every CTA whose MMAs read the stage
      }
#pragma unroll
      for (int b = 0; b < NACC; ++b) {
        mbar_init(&p.acc_full[b], 1);
        mbar_init(&p.acc_empty[b], CG * epi_warps);
      }
      init();
      fence_barrier_init();
      fence_proxy_async();
    }
    if (threadIdx.x / 32 == 1) {
      if (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
      } else {  // the same warp of both CTAs allocates
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
      }
    }
    tc_fence_before();
    if (CL > 1) cluster_sync_all(); else __syncthreads();  // peers must see initialised barriers before any multicast or arrival lands
    tc_fence_after();
    p.tmem_base = *tmem_slot;
    if (CG == 2) p.acc_empty_leader = mapa_u32(smem_u32(p.acc_empty), 0);
    PDL_PROLOGUE();
    return p;
  }

  // TMA producer (one thread): unit(u) prepares unit u and returns its number of k-blocks (returned as a reference into the kernel
  // parameters, it is read again at every k-block, and the loop is not unrolled); load(kb, s) issues the loads of k-block kb into
  // stage s, whose previous contents every MMA has read, and posts the bytes they bring on full[s].
  template <typename Unit, typename Load>
  __device__ __forceinline__ void produce(int u_lo, int u_hi, int u_step, Unit&& unit, Load&& load) const {
    int s = 0;
    uint32_t ph = 0;
    for (int u = u_lo; u < u_hi; u += u_step) {
      decltype(auto) num_kb = unit(u);
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty[s], ph ^ 1);
        load(kb, s);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  }

  // MMA issuer (one thread): unit(u) returns unit u's number of k-blocks (as for produce); mma(d, kb, s) issues the MMAs of
  // k-block kb from stage s into the accumulator at TMEM address d.  A stage is released once its MMAs have completed (in every
  // CTA that reads it: the commit multicasts), the accumulator once the unit's last MMA has.
  template <typename Unit, typename Mma>
  __device__ __forceinline__ void issue(int u_lo, int u_hi, int u_step, Unit&& unit, Mma&& mma) const {
    int s = 0;
    uint32_t ph = 0, it = 0;
    for (int u = u_lo; u < u_hi; u += u_step, ++it) {
      const uint32_t a = it % NACC;
      mbar_wait(&acc_empty[a], ((it / NACC) & 1u) ^ 1u);  // the epilogue has drained this accumulator (first use passes at once)
      tc_fence_after();
      const uint32_t d = tmem_base + a * ACC_COLS;
      decltype(auto) num_kb = unit(u);
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&ready[s], ph);
        tc_fence_after();
        mma(d, kb, s);
        if (CG == 2) umma_commit_2sm(&empty[s]);
        else if (CL > 1) umma_commit_mc(&empty[s], static_cast<uint16_t>((1u << CL) - 1u));
        else umma_commit(&empty[s]);
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
      if (CG == 2) umma_commit_2sm(&acc_full[a]); else umma_commit(&acc_full[a]);
    }
  }

  // Epilogue: waits until the accumulator of this CTA's it-th unit is complete and returns its index.
  __device__ __forceinline__ uint32_t acc_wait(uint32_t it) const {
    const uint32_t a = it % NACC;
    mbar_wait(&acc_full[a], (it / NACC) & 1u);
    tc_fence_after();
    return a;
  }
  // Epilogue: hands accumulator a back to the MMA issuer (on the leader's barrier with a CTA pair) once every TMEM read of this warp
  // has completed (tcgen05.wait::ld).
  __device__ __forceinline__ void acc_release(uint32_t a) const {
    tc_fence_before();
    if (threadIdx.x % 32 == 0) {
      if (CG == 2) mbar_arrive_remote(acc_empty_leader + 8u * a); else mbar_arrive(&acc_empty[a]);
    }
  }

  // Run by every thread: no CTA may exit while a peer can still multicast into / arrive on it.
  __device__ __forceinline__ void teardown() const {
    tc_fence_before();
    if (CL > 1) cluster_sync_all(); else __syncthreads();
    if (threadIdx.x / 32 == 1) {
      tc_fence_after();
      if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
      else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
  }
};

// Problem of unit u in a grouped launch: P holds P.n <= kMaxGroup problems P.p[g], in the order of their first units P.p[g].unit0.
template <typename Params>
__device__ __forceinline__ int problem_of(const Params& P, int u) {
  int g = 0;
#pragma unroll
  for (int i = 1; i < kMaxGroup; ++i)
    if (i < P.n && u >= P.p[i].unit0) g = i;
  return g;
}

// host: K-major bf16 / fp32 operand maps (box = one 128-byte row of k -- 64 bf16 / 32 fp32 -- x box_rows rows, SWIZZLE_128B) and
// output map (box = 32 rows x 64 bytes, SWIZZLE_64B)
int make_tmap(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);
int make_tmap_f32(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);
int make_tmap_out(CUtensorMap* map, void* ptr, uint64_t rows, uint64_t cols, bool f32);

// host: one launch of a CTA-pair kernel over the problems of P.  Their units are numbered in problem order (P.p[g].unit0, P.n_units;
// units(P.p[g]) each) and min(units, SMs / 2) pairs walk them; schedule(pairs) sets what depends on the number of pairs.
// `smem_limit` belongs to the kernel instance (raise_smem_limit).
template <typename Params, typename Units, typename Schedule>
int launch_pair(void (*kernel)(Params), PerDevice<size_t>& smem_limit, int smem, int threads, Params& P, Units&& units,
                Schedule&& schedule, cudaStream_t st) {
  M3PC_CHECK_CUDA(raise_smem_limit(kernel, smem_limit, smem));
  int n_units = 0;
  for (int g = 0; g < P.n; ++g) {
    P.p[g].unit0 = n_units;
    n_units += units(P.p[g]);
  }
  P.n_units = n_units;
  const int pairs = std::min(n_units, device_num_sms() / 2);
  schedule(pairs);
  M3PC_CHECK_CUDA(launch_k_cluster(2, kernel, dim3(2 * pairs), dim3(threads), smem, st, P));
  M3PC_CHECK_LAUNCH();
  return M3PC_OK;
}

}  // namespace m3pc
