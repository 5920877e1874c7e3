// Shared helpers for libtvbf: error plumbing and the sm_100a PTX wrappers (mbarrier, TMA,
// tcgen05 / TMEM).  Everything here is hand-written inline PTX; no CUTLASS/CuTe dependency.
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../include/tvbf.h"

// ---------------------------------------------------------------------------------------------
// error plumbing (no exceptions cross the C ABI)
// ---------------------------------------------------------------------------------------------
void tvbf_set_error(const char* fmt, ...);
void tvbf_count_launch(void);  // every kernel launch of the library is counted (tvbf_kernel_launches)
void tvbf_count_coop_fallback(void);  // K1 launches that fell back from cooperative to plain
// Every ABI call that enqueues device work enters here first (TVBF_ENTER_CALL): it is numbered per
// device and orders `stream` after a pending shared-list clear of the symmetric sweep (hybrid_topk.cu)
// -- except a sweep-only call (sym_sweep = 1), which may be the one that clear was started for.
int tvbf_enter_call(void* stream, int sym_sweep);
// `stream` waits for every shared-list clear started on this device; the pending one is forgotten
// (error returns of the seed / sweep calls, and a sweep call that launches no candidate pass)
int tvbf_absorb_pending_clear(void* stream);

#define TVBF_CUDA_OK(expr)                                                              \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      tvbf_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,  \
                     __LINE__);                                                         \
      return TVBF_ERR_CUDA;                                                             \
    }                                                                                   \
  } while (0)

#define TVBF_REQUIRE(cond, ...)                                                         \
  do {                                                                                  \
    if (!(cond)) {                                                                      \
      tvbf_set_error(__VA_ARGS__);                                                      \
      return TVBF_ERR_INVALID;                                                          \
    }                                                                                   \
  } while (0)

#define TVBF_ENTER_CALL(stream)                                                         \
  do {                                                                                  \
    int _rc = tvbf_enter_call((stream), 0);                                             \
    if (_rc != TVBF_OK) return _rc;                                                     \
  } while (0)

#define TVBF_LAUNCH_OK(name)                                                            \
  do {                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) {                                                            \
      tvbf_set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));          \
      return TVBF_ERR_CUDA;                                                             \
    }                                                                                   \
    tvbf_count_launch();                                                                \
  } while (0)

// Column-side record the epilogue reads once per score (16 bytes -> one LDS.128).
struct __align__(16) TvbfColSide {
  unsigned long long genre_bits;  // multi-hot genre bitmask (G <= 64)
  float genre_rnorm;              // 1/sqrt(popcount), 0 for an all-zero row
  uint32_t meta_bits;             // one-hot bits: platform | type << P | language << (P+T); P+T+L <= 32
};
static_assert(sizeof(TvbfColSide) == 16, "column-side record must be 16 bytes");

#ifdef __CUDACC__
namespace tvbf {

constexpr uint32_t kFullMask = 0xffffffffu;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier --------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
// try_wait may suspend the thread until the phase completes or a time limit passes (system
// default, or TVBF_MBAR_HINT_NS nanoseconds when that is set at compile time).
#ifndef TVBF_MBAR_HINT_NS
#define TVBF_MBAR_HINT_NS 0
#endif
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
#if TVBF_MBAR_HINT_NS > 0
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(static_cast<uint32_t>(TVBF_MBAR_HINT_NS))
      : "memory");
#else
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
#endif
  return ok != 0;
}
// Bounded wait: a protocol bug must trap (-> launch error on the host), never hang the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 23)) {
      printf("tvbf: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x,
             (int)threadIdx.x);
      __trap();
    }
  }
}

// Same, for waits that can last a whole tile (the roles that run AHEAD of the bottleneck: in the
// epilogue-bound regime the producer and the MMA issuer, in the MMA-bound regime the epilogue).  A
// tight try_wait loop issues an instruction every ~12 cycles and, sharing a scheduler with working
// warps, takes issue slots from them (ncu on P80k: half of all executed warp instructions were
// these polls).  After `quick` failed polls the thread sleeps between polls, twice as long each time
// up to 8 * sleep_ns.
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, uint32_t quick = 16,
                                                  uint32_t sleep_ns = 64) {
  uint32_t spins = 0, ns = sleep_ns;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > quick) {
      __nanosleep(ns);
      if (ns < 8 * sleep_ns) ns *= 2;
    }
    if (spins > (1u << 21)) {
      printf("tvbf: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x,
             (int)threadIdx.x);
      __trap();
    }
  }
}

// One lane of a fully converged warp (warp-uniform control flow keeps addresses and descriptors
// in uniform registers; a divergent `if (lane == 0)` region makes the compiler wrap every TMA /
// tcgen05 instruction in an elect-and-loop sequence that costs more than the MMA it issues).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- TMA -------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tiled load: coordinates are (inner = K element, outer = row).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar,
                                            int32_t c_inner, int32_t c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer)
      : "memory");
}
// L2 prefetch of one TMA box (no shared memory involved)
__device__ __forceinline__ void tma_prefetch_2d(const void* tmap, int32_t c_inner, int32_t c_outer) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(c_inner), "r"(c_outer)
               : "memory");
}
// 1-D bulk copy global -> shared (16-byte aligned, size multiple of 16).
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- tcgen05 / TMEM ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_holder)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, kind::f16 (fp16 or bf16 operands, fp32 accumulate).
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all previously issued MMAs of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
          smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives lane (row) t.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// 32 lanes x 16 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// ---- cta_group::2 (CTA pair) variants ---------------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // clears the CTA-rank bit of a shared::cluster address

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same smem offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 remAddr32;\n\t"
      "mapa.shared::cluster.u32 remAddr32, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [remAddr32];\n\t}" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
// TMA load issued by either CTA of a pair; the transaction bytes land on the LEADER's barrier
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap, uint64_t* bar,
                                                 int32_t c_inner, int32_t c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c_inner),
      "r"(c_outer)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_holder)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// issued by the leader CTA only: M = 256 spans both CTAs' TMEM, B is split along N across the pair
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this offset in BOTH CTAs once the pair's MMAs have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64"
      " [%0], %1;" ::"r"(smem_u32(bar)),
      "h"(static_cast<uint16_t>(3))
      : "memory");
}

// K-major, 128-byte-swizzled shared-memory operand descriptor (tile rows are 128 B = 64 halves;
// 8-row groups are 1024 B apart).  Bits: [0,14) addr>>4, [16,30) LBO>>4 (unused for swizzled
// K-major), [32,46) SBO>>4, [46,48) version=1 (sm_100), [61,64) layout 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1024u >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// kind::f16 instruction descriptor: fp32 accumulate, A/B both K-major, M x N tile.
// fmt: 0 = fp16, 1 = bf16.
__host__ __device__ constexpr uint32_t umma_idesc_f16(uint32_t fmt, uint32_t m, uint32_t n) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// order-preserving map float bits -> uint32 (bigger float <=> bigger uint)
__device__ __forceinline__ uint32_t f32_orderable(float f) {
  uint32_t b = __float_as_uint(f);
  return b ^ ((b >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float f32_from_orderable(uint32_t u) {
  uint32_t b = u ^ ((u >> 31) ? 0x80000000u : 0xFFFFFFFFu);
  return __uint_as_float(b);
}

// The reference's hybrid expression `gw * g + tw * t + mw * m` (scripts/populate_database.py:190-192;
// ml/similarity_computer.py:122-124) exactly as numpy evaluates it: three rounded products, two
// rounded sums, left to right, no FMA contraction.  Every fp64 scorer goes through this one
// function, so a score computed by K5, K6, the pair scorer and the N x N combine agree bit for bit.
__device__ __forceinline__ double hybrid_rn(double wg, double g, double wt, double t, double wm, double m) {
  return __dadd_rn(__dadd_rn(__dmul_rn(wg, g), __dmul_rn(wt, t)), __dmul_rn(wm, m));
}

}  // namespace tvbf
#endif  // __CUDACC__
