// K1 + K4 -- the hot kernel: TMA-fed tcgen05 text GEMM (X * X^T, fp16/bf16 operands, fp32
// accumulators in TMEM) whose epilogue adds the popcount genre score and the category-id
// metadata score with the reference's weights and keeps a running per-row candidate list, so
// the N x N matrix is never written anywhere.
//
// Replaces, for all source rows at once, the body of the reference's hot loop
// (scripts/populate_database.py:170-195): five cosine_similarity calls, the (p+t+l)/3 metadata
// mean, the weighted sum and the full argsort.  The selection made here is a conservative
// CANDIDATE selection on an upper bound U >= exact score; rescore.cu recomputes the candidates in
// fp64 and certifies (or repairs) each row, so the final table does not depend on fp16 rounding.
//
// Kernel anatomy (one CTA per SM, persistent over work items = (row block of 128, column split)):
//   warp 0   lane 0 : TMA producer  -- A (128 x 64) and B (256 x 64) operand tiles, 4-stage ring,
//                                      plus the column-side records of each 256-column tile
//   warp 1   lane 0 : MMA issuer    -- tcgen05.mma cta_group::1 kind::f16, M=128 N=256 K=16,
//                                      double-buffered 128x256 fp32 accumulators (2 x 256 TMEM cols)
//   warps 2-5       : epilogue      -- tcgen05.ld 32x32b: thread t owns accumulator row t; scores,
//                                      thresholds and appends to its row's candidate list
#include "internal.cuh"

#include <cuda.h>  // CUtensorMap types only; the encoder is fetched through the runtime
#include <cstdlib>
#include <mutex>

namespace tvbf {

constexpr int BM = 128;     // rows per CTA tile (= TMEM lanes)
constexpr int BN = 256;     // columns per tile (= TMEM columns per accumulator)
constexpr int BK = 64;      // K elements per stage: 64 halves = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr uint32_t A_BYTES = BM * BK * 2;
constexpr uint32_t COL_BYTES = BN * sizeof(TvbfColSide);
constexpr uint32_t MS_BYTES = BN * sizeof(float);
constexpr int RING = 128;   // pending list appends an epilogue warp can hold between two flushes
// warps 0..EPI-1: epilogue (warp w may touch TMEM lanes 32*(w%4)..+31); then the TMA producer and
// the MMA issuer.  The SM's issue arbiter favours higher warp ids, so the two single-lane roles,
// which share schedulers with epilogue warps, are never starved by the epilogue's ALU stream.
// One-sided sweep: 4 epilogue warps (thread t owns accumulator row t and its private list).
// Symmetric sweep: 8 epilogue warps, two per lane quarter, each scoring half of the tile's columns
// -- its epilogue does twice the compares plus the shared-list traffic and, with one warp per
// scheduler, was latency-bound (tensor pipe 74 % active); two warps per scheduler hide it.
// Small vocabularies (K_pad of a few hundred): the MMAs of a tile take ~2 us while its epilogue --
// 65 536 scores through popcounts, FMAs, two compares and the shared-list traffic -- takes ~30 us
// and is LATENCY-bound with 8 warps (ncu: 15 % of the warp slots active, 80 % of the issue slots
// empty).  kWide doubles the epilogue to 16 warps (four per lane quarter, 64 columns each); the
// registers then cap at 112 per thread and one ring stage is given up for the append queues.
template <bool kSym, bool kWide = false> struct Roles {
  static constexpr int EPI = kSym ? (kWide ? 16 : 8) : 4;
  static constexpr int PRODUCER = EPI;
  static constexpr int MMA = EPI + 1;
  static constexpr int THREADS = 32 * (EPI + 2);
};

// Shared-memory plan.  CG = CTAs cooperating on one MMA (tcgen05 cta_group): with CG = 2 the pair
// computes a 256 x 256 tile, each CTA stages its own 128 rows of A and HALF of the B tile, so the
// L2 -> SM operand traffic per MAC drops by a third and the ring gets two more stages.
template <int CG, bool kWide = false>
struct Smem {
  static constexpr int STAGES = CG == 2 ? (kWide ? 5 : 6) : 4;
  static constexpr int QTHREADS = kWide ? 512 : 256;   // epilogue threads of the symmetric sweep
  static constexpr uint32_t B_ROWS = BN / CG;
  static constexpr uint32_t B_BYTES = B_ROWS * BK * 2;
  static constexpr uint32_t OFF_A = 0;
  static constexpr uint32_t OFF_B = OFF_A + STAGES * A_BYTES;
  static constexpr uint32_t OFF_COL = OFF_B + STAGES * B_BYTES;
  static constexpr uint32_t OFF_MS = OFF_COL + 2 * COL_BYTES;
  static constexpr uint32_t OFF_TH = OFF_MS + 2 * MS_BYTES;   // symmetric mode: column thresholds
  // symmetric mode: one ring of pending list appends per epilogue warp, SoA [3][RING] words
  static constexpr uint32_t OFF_Q = OFF_TH + 2 * kMaxSweep * MS_BYTES;   // (one slice per triple of a weight sweep)
  static constexpr uint32_t OFF_BAR = OFF_Q + 3 * RING * (QTHREADS / 32) * 4;
  static constexpr int NUM_BARS = 2 * STAGES + 8;
  static constexpr uint32_t OFF_TMEM = OFF_BAR + NUM_BARS * 8;
  static constexpr uint32_t USED = OFF_TMEM + 16;
  static constexpr uint32_t BYTES = USED + 1024;  // slack for manual 1024-byte alignment
};

// ---- warp-cooperative bitonic sort (descending) of 32*E 64-bit keys, E per lane ----------------
// element index = q * 32 + lane
template <int E>
__device__ __forceinline__ void bitonic_sort_desc(unsigned long long (&key)[E], int lane) {
  constexpr int NTOT = 32 * E;
#pragma unroll
  for (int k = 2; k <= NTOT; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        const int dq = j >> 5;
#pragma unroll
        for (int q = 0; q < E; ++q) {
          const int q2 = q ^ dq;
          if (q2 > q) {
            const bool desc = (((q * 32) & k) == 0);  // lane bits are below k's bit here
            unsigned long long a = key[q], b = key[q2];
            const bool sw = desc ? (a < b) : (a > b);
            key[q] = sw ? b : a;
            key[q2] = sw ? a : b;
          }
        }
      } else {
#pragma unroll
        for (int q = 0; q < E; ++q) {
          const unsigned long long other = __shfl_xor_sync(kFullMask, key[q], j);
          const int idx = q * 32 + lane;
          const bool lower = (lane & j) == 0;
          const bool desc = ((idx & k) == 0);
          const unsigned long long mx = key[q] > other ? key[q] : other;
          const unsigned long long mn = key[q] > other ? other : key[q];
          key[q] = (lower == desc) ? mx : mn;
        }
      }
    }
  }
}

// Sort the `n` entries of one row's list and write the best min(n, kp) to dst (may alias src).
// Returns (to every lane) the score of entry kp-1, i.e. the bound on everything dropped.
// Deliberately NOT inlined: it runs a few times per row per sweep, while the scoring loop around
// it runs for every accumulator element and must stay small enough for the instruction cache.
template <int E>
__device__ __noinline__ float warp_compact(const uint2* src, int n, uint2* dst, int kp,
                                           int lane) {
  unsigned long long key[E];
  __syncwarp();  // the owner lane's appends (st.cg) are ordered before these loads
#pragma unroll
  for (int q = 0; q < E; ++q) {
    const int idx = q * 32 + lane;
    key[q] = 0ull;
    if (idx < n) {
      const uint2 e = __ldcg(src + idx);
      key[q] = (static_cast<unsigned long long>(f32_orderable(__uint_as_float(e.x))) << 32) |
               static_cast<unsigned long long>(0xFFFFFFFFu - e.y);
    }
  }
  __syncwarp();  // all loads done before anyone overwrites (dst may alias src)
  bitonic_sort_desc<E>(key, lane);
  const int keep = n < kp ? n : kp;
  float bound = 0.0f;
#pragma unroll
  for (int q = 0; q < E; ++q) {
    const int idx = q * 32 + lane;
    const float sc = f32_from_orderable(static_cast<uint32_t>(key[q] >> 32));
    if (idx < keep)
      __stcg(dst + idx, make_uint2(__float_as_uint(sc), 0xFFFFFFFFu - static_cast<uint32_t>(key[q])));
    // entry kp-1 lives in register (kp-1)/32 of lane (kp-1)%32
    const float cand = __shfl_sync(kFullMask, sc, (kp - 1) & 31);
    if (q == ((kp - 1) >> 5)) bound = cand;
  }
  __syncwarp();
  return bound;
}

// Keep the kp best of the n entries of one row's list IN PLACE and UNORDERED (the order only matters
// for the final hand-over, which sorts): exact radix select of the kp-th largest score over the bits
// the entries do not share, then a ballot compaction -- about a quarter of the bitonic sort's
// instructions.  The one-sided sweep compacts a row every ~96 appends; in the threshold seed pass,
// which starts from min_similarity, that was four fifths of its time.
// Returns (to every lane) the kp-th largest score: the bound on everything dropped.
template <int E>
__device__ __noinline__ float warp_select_compact(uint2* list, int n, int kp, int lane) {
  if (n <= kp) return __int_as_float(0xff800000);   // nothing to drop
  uint32_t v[E], col[E];
  uint32_t lo = 0xFFFFFFFFu, hi = 0u;
  __syncwarp();  // the owner lane's appends (st.cg) are ordered before these loads
#pragma unroll
  for (int q = 0; q < E; ++q) {
    const int idx = q * 32 + lane;
    v[q] = 0u;
    col[q] = 0u;
    if (idx < n) {
      const uint2 e = __ldcg(list + idx);
      v[q] = f32_orderable(__uint_as_float(e.x));
      col[q] = e.y;
      lo = min(lo, v[q]);
      hi = max(hi, v[q]);
    }
  }
  lo = __reduce_min_sync(kFullMask, lo);
  hi = __reduce_max_sync(kFullMask, hi);
  const int top = 31 - __clz(lo ^ hi);   // highest bit in which two entries differ (-1: all equal)
  uint32_t best = top >= 0 ? ((top == 31 ? 0u : (hi >> (top + 1)) << (top + 1))) : hi;
#pragma unroll 1
  for (int bit = top; bit >= 0; --bit) {
    const uint32_t t = best | (1u << bit);
    int c = 0;
#pragma unroll
    for (int q = 0; q < E; ++q) c += (q * 32 + lane < n && v[q] >= t);
    c = __reduce_add_sync(kFullMask, c);
    if (c >= kp) best = t;
  }
  __syncwarp();  // all loads done before anyone overwrites
  int out = 0;
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
    for (int q = 0; q < E; ++q) {
      const bool take = q * 32 + lane < n && (pass == 0 ? v[q] > best : v[q] == best);
      const unsigned bal = __ballot_sync(kFullMask, take);
      const int pos = out + __popc(bal & ((1u << lane) - 1u));
      if (take && pos < kp)
        __stcg(list + pos, make_uint2(__float_as_uint(f32_from_orderable(v[q])), col[q]));
      out += __popc(bal);
    }
  }
  __syncwarp();
  return f32_from_orderable(best);
}

struct ItemCoord {
  int sb;            // super block (128*CG rows) within the shard, -1 = nothing to do
  int split;
  int tile0, tile1;  // tiles this item walks (pacing); every item of a group walks equally many
  int real0, real1;  // ... of which [real0, real1) are computed, the rest are phantom
};

// local super block number of this launch -> global super block (see K1Params::deal_*)
__host__ __device__ __forceinline__ int global_super_block(const K1Params& p, int local) {
  if (p.seed_theta && p.seed_world > 1) return local * p.seed_world + p.seed_rank;
  if (p.deal_groups == 0) return local;
  const int g = local / p.deal_r;
  if (g >= p.deal_groups) return 0x3fffffff;
  return static_cast<int>(p.deal_gid[g]) * p.deal_r + (local - g * p.deal_r);
}

// kAppend (append sweep): every super block only needs the column tiles >= append_b0, the first one
// holding new shows
template <bool kAppend = false>
__host__ __device__ __forceinline__ ItemCoord item_coord(const K1Params& p, int item) {
  const int per_group = p.rb_per_group * p.splits;
  const int g = item / per_group;
  const int w = item - g * per_group;
  ItemCoord c;
  c.split = w / p.rb_per_group;
  const int local = g * p.rb_per_group + (w - c.split * p.rb_per_group);
  c.sb = global_super_block(p, local);
  if (p.sym) {
    // the group's super blocks lie at or right of tile i0 on the diagonal; only columns >= i0 matter
    // (with several GPUs a wave is one dealt group: rb_per_group == deal_r)
    int i0 = global_super_block(p, g * p.rb_per_group);
    if constexpr (kAppend) i0 = i0 > p.append_b0 ? i0 : p.append_b0;
    const int span = p.col_tiles > i0 ? p.col_tiles - i0 : 0;
    const int tps = (span + p.splits - 1) / p.splits;
    c.tile0 = i0 + c.split * tps;
    c.tile1 = c.tile0 + tps;
  } else {
    c.tile0 = c.split * p.tiles_per_split;
    c.tile1 = c.tile0 + p.tiles_per_split;
  }
  c.real0 = c.tile0;
  c.real1 = c.tile1 < p.col_tiles ? c.tile1 : p.col_tiles;
  if (p.sym && c.sb > c.real0) c.real0 = c.sb;  // tiles left of the diagonal are the mirror's job
  if (local >= p.rb_count) { c.sb = -1; c.real0 = c.real1 = c.tile1; }
  if (c.real0 > c.real1) c.real0 = c.real1;
  return c;
}

// ---- symmetric mode helpers ---------------------------------------------------------------------
// Raise the shared threshold of one show to (a lower bound of) the kp-th largest score of the first
// n entries of its list.  Entries reserved but not yet written read as 0 = -inf, so the result can
// only be too LOW, never too high.  Warp-cooperative, Q entries per lane (32 * Q >= n).
// The radix select starts below the bits all written entries share (scores of one list lie within a
// factor of two of each other, so sign, exponent and the leading mantissa bits are skipped) and stops
// at bit 8: the threshold is rounded DOWN to 23 significant bits of the ordering, 2^-15 relative --
// still a valid bound, and a refresh costs a third of the full 31-bit select.
template <int Q>
__device__ __forceinline__ void refresh_theta_q(const uint2* list, int n, int kp, unsigned int* theta_slot,
                                                int lane) {
  uint32_t v[Q];
  uint32_t lo = 0xFFFFFFFFu, hi = 0u;
  int written = 0;
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const int idx = q * 32 + lane;
    v[q] = idx < n ? __ldcg(list + idx).x : 0u;
    if (v[q] != 0u) { lo = min(lo, v[q]); ++written; }
    hi = max(hi, v[q]);
  }
  lo = __reduce_min_sync(kFullMask, lo);
  hi = __reduce_max_sync(kFullMask, hi);
  written = __reduce_add_sync(kFullMask, written);
  if (written < kp) return;                       // warp-uniform
  const int top = 31 - __clz(lo ^ hi);            // highest bit in which two written entries differ (-1: none)
  uint32_t best = top >= 0 ? (hi >> (top + 1)) << (top + 1) : hi;   // the shared prefix: count(v >= best) = written >= kp
#pragma unroll 1
  for (int bit = top; bit >= 8; --bit) {
    const uint32_t t = best | (1u << bit);
    int c = 0;
#pragma unroll
    for (int q = 0; q < Q; ++q) c += (v[q] >= t);
    c = __reduce_add_sync(kFullMask, c);
    if (c >= kp) best = t;
  }
  if (lane == 0) atomicMax(theta_slot, best);
}

// Deliberately not inlined: it runs a few times per show per sweep.
__device__ __noinline__ void sym_refresh_theta(const uint2* list, int n, int kp,
                                               unsigned int* theta_slot, int lane) {
  // lists longer than 1024 (kp > 64): the most recent 1024 entries -- the kp-th largest of ANY
  // subset is a valid lower bound, and the latest entries passed the highest thresholds
  if (n > 1024) { list += n - 1024; n = 1024; }
  if (n <= 64) refresh_theta_q<2>(list, n, kp, theta_slot, lane);
  else if (n <= 128) refresh_theta_q<4>(list, n, kp, theta_slot, lane);
  else if (n <= 256) refresh_theta_q<8>(list, n, kp, theta_slot, lane);
  else if (n <= 512) refresh_theta_q<16>(list, n, kp, theta_slot, lane);
  else refresh_theta_q<32>(list, n, kp, theta_slot, lane);
}

// Drain one epilogue warp's ring of pending appends {show, score bits, other show} into the shared
// lists.  An append needs the slot returned by an atomicAdd (a ~700-cycle round trip): all atomics of
// the ring are issued back to back, one entry per lane and pass, so the warp pays the round trip once
// per flush.  A list gets its threshold refreshed when it reaches 2*kp entries and then every P further
// ones (P = largest power of two <= kp).  Round 1 refreshed at 2*kp, 4*kp, 8*kp, ...: the threshold
// then lags by up to a factor of two in rank and a show collected ~530 entries per sweep on P80k
// (80 k shows); refreshing every P appends tracks the running kp-th best and needs ~200.
// Not inlined: the scoring loop around it must stay small enough for the instruction cache.
__device__ __noinline__ void sym_ring_flush(const uint32_t* ring, int n, unsigned int* g_cnt, uint2* g_list,
                                            unsigned int* g_theta, unsigned sym_cap, int kp, int period, int lane) {
  constexpr int J = RING / 32;
  uint32_t sh[J];
  unsigned pos[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int i = j * 32 + lane;
    sh[j] = 0u;
    pos[j] = 0xFFFFFFFFu;
    if (i < n) {
      sh[j] = ring[i];
      pos[j] = atomicAdd(g_cnt + sh[j], 1u);
    }
  }
  unsigned trig = 0u;   // bit j: entry j of this lane completed a list length that asks for a refresh
  const unsigned first = static_cast<unsigned>(2 * kp);
  const unsigned period_mask = static_cast<unsigned>(period) - 1u;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int i = j * 32 + lane;
    if (pos[j] < sym_cap) {   // lanes without an entry hold 0xFFFFFFFF; an overflowing list drops the entry
      __stcg(g_list + static_cast<size_t>(sh[j]) * sym_cap + pos[j], make_uint2(ring[RING + i], ring[2 * RING + i]));
      const unsigned np = pos[j] + 1u;
      if (np >= first && (np & (period ? period_mask : pos[j])) == 0u) trig |= 1u << j;
    }
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < J; ++j) {
    if (j * 32 >= n) break;   // warp-uniform
    unsigned need = __ballot_sync(kFullMask, ((trig >> j) & 1u) != 0u);
    while (need) {
      const int src_lane = __ffs(need) - 1;
      need &= need - 1;
      const uint32_t show = __shfl_sync(kFullMask, sh[j], src_lane);
      const int len = static_cast<int>(__shfl_sync(kFullMask, pos[j], src_lane)) + 1;
      sym_refresh_theta(g_list + static_cast<size_t>(show) * sym_cap, len, kp, g_theta + show, lane);
    }
  }
}

// Drain one epilogue warp's ring of pending pairs {row show, column show} into the global pair buffer
// of the neighbour sweep: one 64-bit atomicAdd reserves the slots of the whole ring.  Slots at or past
// cap are counted but not stored.  Not inlined, as sym_ring_flush.
__device__ __noinline__ void pair_ring_flush(const uint32_t* ring, int n, unsigned long long* count, int2* pairs,
                                             long long cap, int lane) {
  unsigned long long base = 0ull;
  if (lane == 0) base = atomicAdd(count, static_cast<unsigned long long>(n));
  base = __shfl_sync(kFullMask, base, 0);
  for (int i = lane; i < n; i += 32) {
    const unsigned long long slot = base + static_cast<unsigned long long>(i);
    if (slot < static_cast<unsigned long long>(cap))
      __stcg(pairs + slot, make_int2(static_cast<int>(ring[i]), static_cast<int>(ring[RING + i])));
  }
}

// u[e] for a run-time e without spilling the array to local memory: a select tree
template <int GW>
__device__ __forceinline__ float pick(const float (&u)[GW], int e) {
  static_assert(GW == 4 || GW == 8, "group width");
  float a[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) a[i] = (GW == 8 && (e & 4) != 0) ? u[(i + 4) % GW] : u[i];
  const bool s2 = (e & 2) != 0, s1 = (e & 1) != 0;
  const float c0 = s2 ? a[2] : a[0], c1 = s2 ? a[3] : a[1];
  return s1 ? c1 : c0;
}

// Grid-wide pacing of the TMA producers.  Operand tiles are shared between CTAs only through L2
// (all CTAs of a column split stream the same B tiles, all CTAs of a row block the same A rows),
// which works only while they request the same bytes within the L2 retention window; without
// pacing the CTAs drift apart (data-dependent epilogues) and every CTA pulls its operands from
// HBM.  Rule: nobody issues chunk c before everybody has issued chunk c - slack.
struct Pacer {
  unsigned int* counter;
  unsigned int n_ctas;
  int slack;
  unsigned int chunk;  // chunks this CTA has issued
  __device__ __forceinline__ void wait_turn() {
    if (counter == nullptr || static_cast<int>(chunk) < slack) return;
    const unsigned int target = n_ctas * (chunk - static_cast<unsigned int>(slack) + 1u);
    unsigned int spins = 0;
    while (true) {
      unsigned int v;
      asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (v >= target) break;
      __nanosleep(64);
      if (++spins > (1u << 24)) {
        printf("tvbf: pacing wait timed out (block %d chunk %u have %u want %u)\n", (int)blockIdx.x,
               chunk, v, target);
        __trap();
      }
    }
  }
  __device__ __forceinline__ void done_chunk(bool do_add) {
    if (counter != nullptr && do_add) atomicAdd(counter, 1u);
    ++chunk;
  }
};

// kMode: 0 one-sided top-k sweep, 1 symmetric top-k sweep, 2 symmetric statistics sweep,
// 3 threshold seed pass (one-sided walk over sampled tiles, per-row score histograms, no lists),
// 5 symmetric top-k sweep for p.n_weights weight triples at once (one shared list per triple and show),
// 6 append sweep: the symmetric top-k sweep restricted to the tiles that hold a new show (column tile
// >= p.append_b0), offering no pair of two old shows (p.append_n_old),
// 7 update sweep: the gathered rows of the updated shows (p.upd_rows) against every column tile, a
// rectangle without a diagonal; offered to the row's show and to every column show not updated itself,
// 8 the threshold seed pass (as 3) over the gathered rows of an update,
// 9 repair sweep of a removal: the update sweep without the column side -- every score goes to the
// gathered row's list only, and that list, its count and its threshold are indexed by the gathered row,
// 10 refresh sweep: the update sweep over the gathered rows of the shows in G = S + A (p.upd_bits), where
// only a row whose show is in S (p.upd_sbits: updated or appended) feeds the column side,
// 11 neighbour sweep: the tiles of the symmetric top-k sweep, no lists and no thresholds -- every pair
// i < j whose upper bound U exceeds theta_init (an fp32 below min_similarity) is appended to
// p.pairs (pair_ring_flush)
// kG2: multi-hot genres with 64 < G <= 128 -- the second word of every column's mask is staged beside
// the column-side records (in the threshold slices a single-triple sweep leaves unused) and the
// popcount runs over both words.
// kFold: the operand carries the packed genre / metadata groups as extra K columns scaled by
// sqrt(w_group / w_text) (tvbf_prep_fold_bits), so the accumulator already is the whole hybrid: the
// epilogue is one FMA and two compares per element instead of three popcounts, two conversions and
// six FMAs.  For small vocabularies, where a tile's MMAs (even with one more k-block) are far shorter
// than its epilogue.
template <int E, bool kDump, int CG, int kMode, bool kWide = false, bool kG2 = false, bool kFold = false>
__global__ void __launch_bounds__(Roles<(kMode != 0), kWide>::THREADS, 1)
hybrid_topk_kernel(const __grid_constant__ CUtensorMap tmap_a,
                   const __grid_constant__ CUtensorMap tmap_b, const K1Params p,
                   const uint32_t idesc) {
  using L = Smem<CG, kWide>;
  constexpr bool kHist = kMode == 3 || kMode == 8;   // threshold seed pass: per-row histograms of the sampled scores
  constexpr bool kSym = kMode != 0 && !kHist;   // tiles on/above the diagonal, 8 (kWide: 16) epilogue warps
  constexpr bool kStats = kMode == 2;    // accumulate statistics instead of candidate lists
  constexpr bool kMulti = kMode == 5;    // weight sweep
  constexpr bool kAppend = kMode == 6;   // append sweep
  constexpr bool kRefresh = kMode == 10;   // refresh sweep
  constexpr bool kUpdate = kMode == 7 || kRefresh;   // update sweep (or its refresh variant)
  constexpr bool kRepair = kMode == 9;   // repair sweep of a removal
  constexpr bool kGather = kMode == 7 || kMode == 8 || kRepair || kRefresh;   // rows are gathered rows
  constexpr bool kPairs = kMode == 11;   // neighbour sweep: pairs above the threshold, no lists
  static_assert(!(kG2 && (kMulti || kStats)), "two-word genre masks: single-triple top-k sweeps only");
  static_assert(!(kFold && (kMulti || kStats || kDump || kG2)), "folded groups: single-triple top-k sweeps only");
  // Seed pass: hist[bin][row of the CTA] (32-bit counters; bank = row % 32, so the 32 lanes of a warp
  // never collide) in the two ring stages a seed launch does not use.  Bin 0 collects everything below
  // the range (and the columns a row may not name), bin b >= 1 the scores in
  // [lo + (b-1) w, lo + b w).  A row's seeded threshold is the lower edge of the bin in which the count
  // from the top reaches kp: at least kp sampled columns score that high, so the kp-th best of ALL columns
  // does too.  No lists, no compaction: the list-based seed pass spent 4/5 of its time selecting.
  constexpr int kHistBins = 64;
  static_assert(!kHist || (2 * A_BYTES >= kHistBins * BM * 4), "histogram does not fit two A stages");
  constexpr uint32_t GH_BYTES = BN * 8;  // second genre word of the tile's 256 columns
  constexpr int STAGES = L::STAGES;
  using R = Roles<(kMode != 0), kWide>;
  constexpr int EPI = R::EPI, PRODUCER_WARP = R::PRODUCER, MMA_WARP = R::MMA;
  constexpr int COLS_PER_WARP = BN / (EPI / 4);   // 256 (one-sided) or 128 (symmetric)
  constexpr int GW = (kWide && !kFold) ? 4 : 8;   // columns scored together (independent chains)
  const uint32_t nstages = static_cast<uint32_t>(p.stages);
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for the 128B-swizzled tiles; done as an OFFSET so the compiler still knows
  // these are shared-memory addresses (LDS/STS instead of generic loads)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::OFF_BAR);
  uint64_t* full = bars;                          // [STAGES] operands landed (leader's copy is used)
  uint64_t* empty = bars + STAGES;                // [STAGES] MMAs finished reading the stage
  uint64_t* acc_full = bars + 2 * STAGES;         // [2] accumulator complete
  uint64_t* acc_empty = bars + 2 * STAGES + 2;    // [2] accumulator drained (leader's copy is used)
  uint64_t* col_full = bars + 2 * STAGES + 4;     // [2] column-side records landed
  uint64_t* col_empty = bars + 2 * STAGES + 6;    // [2] column-side buffer free again
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + L::OFF_TMEM);
  unsigned int* hist = reinterpret_cast<unsigned int*>(smem + L::OFF_A + (STAGES - 2) * A_BYTES);   // kHist only

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  const int cluster_id = blockIdx.x / CG;
  const int num_clusters = gridDim.x / CG;

  if (warp == PRODUCER_WARP && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], 32 * EPI * CG);
      mbar_init(&col_full[b], 1);
      mbar_init(&col_empty[b], 32 * EPI);
    }
    fence_barrier_init();
  }
  if (warp == MMA_WARP) {
    if (CG == 2) tmem_alloc_pair(tmem_holder, 512);
    else tmem_alloc(tmem_holder, 512);
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  const int n_items = kDump ? 1
                            : ((p.rb_count + p.rb_per_group - 1) / p.rb_per_group) *
                                  p.rb_per_group * p.splits;

  if (warp == PRODUCER_WARP) {
    // =============================== TMA producer ===============================
    // the whole warp walks the loops (uniform control flow); one elected lane issues
    {
      uint32_t stage = 0, phase = 0, it = 0;
      Pacer pacer{p.sync_kb > 0 ? p.progress : nullptr, gridDim.x, p.sync_slack, 0u};
      const int chunks_per_tile = p.sync_kb > 0 ? (p.k_blocks + p.sync_kb - 1) / p.sync_kb : 0;
      for (int item = cluster_id; item < n_items; item += num_clusters) {
        ItemCoord c = item_coord<kAppend>(p, item);
        if (kDump) { c.sb = 0; c.tile0 = 0; c.tile1 = 1; }
        const int row0 = p.row_begin + (kDump ? 0 : c.sb * BM * CG) + static_cast<int>(cta_rank) * BM;
        for (int jt = c.tile0; jt < c.tile1; jt += p.tile_stride) {
          if (!kDump && (jt < c.real0 || jt >= c.real1)) {
            // phantom tile: keep the pacing counter moving, touch nothing else
            for (int ch = 0; ch < chunks_per_tile; ++ch) {
              pacer.wait_turn();
              pacer.done_chunk(lane == 0);
            }
            continue;
          }
          const uint32_t b = it & 1;
          const int col0 = kDump ? p.dump_col0 : jt * BN;
          if (!kDump) {
            mbar_wait_backoff(&col_empty[b], ((it >> 1) & 1) ^ 1, 16, p.wait_ns);  // epilogue done with buffer b
            if (elect_one()) {
              const uint32_t n_th = kMulti ? static_cast<uint32_t>(p.n_weights) : 1u;
              mbar_arrive_expect_tx(&col_full[b], (kFold ? 0u : COL_BYTES + MS_BYTES) +
                                                      ((kSym && !kStats && !kRepair && !kPairs) ? n_th * MS_BYTES : 0u) +
                                                      (kG2 ? GH_BYTES : 0u));
              if (!kFold) bulk_load_1d(smem + L::OFF_COL + b * COL_BYTES, p.col_side + col0, COL_BYTES, &col_full[b]);
              if (kG2)   // threshold slices 1-2 of this buffer (slice 0 holds the thresholds)
                bulk_load_1d(smem + L::OFF_TH + (b * kMaxSweep + 1) * MS_BYTES, p.genre_hi + col0, GH_BYTES,
                             &col_full[b]);
              if (!kFold) bulk_load_1d(smem + L::OFF_MS + b * MS_BYTES, p.meta_scale + col0, MS_BYTES, &col_full[b]);
              if (kSym && !kStats && !kRepair && !kPairs)  // snapshot of the column shows' thresholds (stale = lower = conservative)
                for (uint32_t w = 0; w < n_th; ++w)
                  bulk_load_1d(smem + L::OFF_TH + (b * kMaxSweep + w) * MS_BYTES,
                               p.g_theta + static_cast<size_t>(w) * (kMulti ? p.n_pad : 0) + col0, MS_BYTES,
                               &col_full[b]);
            }
            __syncwarp();
          }
          const int brow0 = col0 + static_cast<int>(cta_rank) * static_cast<int>(L::B_ROWS);
          for (int kb = 0; kb < p.k_blocks; ++kb) {
            if (p.sync_kb > 0 && kb % p.sync_kb == 0) {
              if (kb) pacer.done_chunk(lane == 0);
              pacer.wait_turn();
            }
            mbar_wait_backoff(&empty[stage], phase ^ 1, 16, p.wait_ns);
            if (elect_one()) {
              uint8_t* sa = smem + L::OFF_A + stage * A_BYTES;
              uint8_t* sb = smem + L::OFF_B + stage * L::B_BYTES;
              if (CG == 2) {
                // both CTAs' bytes are accounted on the leader's barrier
                if (leader) mbar_arrive_expect_tx(&full[stage], 2 * (A_BYTES + L::B_BYTES));
                tma_load_2d_pair(sa, &tmap_a, &full[stage], kb * BK, row0);
                tma_load_2d_pair(sb, &tmap_b, &full[stage], kb * BK, brow0);
              } else {
                mbar_arrive_expect_tx(&full[stage], A_BYTES + L::B_BYTES);
                tma_load_2d(sa, &tmap_a, &full[stage], kb * BK, row0);
                tma_load_2d(sb, &tmap_b, &full[stage], kb * BK, brow0);
              }
            }
            __syncwarp();
            if (++stage == nstages) { stage = 0; phase ^= 1; }
          }
          if (p.sync_kb > 0) pacer.done_chunk(lane == 0);
          ++it;
        }
      }
    }
  } else if (warp == MMA_WARP) {
    // =============================== MMA issuer (leader CTA) ====================
    // whole warp in the loops, one elected lane issues: keeps the descriptors in uniform registers
    if (leader) {
      uint32_t stage = 0, phase = 0, it = 0;
      // descriptor of stage 0; stage s / K sub-block k are reached by adding to the address field
      const uint64_t desc_a0 = umma_desc_sw128(smem_u32(smem + L::OFF_A));
      const uint64_t desc_b0 = umma_desc_sw128(smem_u32(smem + L::OFF_B));
      for (int item = cluster_id; item < n_items; item += num_clusters) {
        ItemCoord c = item_coord<kAppend>(p, item);
        if (kDump) { c.sb = 0; c.tile0 = 0; c.tile1 = 1; }
        if (c.sb < 0) continue;
        const int tile_beg = kDump ? c.tile0 : c.real0, tile_end = kDump ? c.tile1 : c.real1;
        for (int jt = tile_beg; jt < tile_end; jt += p.tile_stride, ++it) {
          const uint32_t b = it & 1;
          mbar_wait_backoff(&acc_empty[b], ((it >> 1) & 1) ^ 1, 16, p.wait_ns);  // every epilogue drained accumulator b
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + b * BN;
          for (int kb = 0; kb < p.k_blocks; ++kb) {
            mbar_wait_backoff(&full[stage], phase, 64, 32);
            tc_fence_after();
            if (elect_one()) {
              const uint64_t da = desc_a0 + static_cast<uint64_t>(stage * (A_BYTES >> 4));
              const uint64_t db = desc_b0 + static_cast<uint64_t>(stage * (L::B_BYTES >> 4));
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                // advance 32 bytes (16 halves) along K inside the 128-byte swizzle row
                const uint64_t ka = da + static_cast<uint64_t>(k * 2), kb2 = db + static_cast<uint64_t>(k * 2);
                if (CG == 2) umma_f16_pair(tmem_d, ka, kb2, idesc, (kb | k) != 0 ? 1u : 0u);
                else umma_f16(tmem_d, ka, kb2, idesc, (kb | k) != 0 ? 1u : 0u);
              }
              // smem slot reusable once these MMAs have read it; accumulator ready after the last
              if (CG == 2) {
                umma_commit_pair(&empty[stage]);
                if (kb == p.k_blocks - 1) umma_commit_pair(&acc_full[b]);
              } else {
                umma_commit(&empty[stage]);
                if (kb == p.k_blocks - 1) umma_commit(&acc_full[b]);
              }
            }
            __syncwarp();
            if (++stage == nstages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else {
    // =============================== epilogue ===================================
    const int quarter = warp & 3;                 // TMEM lanes this warp may touch
    const int row_in_tile = quarter * 32 + lane;
    const uint32_t tmem_lane = static_cast<uint32_t>(quarter * 32) << 16;
    constexpr int CAP = 32 * E;
    uint2* my_list = p.scratch + (static_cast<size_t>(blockIdx.x) * BM + row_in_tile) * CAP;
    uint32_t it = 0;
    // ---- statistics sweep state (kStats): per-thread fp64 sums, extrema, argmax of text / hybrid,
    // and a CTA-wide histogram in the shared memory of the (unused) last ring stage
    double st_sum[4] = {0, 0, 0, 0}, st_sq[4] = {0, 0, 0, 0}, st_gm = 0.0;
    float st_min[4] = {3e38f, 3e38f, 3e38f, 3e38f}, st_max[4] = {-1.f, -1.f, -1.f, -1.f};
    unsigned long long st_zero[4] = {0, 0, 0, 0};
    int st_arg_i[2] = {-1, -1}, st_arg_j[2] = {-1, -1};
    float st_arg_v[2] = {-1.f, -1.f};
    unsigned int* shist = reinterpret_cast<unsigned int*>(smem + L::OFF_A + (STAGES - 1) * A_BYTES);
    if (kStats) {
      for (int b = threadIdx.x; b < 4 * kStatsBins; b += 32 * EPI) shist[b] = 0u;
      asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI) : "memory");
    }
    if (kHist) {
      for (int i = threadIdx.x; i < kHistBins * BM; i += 32 * EPI) hist[i] = 0u;
      asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI) : "memory");
    }
    // symmetric sweeps: this warp's ring of pending list appends and its (warp-uniform) fill count
    uint32_t* ring = reinterpret_cast<uint32_t*>(smem + L::OFF_Q) + warp * (3 * RING);
    int ring_n = 0;
    for (int item = cluster_id; item < n_items; item += num_clusters) {
      ItemCoord c = item_coord<kAppend>(p, item);
      if (kDump) { c.sb = 0; c.tile0 = 0; c.tile1 = 1; }
      if (c.sb < 0) continue;
      const int row_local0 = (kDump ? 0 : c.sb * BM * CG) + static_cast<int>(cta_rank) * BM;  // within shard
      const int grow = p.row_begin + row_local0 + row_in_tile;
      const bool row_valid = kGather ? grow < p.upd_q : grow < p.row_end;
      const int row = kGather ? (row_valid ? p.upd_rows[grow] : -1) : grow;   // the show of this row
      const int lrow = kRepair ? grow : row;   // the list (and threshold) of this row
      // refresh: a row of A (its scores are unchanged) feeds its own list only
      const bool feeds_cols = !kRefresh || (row_valid && ((p.upd_sbits[row >> 5] >> (row & 31)) & 1u) != 0u);
      // row-side operands of the fused scores
      unsigned long long g_bits = 0ull, g_hi = 0ull;
      uint32_t m_bits = 0u;
      float rn_wg = 0.0f, ci_wm = 0.0f;
      if (row_valid && !kDump && !kFold) {
        const TvbfColSide rs = p.col_side[row];
        g_bits = rs.genre_bits;
        if (kG2) g_hi = p.genre_hi[row];
        m_bits = rs.meta_bits;
        rn_wg = rs.genre_rnorm * p.w_genre;
        // MEAN3: (matches / 3) * w = matches * (1/sqrt3)^2 * w; HSTACK: per-show 1/sqrt(#categories);
        // meta_scale[] holds the factor of either kind, for the row here and per column in the epilogue
        ci_wm = p.meta_scale[row] * p.w_meta;
        if (kStats || kMulti) {  // plain cosines here; the weights enter only the hybrid
          rn_wg = rs.genre_rnorm;
          ci_wm = p.meta_scale[row];
        }
      }
      float theta = row_valid ? p.theta_init : __int_as_float(0x7f800000);  // +inf: never append
      float thw[kMaxSweep];   // weight sweep: this show's threshold under every triple
#pragma unroll
      for (int w = 0; w < kMaxSweep; ++w) thw[w] = __int_as_float(0x7f800000);
      auto load_thw = [&]() {
#pragma unroll
        for (int w = 0; w < kMaxSweep; ++w)
          if (w < p.n_weights && row_valid) {
            unsigned int tb;
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];"
                         : "=r"(tb) : "l"(p.g_theta + static_cast<size_t>(w) * p.n_pad + row) : "memory");
            thw[w] = __uint_as_float(tb);
          }
      };
      int cnt = 0;
      bool dropped = false;
      const int self_col = p.exclude_self ? row : -1;
      // per-row slack of the upper bound: the accumulation error is bounded per non-zero product,
      // and a pair has at most `terms` of them (non-zero operand entries of this row)
      float terms = 0.0f;
      if (row_valid && !kDump && !kStats)
        terms = static_cast<float>(p.text_indptr[row + 1] - p.text_indptr[row]) + static_cast<float>(p.folded_cols);
      const float w_text = p.w_text, w_text_err = fmaf(terms, p.w_text_acc, p.w_text_err),
                  eps = fmaf(terms, p.eps_term, p.eps);
      const float w_fold = w_text + w_text_err;   // kFold: upper bound = acc * (w + err) + eps
      const unsigned sym_cap = static_cast<unsigned>(p.sym_cap);

      // Shared-list appends need the slot returned by an atomicAdd; done on the spot that round trip
      // (~700 cycles) would stall the warp once per append.  Appends are therefore collected in a
      // per-warp ring in shared memory -- filled densely by warp-uniform code: ballot + prefix, the
      // fill count lives in a register -- and drained by sym_ring_flush with one entry per lane, all
      // atomics of the ring in flight together.  A later append only delays a candidate, it never
      // loses one.
      auto ring_flush = [&]() {
        __syncwarp();
        if constexpr (kPairs) pair_ring_flush(ring, ring_n, p.pair_count, p.pairs, p.pair_cap, lane);
        else sym_ring_flush(ring, ring_n, p.g_cnt, p.g_list, p.g_theta, sym_cap, p.kp, p.refresh_period, lane);
        ring_n = 0;
        __syncwarp();
      };
      // hits: bit e (e < GW) = offer u[e] to this thread's show, bit GW + e = offer it to column
      // colbase + e; voff = first virtual show id of the weight triple
      auto push_hits = [&](uint32_t hits, const float (&u)[GW], int colbase, int voff) {
        while (__any_sync(kFullMask, hits != 0u)) {   // warp-uniform: max hits of any lane (usually 1)
          if (ring_n > RING - 32) ring_flush();
          const int bit = hits != 0u ? __ffs(hits) - 1 : 0;
          const bool to_row = bit < GW;
          const float ue = pick<GW>(u, bit & (GW - 1));
          const int col = colbase + (bit & (GW - 1));
          // a row-side append may only name a real show other than the row's own (checked here, on the
          // rare path, instead of masking every group); padded columns carry threshold +inf
          const bool act = hits != 0u && (!to_row || (col != self_col && col < p.n_shows));
          hits &= hits - 1u;
          const unsigned m = __ballot_sync(kFullMask, act);
          const int slot = ring_n + __popc(m & ((1u << lane) - 1u));
          if (act) {
            ring[slot] = static_cast<uint32_t>(voff + (to_row ? lrow : col));
            ring[RING + slot] = __float_as_uint(ue);
            ring[2 * RING + slot] = static_cast<uint32_t>(to_row ? col : row);
          }
          ring_n += __popc(m);
        }
      };
      // neighbour sweep: bit e of hits = U of column colbase + e passed; only the pairs row < column
      // < n_shows are kept (the diagonal tile holds both orders of its pairs and the show itself)
      auto push_pairs = [&](uint32_t hits, int colbase) {
        if (!__any_sync(kFullMask, hits != 0u)) return;   // the usual case: one vote per group
        const int lo = row + 1 - colbase, hi = p.n_shows - colbase;   // bits [lo, hi) are real columns > row
        if (lo > 0) hits = lo >= GW ? 0u : hits & ~((1u << lo) - 1u);
        if (hi < GW) hits = hi <= 0 ? 0u : hits & ((1u << hi) - 1u);
        while (__any_sync(kFullMask, hits != 0u)) {
          if (ring_n > RING - 32) ring_flush();
          const bool act = hits != 0u;
          const int col = colbase + (act ? __ffs(hits) - 1 : 0);
          hits &= hits - 1u;
          const unsigned m = __ballot_sync(kFullMask, act);
          const int slot = ring_n + __popc(m & ((1u << lane) - 1u));
          if (act) {
            ring[slot] = static_cast<uint32_t>(row);
            ring[RING + slot] = static_cast<uint32_t>(col);
          }
          ring_n += __popc(m);
        }
      };

      const int tile_beg = kDump ? c.tile0 : c.real0, tile_end = kDump ? c.tile1 : c.real1;
      for (int jt = tile_beg; jt < tile_end; jt += p.tile_stride, ++it) {
        const uint32_t b = it & 1;
        const uint32_t ph = (it >> 1) & 1;
        const int col0 = kDump ? p.dump_col0 : jt * BN;
        if (kMulti) {
          load_thw();
        } else if (kSym && !kStats && !kPairs) {
          // current shared threshold of this thread's show (raised by any CTA working on it)
          unsigned int tb = 0x7f800000u;
          if (row_valid)
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(tb) : "l"(p.g_theta + lrow) : "memory");
          theta = __uint_as_float(tb);
        }
        if (!kDump) mbar_wait_backoff(&col_full[b], ph, 32, 32);
        mbar_wait_backoff(&acc_full[b], ph, 32, 32);
        tc_fence_after();
        const TvbfColSide* scol = reinterpret_cast<const TvbfColSide*>(smem + L::OFF_COL + b * COL_BYTES);
        const float* sms = reinterpret_cast<const float*>(smem + L::OFF_MS + b * MS_BYTES);
        const float* sth = reinterpret_cast<const float*>(smem + L::OFF_TH + b * kMaxSweep * MS_BYTES);
        const unsigned long long* sgh =
            reinterpret_cast<const unsigned long long*>(smem + L::OFF_TH + (b * kMaxSweep + 1) * MS_BYTES);
        const uint32_t taddr = tmem_base + tmem_lane + b * BN;
        // off-diagonal tiles also feed the column shows (their mirror tile is never computed); the
        // update sweep's rectangle has no mirror tiles; the repair sweep feeds its rows only
        const bool do_col = kSym && !kRepair && row_valid && (kUpdate || jt != c.sb) && feeds_cols;

        float tile_sum[4] = {0.f, 0.f, 0.f, 0.f}, tile_sq[4] = {0.f, 0.f, 0.f, 0.f}, tile_gm = 0.f;
        float stat_scale[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) stat_scale[q] = kStats ? static_cast<float>(kStatsBins) / p.stats->hi[q] : 0.f;

        // plain genre / metadata dots of accumulator column cbase + e against this thread's show
        auto side_dots = [&](int ce, float& gdot, float& mdot) {
          // one LDS.128: {genre bits lo, hi, 1/sqrt(popcount) as float bits, metadata bits}
          const uint4 cs = reinterpret_cast<const uint4*>(scol)[ce];
          int gcount = __popc(static_cast<uint32_t>(g_bits) & cs.x) + __popc(static_cast<uint32_t>(g_bits >> 32) & cs.y);
          if (kG2) gcount += __popcll(g_hi & sgh[ce]);
          gdot = static_cast<float>(gcount) * __uint_as_float(cs.z);
          // per-column scale: 1/sqrt(#categories) (HSTACK) or 1/sqrt(3) (MEAN3: matches / 3), 0 for padding
          mdot = static_cast<float>(__popc(m_bits & cs.w)) * sms[ce];
        };
        // Score 16 accumulator columns held in registers.  The candidate sweeps (everything but the
        // statistics and dump variants) are written BRANCH-FREE: the sixteen upper bounds are
        // independent dependency chains (LDS -> POPC -> I2F -> FMUL -> 4 FFMA) the scheduler can
        // overlap (in groups of GW = 8, or 4 under the 96-register cap of the 16-warp variant), and the comparisons only set
        // bits of two hit masks.  With a branch per element
        // (round 1) the chains ran one after the other and the epilogue was latency-bound at ~13 % of
        // the issue slots on small vocabularies.
        auto score16 = [&](const uint32_t (&acc)[16], int cbase) {
          if constexpr (kDump) {
#pragma unroll
            for (int e = 0; e < 16; ++e)
              p.dump[(row_local0 + row_in_tile) * BN + cbase + e] = __uint_as_float(acc[e]);
          } else if constexpr (kStats) {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const float a = __uint_as_float(acc[e]);
              float gdot, mdot;
              side_dots(cbase + e, gdot, mdot);
              const int col = col0 + cbase + e;
              if (row_valid && col > row && col < p.n_shows) {   // strict upper triangle
                float v[4];
                v[0] = gdot * rn_wg;
                v[1] = a * p.inv_scale2;
                v[2] = mdot * ci_wm;
                v[3] = fmaf(p.w_genre, v[0], fmaf(p.w_text_plain, v[1], p.w_meta * v[2]));
                tile_gm = fmaf(v[0], v[2], tile_gm);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  tile_sum[q] += v[q];
                  tile_sq[q] = fmaf(v[q], v[q], tile_sq[q]);
                  st_min[q] = fminf(st_min[q], v[q]);
                  st_max[q] = fmaxf(st_max[q], v[q]);
                  if (v[q] == 0.0f) {
                    ++st_zero[q];
                  } else {
                    int bin = static_cast<int>(v[q] * stat_scale[q]);
                    bin = bin < 0 ? 0 : (bin >= kStatsBins ? kStatsBins - 1 : bin);
                    atomicAdd(&shist[q * kStatsBins + bin], 1u);
                  }
                }
                if (v[1] > st_arg_v[0]) { st_arg_v[0] = v[1]; st_arg_i[0] = row; st_arg_j[0] = col; }
                if (v[3] > st_arg_v[1]) { st_arg_v[1] = v[3]; st_arg_i[1] = row; st_arg_j[1] = col; }
              }
            }
          } else if constexpr (kMulti) {
            // Weight sweep: the plain cosines of 8 columns once, then one branch-free pass per triple
            // (rolled over the triples so that the code stays the size of the single-triple kernel).
            // Triple w's lists live under the virtual show id w * n_pad + show.
#pragma unroll
            for (int h = 0; h < 16 / GW; ++h) {
              float gcv[GW], mcv[GW];
#pragma unroll
              for (int e = 0; e < GW; ++e) {
                float gdot, mdot;
                side_dots(cbase + h * GW + e, gdot, mdot);
                gcv[e] = gdot * rn_wg;
                mcv[e] = mdot * ci_wm;
              }
#pragma unroll 1
              for (int w = 0; w < p.n_weights; ++w) {
                const float wg = p.mw_genre[w], wm = p.mw_meta[w], wt = p.mw_text[w],
                            wte = fmaf(terms, p.mw_text_acc[w], p.mw_text_err[w]),
                            we = fmaf(terms, p.mw_eps_term[w], p.mw_eps[w]);
                const float th = w == 0 ? thw[0] : (w == 1 ? thw[1] : (w == 2 ? thw[2] : (w == 3 ? thw[3] : thw[4])));
                const float4* t4p = reinterpret_cast<const float4*>(sth + w * BN + cbase + h * GW);
                float u[GW];
                uint32_t hit_r = 0u, hit_c = 0u;
#pragma unroll
                for (int e4 = 0; e4 < GW / 4; ++e4) {
                  const float4 t4 = t4p[e4];
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    const int e = e4 * 4 + q;
                    const float a = __uint_as_float(acc[h * GW + e]);
                    float uw = fmaf(gcv[e], wg, fmaf(mcv[e], wm, we));
                    uw = fmaf(a, wt, uw);
                    uw = fmaf(fabsf(a), wte, uw);
                    u[e] = uw;
                    const float tc = q == 0 ? t4.x : (q == 1 ? t4.y : (q == 2 ? t4.z : t4.w));
                    hit_r |= uw > th ? (1u << e) : 0u;
                    hit_c |= uw > tc ? (1u << e) : 0u;   // padded columns carry threshold +inf
                  }
                }
                if (!do_col) hit_c = 0u;
                push_hits(hit_r | (hit_c << GW), u, col0 + cbase + h * GW, w * p.n_pad);
              }
            }
          } else {
#pragma unroll
            for (int h = 0; h < 16 / GW; ++h) {
              float u[GW];
              uint32_t hit_r = 0u, hit_c = 0u;
#pragma unroll
              for (int e4 = 0; e4 < GW / 4; ++e4) {
                float4 t4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (kSym && !kPairs) t4 = reinterpret_cast<const float4*>(sth + cbase + h * GW)[e4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const int e = e4 * 4 + q;
                  const float a = __uint_as_float(acc[h * GW + e]);
                  float ue;
                  if (kFold) {
                    ue = fmaf(a, w_fold, eps);   // all products are non-negative: |a| == a
                  } else {
                    float gdot, mdot;
                    side_dots(cbase + h * GW + e, gdot, mdot);
                    ue = fmaf(gdot, rn_wg, fmaf(mdot, ci_wm, eps));
                    ue = fmaf(a, w_text, ue);
                    ue = fmaf(fabsf(a), w_text_err, ue);
                  }
                  u[e] = ue;
                  hit_r |= ue > theta ? (1u << e) : 0u;
                  if (kSym && !kPairs) {
                    const float tc = q == 0 ? t4.x : (q == 1 ? t4.y : (q == 2 ? t4.z : t4.w));
                    hit_c |= ue > tc ? (1u << e) : 0u;   // padded columns carry threshold +inf
                  }
                }
              }
              if constexpr (kPairs) {
                push_pairs(hit_r, col0 + cbase + h * GW);
              } else if (kSym) {
                if (!do_col) hit_c = 0u;
                if constexpr (kAppend) {
                  // a pair of two old shows is in the previous table already (or ranks below all of it):
                  // offered to neither list.  Only the column tile append_b0 mixes old and new columns.
                  const int old_cols = p.append_n_old - (col0 + cbase + h * GW);
                  if (row < p.append_n_old && old_cols > 0) {
                    const uint32_t m = old_cols >= GW ? (1u << GW) - 1u : (1u << old_cols) - 1u;
                    hit_r &= ~m;
                    hit_c &= ~m;
                  }
                }
                if constexpr (kUpdate) {
                  // an updated column has a gathered row of its own, which offers it this pair
                  if (hit_c != 0u) {
                    const int c0 = col0 + cbase + h * GW;   // GW-aligned: one word of the bit set
                    hit_c &= ~((p.upd_bits[c0 >> 5] >> (c0 & 31)) & ((1u << GW) - 1u));
                  }
                }
                push_hits(hit_r | (hit_c << GW), u, col0 + cbase + h * GW, 0);
              } else if (kHist) {
#pragma unroll
                for (int e = 0; e < GW; ++e) {
                  const int col = col0 + cbase + h * GW + e;
                  int bin = __float2int_rd(fmaf(u[e], p.hist_inv_w, p.hist_off));
                  bin = min(max(bin, 0), kHistBins - 1);
                  if (col == self_col || col >= p.n_shows) bin = 0;
                  atomicAdd(&hist[bin * BM + row_in_tile], 1u);
                }
              } else {
                // private list of this thread's row (at most GW appends; 32 free slots are guaranteed)
                while (hit_r) {
                  const int e = __ffs(hit_r) - 1;
                  hit_r &= hit_r - 1u;
                  const int col = col0 + cbase + h * GW + e;
                  if (col != self_col && col < p.n_shows) {
                    __stcg(my_list + cnt, make_uint2(__float_as_uint(pick<GW>(u, e)), static_cast<uint32_t>(col)));
                    ++cnt;
                  }
                }
              }
            }
          }
        };

        // 16 chunks of 16 columns, two per loop iteration so that the TMEM load of the next chunk
        // is in flight while the current one is scored.  The loop is kept rolled on purpose: the
        // whole body stays resident in the instruction cache.
        uint32_t acc_a[16], acc_b[kWide ? 1 : 16];
        const int ch0 = (warp >> 2) * (COLS_PER_WARP / 16), ch1 = ch0 + COLS_PER_WARP / 16;
        if (!kWide) tmem_ld_32x16(taddr + ch0 * 16, acc_a);
#pragma unroll 1
        for (int ch = ch0; ch < ch1; ch += 2) {
          if constexpr (kWide) {
            // 16 epilogue warps: four warps per scheduler hide the TMEM load latency, and the register
            // budget (96 per thread at 576 threads) has no room for a second accumulator buffer
#pragma unroll 1
            for (int c2 = ch; c2 < ch + 2; ++c2) {
              tmem_ld_32x16(taddr + c2 * 16, acc_a);
              tmem_ld_wait();
              if (c2 + 1 >= ch1) {
                tc_fence_before();
                if (CG == 2) mbar_arrive_cluster(&acc_empty[b], 0u);
                else mbar_arrive(&acc_empty[b]);
              }
              score16(acc_a, c2 * 16);
            }
          } else {
            tmem_ld_wait();
            tmem_ld_32x16(taddr + (ch + 1) * 16, acc_b);
            score16(acc_a, ch * 16);
            tmem_ld_wait();
            if (ch + 2 < ch1) {
              tmem_ld_32x16(taddr + (ch + 2) * 16, acc_a);
            } else {
              // every accumulator column of this tile is in registers: hand the TMEM buffer back
              tc_fence_before();
              if (CG == 2) mbar_arrive_cluster(&acc_empty[b], 0u);
              else mbar_arrive(&acc_empty[b]);
            }
            score16(acc_b, (ch + 1) * 16);
          }
          if (kSym && !kStats) {
            // drain the ring when it holds two full passes of the flush, or a lane-full at the end of
            // the tile; then pick up the raises made by other CTAs (and by the refreshes of the flush)
            const bool tile_done = ch + 2 >= ch1;
            if (ring_n >= 64 || (tile_done && ring_n >= 32)) {
              ring_flush();
              if (kMulti) {
                load_thw();
              } else if (!kPairs && row_valid) {
                unsigned int tb;
                asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(tb) : "l"(p.g_theta + lrow) : "memory");
                theta = __uint_as_float(tb);
              }
            }
          } else if (!kDump && !kSym && !kHist) {
            // keep 32 free slots for the next 32 columns; compact rows that are nearly full
            unsigned need = __ballot_sync(kFullMask, cnt > CAP - 32);
            while (need) {
              const int src_lane = __ffs(need) - 1;
              need &= need - 1;
              const uint2* lp = reinterpret_cast<const uint2*>(__shfl_sync(
                  kFullMask, reinterpret_cast<unsigned long long>(my_list), src_lane));
              const int n = __shfl_sync(kFullMask, cnt, src_lane);
              const float bound = warp_select_compact<E>(const_cast<uint2*>(lp), n, p.kp, lane);
              if (lane == src_lane) {
                cnt = p.kp;
                theta = fmaxf(theta, bound);
                dropped = true;
              }
            }
          }
        }
        if (!kDump) mbar_arrive(&col_empty[b]);  // column-side buffer b may be refilled
        if (kStats) {
#pragma unroll
          for (int q = 0; q < 4; ++q) { st_sum[q] += tile_sum[q]; st_sq[q] += tile_sq[q]; }
          st_gm += tile_gm;
        }
      }
      if (kSym && !kStats && ring_n > 0) ring_flush();   // nothing stays queued past the item (or the kernel)

      if (kHist) {
        // every epilogue warp has added its columns: the first warp of each lane quarter turns the 32
        // histograms of its rows into thresholds and clears them for the next item
        asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI) : "memory");
        if ((warp >> 2) == 0) {
          int c = 0, found = 0;
          hist[row_in_tile] = 0u;
#pragma unroll 4
          for (int bin = kHistBins - 1; bin >= 1; --bin) {
            c += static_cast<int>(hist[bin * BM + row_in_tile]);
            hist[bin * BM + row_in_tile] = 0u;
            if (c >= p.kp && found == 0) found = bin;
          }
          if (found != 0 && row_valid) {
            // lower edge of the bin, minus a margin for the rounding of the bin computation
            const float th = fmaf(static_cast<float>(found - 1) - 1e-3f, p.hist_w, p.hist_lo);
            if (th > p.theta_init) p.g_theta[row] = __float_as_uint(th);
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI) : "memory");
      }

      if (!kDump && !kSym && !kHist) {
        // final compaction of every row of this warp: sorted best-kp list -> cand
        const int rows_in_shard = p.row_end - p.row_begin;
        for (int src_lane = 0; src_lane < 32; ++src_lane) {
          const int r = row_local0 + quarter * 32 + src_lane;  // row within the shard
          if (r >= rows_in_shard) break;                       // warp-uniform
          const uint2* lp = reinterpret_cast<const uint2*>(__shfl_sync(
              kFullMask, reinterpret_cast<unsigned long long>(my_list), src_lane));
          const int n = __shfl_sync(kFullMask, cnt, src_lane);
          if (p.seed_theta) {
            // sampled sweep: the kp-th best sampled score is a valid lower bound of the show's
            // final threshold; it spares the symmetric sweep its warm-up flood of appends
            float bound = warp_select_compact<E>(const_cast<uint2*>(lp), n, p.kp, lane);
            if (n == p.kp) {   // exactly kp sampled candidates: the smallest of them
              float mn = __int_as_float(0x7f800000);
              for (int i = lane; i < n; i += 32) mn = fminf(mn, __uint_as_float(__ldcg(lp + i).x));
#pragma unroll
              for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(kFullMask, mn, o));
              bound = mn;
            }
            if (lane == src_lane && n >= p.kp && bound > p.theta_init)
              p.g_theta[p.row_begin + r] = __float_as_uint(bound);
            continue;
          }
          uint2* dst = p.cand + (static_cast<size_t>(r) * p.splits + c.split) * p.kp;
          const float bound = warp_compact<E>(lp, n, dst, p.kp, lane);
          if (lane == src_lane) {
            float th = dropped ? theta : __int_as_float(0xff800000);  // -inf: nothing dropped
            if (n > p.kp) th = fmaxf(dropped ? theta : bound, bound);
            p.cand_cnt[static_cast<size_t>(r) * p.splits + c.split] = n < p.kp ? n : p.kp;
            p.cand_theta[static_cast<size_t>(r) * p.splits + c.split] = th;
          }
        }
      }
    }
    if (kStats) {
      StatsAccum* sa = p.stats;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        double s1 = st_sum[q], s2 = st_sq[q];
        unsigned long long z = st_zero[q];
        float mn = st_min[q], mx = st_max[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          s1 += __shfl_xor_sync(kFullMask, s1, o);
          s2 += __shfl_xor_sync(kFullMask, s2, o);
          z += __shfl_xor_sync(kFullMask, z, o);
          mn = fminf(mn, __shfl_xor_sync(kFullMask, mn, o));
          mx = fmaxf(mx, __shfl_xor_sync(kFullMask, mx, o));
        }
        if (lane == 0) {
          atomicAdd(&sa->sum[q], s1);
          atomicAdd(&sa->sumsq[q], s2);
          atomicAdd(&sa->zeros[q], z);
          if (mx >= 0.f) {   // at least one element seen (all values are >= 0)
            atomicMin(&sa->min_bits[q], __float_as_uint(mn));
            atomicMax(&sa->max_bits[q], __float_as_uint(mx));
          }
        }
      }
      {
        double s = st_gm;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
        if (lane == 0) atomicAdd(&sa->sum_gm, s);
      }
      // argmax candidates of text (0) and hybrid (1): best of the warp -> one slot per warp
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        float v = st_arg_v[q];
        int bi = st_arg_i[q], bj = st_arg_j[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(kFullMask, v, o);
          const int oi = __shfl_xor_sync(kFullMask, bi, o), oj = __shfl_xor_sync(kFullMask, bj, o);
          if (ov > v) { v = ov; bi = oi; bj = oj; }
        }
        if (lane == 0 && bi >= 0) {
          const int slot = (blockIdx.x * EPI + warp) % kStatsCand;   // private to this warp (grid <= 256 CTAs)
          if (v > sa->cand_val[q][slot]) {
            sa->cand_val[q][slot] = v;
            sa->cand_ij[q][slot][0] = bi;
            sa->cand_ij[q][slot][1] = bj;
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI) : "memory");
      for (int b = threadIdx.x; b < 4 * kStatsBins; b += 32 * EPI)
        if (shist[b]) atomicAdd(&sa->hist[b / kStatsBins][b % kStatsBins], static_cast<unsigned long long>(shist[b]));
    }
  }

  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_pair(tmem_base, 512);
    else tmem_dealloc(tmem_base, 512);
  }
}

// K4s: symmetric mode -- one warp per show: keep the kp best entries of its shared list as the
// candidate set and derive the bound on everything that is not in it.
// Lists of up to 32 * Q entries are selected in one go from registers (Q per lane; Q = 8 covers the
// usual list and every partial list of a multi-GPU job at a quarter of the compares, Q = 32 the
// rest).  Longer ones (kp > 64, Q = 32) in windows: the kp survivors so far, parked at the head of
// the list, plus the next 1024 - kp entries; the kp-th value only rises from window to window, so
// the last one bounds everything that was cut.  All loads of a window are issued back to back.
template <int Q>
__device__ __forceinline__ void compact_list(uint2* list, int n_all, int kp, uint2* dst, int lane,
                                             uint32_t* best_out, int* kept_out) {
  constexpr int W = 32 * Q;
  uint32_t best = 0u;  // kp-th largest score bits (0 when n <= kp)
  int done = 0, kept = 0;
  do {
    const int fresh = n_all - done < W - kept ? n_all - done : W - kept;
    const int n = kept + fresh;
    uint32_t v[Q], cidx[Q];
    uint32_t lo = 0xFFFFFFFFu, hi = 0u;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int idx = q * 32 + lane;
      uint2 e = make_uint2(0u, 0u);
      if (idx < n) e = __ldcg(list + (idx < kept ? idx : done + (idx - kept)));
      v[q] = idx < n ? e.x : 0u;
      cidx[q] = e.y;
      if (idx < n) { lo = min(lo, v[q]); hi = max(hi, v[q]); }
    }
    done += fresh;
    const bool last = done >= n_all;
    uint2* out_p = last ? dst : list;
    best = 0u;
    if (n > kp) {
      // exact radix select below the bits all n entries share (scores of one list lie within a
      // factor of two: sign, exponent and the leading mantissa bits are skipped)
      lo = __reduce_min_sync(kFullMask, lo);
      hi = __reduce_max_sync(kFullMask, hi);
      const int top = 31 - __clz(lo ^ hi);     // -1: all entries equal
      best = top >= 0 ? (hi >> (top + 1)) << (top + 1) : hi;   // positive floats: top <= 30
#pragma unroll 1
      for (int bit = top; bit >= 0; --bit) {
        const uint32_t t = best | (1u << bit);
        int c = 0;
#pragma unroll
        for (int q = 0; q < Q; ++q) c += (v[q] >= t);
        c = __reduce_add_sync(kFullMask, c);
        if (c >= kp) best = t;
      }
    }
    __syncwarp();   // all loads of this window are done before its head is overwritten
    // entries strictly above the kp-th value always fit; entries equal to it fill the rest
    int out = 0;
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int idx = q * 32 + lane;
        const bool take = idx < n && (pass == 0 ? v[q] > best : v[q] == best);
        const unsigned bal = __ballot_sync(kFullMask, take);
        const int pos = out + __popc(bal & ((1u << lane) - 1u));
        if (take && pos < kp) out_p[pos] = make_uint2(v[q], cidx[q]);
        out += __popc(bal);
      }
      if (n <= kp) break;  // everything was taken in pass 0 (best == 0, all scores positive)
    }
    kept = n < kp ? n : kp;
    __syncwarp();
    if (last) break;
    __threadfence_block();
  } while (true);
  *best_out = best;
  *kept_out = kept;
}

__global__ void __launch_bounds__(128, 6)
sym_compact_kernel(const K1Params p, int n_rows) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const unsigned total = p.g_cnt[r];
  const int n_all = static_cast<int>(total < static_cast<unsigned>(p.sym_cap) ? total : p.sym_cap);
  if (p.dbg_entries != nullptr && lane == 0) atomicAdd(p.dbg_entries, n_all >> 4);   // in units of 16 entries
  uint2* list = p.g_list + static_cast<size_t>(r) * p.sym_cap;
  const int kp = p.kp;
  uint2* dst = p.cand + static_cast<size_t>(r) * (p.cand_packed ? kp + 1 : kp);
  if (p.cand_packed == 2) {
    // fused compaction + exchange: the finished list goes to the GPU that rescores this show
    const int owner = r / p.peer_shard_rows;
    dst = p.peer_cand[owner] + (static_cast<size_t>(p.peer_rank) * p.peer_shard_rows + (r - owner * p.peer_shard_rows)) *
                                   static_cast<size_t>(kp + 1);
  }
  uint32_t best = 0u;
  int kept = 0;
  if (n_all <= 256) compact_list<8>(list, n_all, kp, dst, lane, &best, &kept);     // warp-uniform
  else if (n_all <= 512) compact_list<16>(list, n_all, kp, dst, lane, &best, &kept);
  else compact_list<32>(list, n_all, kp, dst, lane, &best, &kept);
  if (lane == 0) {
    const unsigned int th_bits = p.g_theta[r];
    float bound = __int_as_float(0xff800000);                        // nothing dropped so far
    if (th_bits > __float_as_uint(p.theta_init)) bound = __uint_as_float(th_bits);  // elements were rejected
    if (n_all > kp) bound = fmaxf(bound, __uint_as_float(best));     // list entries cut here
    if (total > static_cast<unsigned>(p.sym_cap)) bound = __int_as_float(0x7f800000);  // overflow: send to K6
    if (p.cand_packed) {
      dst[kp] = make_uint2(static_cast<unsigned>(kept), __float_as_uint(bound));
    } else {
      p.cand_cnt[r] = kept;
      p.cand_theta[r] = bound;
    }
  }
}

__global__ void sym_init_kernel(unsigned int* theta, int n_shows, int n_pad, int n_virtual, float theta_init) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_virtual) theta[i] = (i % n_pad) < n_shows ? __float_as_uint(theta_init) : 0x7f800000u;
}

// Append: every old show's previous row becomes its candidate list 1 (bound -inf: an old column missing
// from the row ranks below all k entries of it and can never enter), and an old show with a full row
// starts the sweep with the largest float strictly BELOW its k-th previous score -- a new column that
// does not beat that cannot enter either, and the strict certificate "theta < k-th" of K5 still passes
// for an unchanged row.  New shows get an empty list 1 and keep their seeded thresholds.
__global__ void append_prev_kernel(AppendPrev a, unsigned int* theta, float theta_init, int n_shows, int kp) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_shows) return;
  int cnt = 0;
  if (r < a.n_old) {
    cnt = a.counts[r];
    uint2* dst = a.list + static_cast<size_t>(r) * kp;
    const size_t base = static_cast<size_t>(r) * a.k;
    for (int e = 0; e < cnt; ++e)
      dst[e] = make_uint2(__float_as_uint(__double2float_ru(a.hybrid[base + e])), static_cast<uint32_t>(a.indices[base + e]));
    float th = theta_init;   // a short row: every new column that qualifies may enter
    if (cnt == a.k) {
      const double kth = a.hybrid[base + a.k - 1];
      th = __double2float_rd(kth);
      if (static_cast<double>(th) >= kth) th = nextafterf(th, -INFINITY);
      th = fmaxf(th, theta_init);
    }
    theta[r] = __float_as_uint(th);   // (the seed pass over block append_b0 also wrote the old shows there)
  }
  a.cnt[r] = cnt;
  a.bound[r] = __int_as_float(0xff800000);
}

// Update: a show that was not updated gets its previous row without the updated shows as list 1 (bound
// -inf) and, when that row was full, the threshold of append_prev_kernel and a rank cut at its previous
// k-th entry e_k: a column missing from the row that was not updated ranks below e_k, and K5 accepts the
// merged row only if its k-th entry ranks at or above e_k.  An updated show gets an empty list 1, no
// cut, and keeps the threshold its seed pass writes.
__global__ void update_prev_kernel(UpdatePrev a, unsigned int* theta, float theta_init, int n_shows, int kp) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_shows) return;
  int cnt = 0, cut_j = -1;
  double cut_h = 0.0;
  if (((a.upd_bits[r >> 5] >> (r & 31)) & 1u) == 0u) {
    const int n = a.counts[r];
    uint2* dst = a.list + static_cast<size_t>(r) * kp;
    const size_t base = static_cast<size_t>(r) * a.k;
    for (int e = 0; e < n; ++e) {
      const int j = a.indices[base + e];
      if ((a.upd_bits[j >> 5] >> (j & 31)) & 1u) continue;
      dst[cnt++] = make_uint2(__float_as_uint(__double2float_ru(a.hybrid[base + e])), static_cast<uint32_t>(j));
    }
    float th = theta_init;
    if (n == a.k) {
      const double kth = a.hybrid[base + a.k - 1];
      th = __double2float_rd(kth);
      if (static_cast<double>(th) >= kth) th = nextafterf(th, -INFINITY);
      th = fmaxf(th, theta_init);
      cut_h = kth;
      cut_j = a.indices[base + a.k - 1];
    }
    theta[r] = __float_as_uint(th);
  }
  a.cnt[r] = cnt;
  a.bound[r] = __int_as_float(0xff800000);
  a.cut_score[r] = cut_h;
  a.cut_index[r] = cut_j;
}

// Refresh: update_prev_kernel on the renumbered previous table T' with two bit sets.  A show outside G
// (remaining, not updated, its previous row names no removed show) gets T'_r without the shows of S as
// list 1, the threshold of its previous k-th entry and the rank cut there when the row was full.  A show
// in G gets an empty list 1 and no cut: the rows of A in T' name removed shows and are not read.
__global__ void refresh_prev_kernel(RefreshPrev a, unsigned int* theta, float theta_init, int n_shows, int kp) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_shows) return;
  int cnt = 0, cut_j = -1;
  double cut_h = 0.0;
  if (((a.g_bits[r >> 5] >> (r & 31)) & 1u) == 0u) {
    const int o = a.old_row[r];
    const int n = a.counts[o];
    uint2* dst = a.list + static_cast<size_t>(r) * kp;
    const size_t base = static_cast<size_t>(o) * a.k;
    for (int e = 0; e < n; ++e) {
      const int j = a.map[a.indices[base + e]];
      if ((a.s_bits[j >> 5] >> (j & 31)) & 1u) continue;
      dst[cnt++] = make_uint2(__float_as_uint(__double2float_ru(a.hybrid[base + e])), static_cast<uint32_t>(j));
    }
    float th = theta_init;
    if (n == a.k) {
      const double kth = a.hybrid[base + a.k - 1];
      th = __double2float_rd(kth);
      if (static_cast<double>(th) >= kth) th = nextafterf(th, -INFINITY);
      th = fmaxf(th, theta_init);
      cut_h = kth;
      cut_j = a.map[a.indices[base + a.k - 1]];
    }
    theta[r] = __float_as_uint(th);
  }
  a.cnt[r] = cnt;
  a.bound[r] = __int_as_float(0xff800000);
  a.cut_score[r] = cut_h;
  a.cut_index[r] = cut_j;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int get_encoder(EncodeTiledFn* fn) {
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  TVBF_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres));
  if (sym == nullptr || qres != cudaDriverEntryPointSuccess) {
    tvbf_set_error("cuTensorMapEncodeTiled is not available from this driver");
    return TVBF_ERR_CUDA;
  }
  *fn = reinterpret_cast<EncodeTiledFn>(sym);
  return TVBF_OK;
}

// 2-D map over the [n_pad, k_pad] 16-bit operand; box = 64 K-elements x box_rows, 128B swizzle.
static int make_operand_map(const tvbf_features* f, int box_rows, CUtensorMap* out) {
  EncodeTiledFn enc = nullptr;
  int rc = get_encoder(&enc);
  if (rc != TVBF_OK) return rc;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(f->k_pad), static_cast<cuuint64_t>(f->n_pad)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(f->k_pad) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMapDataType dt = f->text_dtype == TVBF_TEXT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                          : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = enc(out, dt, 2, const_cast<void*>(f->operand), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    tvbf_set_error("cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(r));
    return TVBF_ERR_CUDA;
  }
  return TVBF_OK;
}

int k1_deal_groups(int total_super_blocks, int r, int world, int rank, unsigned short* gid, int* local_sb) {
  // cost of group g = tiles on/above the diagonal of its super blocks; groups are visited in cost
  // order (ascending g) and each goes to the GPU with the least work so far (lowest rank on ties)
  const int groups = (total_super_blocks + r - 1) / r;
  long long load[64] = {0};
  int mine = 0, sbs = 0;
  if (world > 64) return -1;
  for (int g = 0; g < groups; ++g) {
    const int b = g * r, e = (b + r < total_super_blocks) ? b + r : total_super_blocks;
    long long cost = 0;
    for (int sb = b; sb < e; ++sb) cost += total_super_blocks - sb;
    int best = 0;
    for (int w = 1; w < world; ++w)
      if (load[w] < load[best]) best = w;
    load[best] += cost;
    if (best == rank) {
      if (mine >= kMaxDealGroups || g > 0xFFFF) return -1;
      gid[mine++] = static_cast<unsigned short>(g);
      sbs += e - b;
    }
  }
  *local_sb = sbs;
  return mine;
}

// Host copy of the kernel's work decomposition (tests check coverage without a GPU): item i ->
// {super block, split, tile0, tile1, real0, real1}; returns the number of items.
int k1_debug_schedule(const K1Params& p, int* out, int max_items) {
  const int n_items = ((p.rb_count + p.rb_per_group - 1) / p.rb_per_group) * p.rb_per_group * p.splits;
  for (int item = 0; item < n_items && item < max_items; ++item) {
    const ItemCoord c = item_coord(p, item);
    int* o = out + 6 * item;
    o[0] = c.sb; o[1] = c.split; o[2] = c.tile0; o[3] = c.tile1; o[4] = c.real0; o[5] = c.real1;
  }
  return n_items;
}

// Append sweep: old super blocks all cover the same narrow band [b0, col_tiles) (1 to ~20 tiles), new
// ones the rest of their row.  Items = (super block, column split), dealt round-robin to the clusters;
// the split count minimises the tiles of the busiest cluster (rounds of items x tiles per item), so
// that a band of a few tiles still spreads over every SM.  No pacing: nothing waits for anyone.
void k1_append_geometry(int n_old, int n_shows, int clusters, K1Params* p) {
  p->sym = 1;
  p->col_tiles = (n_shows + 255) / 256;
  p->rb_count = p->col_tiles;
  p->append_n_old = n_old;
  p->append_b0 = n_old / 256;
  p->deal_groups = 0;
  p->deal_r = 1;
  const int span = p->col_tiles - p->append_b0;
  if (clusters < 1) clusters = 1;
  long long best_cost = -1;
  for (int s = 1; s <= span && s <= 16 && s <= clusters; ++s) {
    int rb = clusters / s;
    if (rb > p->rb_count) rb = p->rb_count;
    const long long items = static_cast<long long>((p->rb_count + rb - 1) / rb) * rb * s;
    const long long cost = (items + clusters - 1) / clusters * ((span + s - 1) / s);
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      p->splits = s;
      p->rb_per_group = rb;
    }
  }
  p->tiles_per_split = (span + p->splits - 1) / p->splits;
}

int k1_debug_append_schedule(const K1Params& p, int* out, int max_items) {
  const int n_items = ((p.rb_count + p.rb_per_group - 1) / p.rb_per_group) * p.rb_per_group * p.splits;
  for (int item = 0; item < n_items && item < max_items; ++item) {
    const ItemCoord c = item_coord<true>(p, item);
    int* o = out + 6 * item;
    o[0] = c.sb; o[1] = c.split; o[2] = c.tile0; o[3] = c.tile1; o[4] = c.real0; o[5] = c.real1;
  }
  return n_items;
}

// Update sweep: a rectangle of ceil(q / 256) gathered super blocks x every column tile, on the one-sided
// schedule (p->sym = 0: no diagonal, split s of a super block walks tiles [s * tps, (s + 1) * tps)).
// Items = (super block, column split) dealt round-robin to the clusters; as for the append, the split
// count minimises the tiles of the busiest cluster, so that one or a few super blocks still spread
// over every SM.
void k1_update_geometry(int q, int n_shows, int clusters, K1Params* p) {
  p->sym = 0;
  p->col_tiles = (n_shows + 255) / 256;
  p->rb_count = (q + 255) / 256;
  p->deal_groups = 0;
  p->deal_r = 1;
  if (clusters < 1) clusters = 1;
  long long best_cost = -1;
  for (int s = 1; s <= p->col_tiles && s <= clusters; ++s) {
    int rb = clusters / s;
    if (rb > p->rb_count) rb = p->rb_count;
    const long long items = static_cast<long long>((p->rb_count + rb - 1) / rb) * rb * s;
    const long long cost = (items + clusters - 1) / clusters * ((p->col_tiles + s - 1) / s);
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      p->splits = s;
      p->rb_per_group = rb;
    }
  }
  p->tiles_per_split = (p->col_tiles + p->splits - 1) / p->splits;
}

int k1_entries_per_lane(int k) {
  if (k <= 48) return 4;
  if (k <= 160) return 8;
  if (k <= 400) return 16;
  return 0;
}

int k1_default_candidates(int k) {
  const int e = k1_entries_per_lane(k);
  const int cap = 32 * e;
  int kp = k <= 48 ? (k + 12 > 32 ? k + 12 : 32) : k + 28;
  kp = (kp + 7) & ~7;
  if (kp > cap - 64) kp = cap - 64;
  return kp;
}

int k1_choose_splits(int rb_count, int col_tiles, int sm_count) {
  // rb_count: super blocks (128*CG rows); sm_count: concurrently resident clusters.
  // Concurrently running clusters cover (R super blocks) x (S column splits): A rows are shared
  // S-way and B tiles R-way through L2, and the R A-blocks stay L2-resident across column tiles
  // when R is small.  Measured on C3: S = 4 is best (S = 2: +3 % K1 time and 1.8x the DRAM
  // traffic; S >= 6: same K1 time but the rescoring cost grows linearly with S).
  int best = 1;
  double best_score = -1.0;
  for (int s = 1; s <= 8; ++s) {
    if (s > 1 && col_tiles / s < 8) break;
    const int r = sm_count / s;
    if (r < 1) break;
    const int r_used = r < rb_count ? r : rb_count;
    const int groups = (rb_count + r_used - 1) / r_used;
    // fraction of cluster-slots doing useful work over the whole launch
    double score = static_cast<double>(rb_count) / (static_cast<double>(groups) * r_used) *
                   (static_cast<double>(r_used * s) / sm_count);
    if (s == 4) score += 0.03;
    else if (s == 3) score += 0.02;
    else if (s == 2) score += 0.01;
    else if (s >= 6) score -= 0.02;
    if (score > best_score + 1e-9) { best_score = score; best = s; }
  }
  return best;
}

// Profilers that serialise and replay kernels (Nsight Compute) make the driver fail a cooperative
// cluster launch outright -- the error is raised inside the profiler and ends the process before the
// runtime could report it to us.  Their injection library is visible in the process map, so K1 is
// launched plainly under them (the grid never exceeds one CTA per SM: co-resident on an idle device).
// TVBF_COOPERATIVE=0 / 1 overrides the detection.
static bool profiler_attached() {
  static const int cached = [] {
    if (const char* env = getenv("TVBF_COOPERATIVE")) return env[0] == '0' ? 1 : 0;
    if (getenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR") != nullptr) return 1;
    FILE* maps = fopen("/proc/self/maps", "r");
    if (maps == nullptr) return 0;
    char line[1024];
    int found = 0;
    while (!found && fgets(line, sizeof(line), maps) != nullptr)
      found = strstr(line, "nsight-compute") != nullptr || strstr(line, "libcuda-injection") != nullptr ||
              strstr(line, "libnvperf_host") != nullptr || strstr(line, "libInterceptorInjectionTarget") != nullptr;
    fclose(maps);
    return found;
  }();
  return cached != 0;
}

// fa: the features whose operand feeds the A (row) side, when not f's (the gathered rows of an update)
template <int E, bool kDump, int CG, int kMode, bool kWide = false, bool kG2 = false, bool kFold = false>
static int launch_k1(const tvbf_features* f, const K1Params& kp, int grid, cudaStream_t st,
                     const tvbf_features* fa = nullptr) {
  using L = Smem<CG, kWide>;
  CUtensorMap ta, tb;
  int rc = make_operand_map(fa != nullptr ? fa : f, BM, &ta);
  if (rc != TVBF_OK) return rc;
  rc = make_operand_map(f, static_cast<int>(L::B_ROWS), &tb);
  if (rc != TVBF_OK) return rc;
  auto kern = hybrid_topk_kernel<E, kDump, CG, kMode, kWide, kG2, kFold>;
  TVBF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(L::BYTES)));
  const uint32_t idesc = umma_idesc_f16(f->text_dtype == TVBF_TEXT_BF16 ? 1u : 0u, BM * CG, BN);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(Roles<(kMode != 0), kWide>::THREADS);
  cfg.dynamicSmemBytes = L::BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  // the pacing counter makes CTAs wait on one another: require co-residency of the whole grid
  attr[1].id = cudaLaunchAttributeCooperative;
  attr[1].val.cooperative = (kp.sync_kb > 0 && kp.cooperative) ? 1 : 0;
  if (attr[1].val.cooperative && profiler_attached()) {
    attr[1].val.cooperative = 0;
    tvbf_count_coop_fallback();
  }
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cudaError_t err = cudaLaunchKernelEx(&cfg, kern, ta, tb, kp, idesc);
  if (err != cudaSuccess && attr[1].val.cooperative) {
    // A profiler that patches the SASS (ncu's instruction-level passes) changes the kernel's
    // footprint and the runtime then refuses the cooperative launch.  The grid never exceeds one
    // CTA per SM, so on an otherwise idle device it is co-resident anyway: retry as a plain launch
    // (counted in tvbf_noncooperative_fallbacks; the pacing waits are bounded and trap, not hang).
    (void)cudaGetLastError();
    attr[1].val.cooperative = 0;
    err = cudaLaunchKernelEx(&cfg, kern, ta, tb, kp, idesc);
    if (err == cudaSuccess) tvbf_count_coop_fallback();
  }
  TVBF_CUDA_OK(err);
  tvbf_count_launch();
  return TVBF_OK;
}

// Parameters of the threshold seed pass of a symmetric job: a one-sided sweep over every
// tile_stride-th column tile that only writes g_theta (triple w of a weight sweep).
static K1Params make_seed_params(const K1Params& kp, int grid, int w) {
  K1Params seed = kp;
  seed.sym = 0;
  seed.seed_theta = 1;
  seed.splits = 1;
  seed.tiles_per_split = kp.col_tiles;
  seed.n_weights = 1;
  if (kp.n_weights > 1) {
    seed.w_text = kp.mw_text[w];
    seed.w_text_err = kp.mw_text_err[w];
    seed.w_genre = kp.mw_genre[w];
    seed.w_meta = kp.mw_meta[w];
    seed.eps = kp.mw_eps[w];
    seed.w_text_acc = kp.mw_text_acc[w];
    seed.eps_term = kp.mw_eps_term[w];
    seed.g_theta = kp.g_theta + static_cast<size_t>(w) * kp.n_pad;
    seed.score_hi = kp.mw_score_hi[w];
  }
  {
    // score histogram of the seed pass: 63 bins over [theta_init, score_hi)
    const float lo = kp.theta_init, span = seed.score_hi > lo ? seed.score_hi - lo : 1.0f;
    seed.hist_lo = lo;
    seed.hist_w = span / 63.0f;
    seed.hist_inv_w = 63.0f / span;
    seed.hist_off = 1.0f - lo * seed.hist_inv_w;
    const int max_stages = (kp.wide_epilogue ? Smem<2, true>::STAGES : Smem<2, false>::STAGES) - 2;
    if (seed.stages > max_stages) seed.stages = max_stages;   // the histogram lives in the last two A stages
  }
  if (kp.seed_world > 1)   // blocks seed_rank, seed_rank + seed_world, ... of the col_tiles super blocks
    seed.rb_count = kp.col_tiles > kp.seed_rank ? (kp.col_tiles - kp.seed_rank + kp.seed_world - 1) / kp.seed_world : 0;
  // all SMs, whatever the sweep's wave shape
  const int clusters = kp.seed_world > 1 ? kp.seed_clusters : grid / 2;
  seed.rb_per_group = clusters < seed.rb_count ? clusters : seed.rb_count;
  if (seed.rb_per_group < 1) seed.rb_per_group = 1;
  return seed;
}

static long long count_tiles(const K1Params& p) {
  const int n_items = ((p.rb_count + p.rb_per_group - 1) / p.rb_per_group) * p.rb_per_group * p.splits;
  long long t = 0;
  for (int item = 0; item < n_items; ++item) {
    const ItemCoord c = item_coord(p, item);
    if (c.sb < 0) continue;
    for (int jt = c.real0; jt < c.real1; jt += p.tile_stride) ++t;
  }
  return t;
}

// MMA tiles ((128 * cta_group) x 256 x k_pad each) one k1_launch of these parameters executes:
// out[0] threshold seed pass, out[1] main sweep.
void k1_executed_tiles(const K1Params& kp, int grid, long long* out) {
  out[0] = out[1] = 0;
  if (kp.sym) {
    const int nw = kp.n_weights > 1 ? kp.n_weights : 1;
    if (kp.sym_phase != 2 && kp.tile_stride > 1)
      for (int w = 0; w < nw; ++w) out[0] += count_tiles(make_seed_params(kp, grid, w));
    if (kp.sym_phase != 1) {
      K1Params sweep = kp;
      sweep.tile_stride = 1;
      out[1] = count_tiles(sweep);
    }
  } else {
    out[1] = count_tiles(kp);
  }
}

// The shared lists must read as zeros before the sweep (a reserved-but-unwritten entry counts as
// -inf); clearing them (820 MB at C3) is independent of the threshold seed pass that precedes the
// sweep, so it runs on a side stream beside it.  One side stream + event pair per device, created on
// first use; `pending` remembers a clear started by a seed-only call (multi-GPU: the caller's
// all-reduce sits between the two calls) for the sweep-only call that follows.
//
// A sweep-only call skips its own clear only when the pending clear covers exactly its lists and no
// other libtvbf call has enqueued work on the device since the seed-only call that started it: every
// such call is numbered per device (tvbf_enter_call), and the sweep must be the very next one.  Any
// other call first orders its stream after the pending clear and drops it -- an abandoned seed's clear
// can then neither be trusted by a later job nor race with the writes of one.
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  const void* pending = nullptr;          // g_list of the clear the last seed-only call started
  const void* pending_cnt = nullptr;      // ... its g_cnt
  size_t pending_bytes = 0;               // ... bytes of g_list cleared
  unsigned long long pending_call = 0;    // number of that seed-only call
  unsigned long long calls = 0;           // libtvbf calls that enqueued work on this device
};
static std::mutex g_side_mutex;
static SideStream g_side[64];

static int side_stream(SideStream** out) {
  int dev = 0;
  TVBF_CUDA_OK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) {
    tvbf_set_error("device ordinal %d out of range", dev);
    return TVBF_ERR_INVALID;
  }
  SideStream& s = g_side[dev];
  if (s.stream == nullptr) {
    TVBF_CUDA_OK(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    TVBF_CUDA_OK(cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming));
    TVBF_CUDA_OK(cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming));
  }
  *out = &s;
  return TVBF_OK;
}

// st waits for the pending clear, which is forgotten.  `always`: st waits for the side stream's last
// clear even when none is pending -- a sweep's own clear may have been absorbed by another call, on
// another stream.  Caller holds g_side_mutex.
static int absorb_pending(SideStream* s, cudaStream_t st, bool always) {
  if (s->pending == nullptr && !(always && s->join != nullptr)) return TVBF_OK;
  s->pending = nullptr;
  TVBF_CUDA_OK(cudaStreamWaitEvent(st, s->join, 0));
  return TVBF_OK;
}

}  // namespace tvbf

// The state of the current device, or nullptr without one.  Sets no error: without a device the
// call's own argument checks or its first CUDA call report what is wrong.
static tvbf::SideStream* current_side() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) {
    cudaGetLastError();
    return nullptr;
  }
  return &tvbf::g_side[dev];
}

int tvbf_enter_call(void* stream, int sym_sweep) {
  std::lock_guard<std::mutex> lock(tvbf::g_side_mutex);
  tvbf::SideStream* s = current_side();
  if (s == nullptr) return TVBF_OK;
  ++s->calls;
  // a sweep-only call decides in k1_launch, where it knows its lists
  return sym_sweep ? TVBF_OK : tvbf::absorb_pending(s, static_cast<cudaStream_t>(stream), false);
}

int tvbf_absorb_pending_clear(void* stream) {
  std::lock_guard<std::mutex> lock(tvbf::g_side_mutex);
  tvbf::SideStream* s = current_side();
  return s == nullptr ? TVBF_OK : tvbf::absorb_pending(s, static_cast<cudaStream_t>(stream), true);
}

namespace tvbf {

int k1_launch(const tvbf_features* f, const K1Params& kp, int entries_per_lane, int cta_group,
              int grid, cudaStream_t st) {
  if (kp.fold && (cta_group != 2 || entries_per_lane != 4 || kp.kp > 64 || kp.n_weights > 1)) {
    tvbf_set_error("an operand with folded genre / metadata columns supports CTA pairs and k <= 48 only");
    return TVBF_ERR_INVALID;
  }
  if (kp.sym) {
    if (cta_group != 2) {
      tvbf_set_error("symmetric mode needs cta_group 2");
      return TVBF_ERR_INVALID;
    }
    const int n_pad = f->n_pad;
    const int nw = kp.n_weights > 1 ? kp.n_weights : 1;   // weight sweep: nw * n_pad virtual shows
    const size_t n_virtual = static_cast<size_t>(nw) * n_pad;
    const size_t list_bytes = n_virtual * kp.sym_cap * 8;
    std::lock_guard<std::mutex> lock(g_side_mutex);
    SideStream* side = nullptr;
    int rcs = side_stream(&side);
    if (rcs != TVBF_OK) return rcs;
    bool cleared = false;
    if (kp.sym_phase != 2 && kp.tile_stride > 1) {
      // a seed pass follows: clear the lists beside it
      TVBF_CUDA_OK(cudaEventRecord(side->fork, st));
      TVBF_CUDA_OK(cudaStreamWaitEvent(side->stream, side->fork, 0));
      TVBF_CUDA_OK(cudaMemsetAsync(kp.g_cnt, 0, n_virtual * 4, side->stream));
      TVBF_CUDA_OK(cudaMemsetAsync(kp.g_list, 0, list_bytes, side->stream));
      TVBF_CUDA_OK(cudaEventRecord(side->join, side->stream));
      side->pending = kp.g_list;
      side->pending_cnt = kp.g_cnt;
      side->pending_bytes = list_bytes;
      side->pending_call = side->calls;
      cleared = true;
    }
    if (kp.sym_phase != 2) {
      sym_init_kernel<<<static_cast<unsigned>((n_virtual + 255) / 256), 256, 0, st>>>(
          kp.g_theta, f->n_shows, n_pad, static_cast<int>(n_virtual), kp.theta_init);
      TVBF_LAUNCH_OK("sym_init_kernel");
      if (kp.tile_stride > 1) {
        // seed pass: one-sided sweep over every tile_stride-th column tile, thresholds only
        // (once per triple of a weight sweep, into that triple's slice of g_theta)
        for (int w = 0; w < nw; ++w) {
          const K1Params seed = make_seed_params(kp, grid, w);
          int rc;
          // kMode 3: per-row score histograms instead of private candidate lists (P80k: 1.43 ms with
          // lists -- 4/5 of it selecting and compacting, with 4 epilogue warps -- against the sweep's 4.7)
          const int sg = seed.rb_per_group * 2;
          if (kp.wide_epilogue) {
            if (kp.fold) rc = launch_k1<4, false, 2, 3, true, false, true>(f, seed, sg, st);
            else if (kp.genre_hi != nullptr) rc = launch_k1<4, false, 2, 3, true, true>(f, seed, sg, st);
            else rc = launch_k1<4, false, 2, 3, true>(f, seed, sg, st);
          } else {
            if (kp.fold) rc = launch_k1<4, false, 2, 3, false, false, true>(f, seed, sg, st);
            else if (kp.genre_hi != nullptr) rc = launch_k1<4, false, 2, 3, false, true>(f, seed, sg, st);
            else rc = launch_k1<4, false, 2, 3>(f, seed, sg, st);
          }
          if (rc != TVBF_OK) return rc;
          TVBF_CUDA_OK(cudaMemsetAsync(kp.progress, 0, 256, st));
        }
      }
      if (kp.sym_phase == 1) return TVBF_OK;   // the sweep-only call joins the clear
    }
    // a sweep-only call right after the seed-only call that started the clear of these lists
    if (!cleared && kp.sym_phase == 2 && side->pending == kp.g_list && side->pending_cnt == kp.g_cnt &&
        side->pending_bytes == list_bytes && side->calls == side->pending_call + 1)
      cleared = true;
    if (cleared) {
      TVBF_CUDA_OK(cudaStreamWaitEvent(st, side->join, 0));
      side->pending = nullptr;
    } else {
      const int rca = absorb_pending(side, st, true);
      if (rca != TVBF_OK) return rca;
      TVBF_CUDA_OK(cudaMemsetAsync(kp.g_cnt, 0, n_virtual * 4, st));
      TVBF_CUDA_OK(cudaMemsetAsync(kp.g_list, 0, list_bytes, st));
    }
    K1Params sweep = kp;
    sweep.tile_stride = 1;
    if (nw > 1) {
      if (kp.genre_hi != nullptr) {
        tvbf_set_error("the shared weight sweep supports at most 64 genre columns");
        return TVBF_ERR_INVALID;
      }
      return launch_k1<4, false, 2, 5>(f, sweep, grid, st);
    }
    if (kp.wide_epilogue) {
      if (sweep.stages > Smem<2, true>::STAGES) sweep.stages = Smem<2, true>::STAGES;
      if (kp.fold) return launch_k1<4, false, 2, 1, true, false, true>(f, sweep, grid, st);
      return kp.genre_hi ? launch_k1<4, false, 2, 1, true, true>(f, sweep, grid, st)
                         : launch_k1<4, false, 2, 1, true>(f, sweep, grid, st);
    }
    if (kp.fold) return launch_k1<4, false, 2, 1, false, false, true>(f, sweep, grid, st);
    return kp.genre_hi ? launch_k1<4, false, 2, 1, false, true>(f, sweep, grid, st)
                       : launch_k1<4, false, 2, 1>(f, sweep, grid, st);
  }
  if (kp.fold) return launch_k1<4, false, 2, 0, false, false, true>(f, kp, grid, st);
  if (kp.genre_hi != nullptr) {
    if (cta_group != 2) {
      tvbf_set_error("two-word genre masks (G > 64) need cta_group 2");
      return TVBF_ERR_INVALID;
    }
    switch (entries_per_lane) {
      case 4: return launch_k1<4, false, 2, 0, false, true>(f, kp, grid, st);
      case 8: return launch_k1<8, false, 2, 0, false, true>(f, kp, grid, st);
      case 16: return launch_k1<16, false, 2, 0, false, true>(f, kp, grid, st);
      default: break;
    }
  } else if (cta_group == 2) {
    switch (entries_per_lane) {
      case 4: return launch_k1<4, false, 2, 0>(f, kp, grid, st);
      case 8: return launch_k1<8, false, 2, 0>(f, kp, grid, st);
      case 16: return launch_k1<16, false, 2, 0>(f, kp, grid, st);
      default: break;
    }
  } else {
    switch (entries_per_lane) {
      case 4: return launch_k1<4, false, 1, 0>(f, kp, grid, st);
      case 8: return launch_k1<8, false, 1, 0>(f, kp, grid, st);
      case 16: return launch_k1<16, false, 1, 0>(f, kp, grid, st);
      default: break;
    }
  }
  tvbf_set_error("unsupported candidate capacity (entries per lane %d)", entries_per_lane);
  return TVBF_ERR_INVALID;
}

// the same operands, tiles and epilogue width as the symmetric top-k sweep; no lists to clear, no seed
int k1_launch_pairs(const tvbf_features* f, const K1Params& kp, int grid, cudaStream_t st) {
  // a NULL pair buffer is fine at capacity 0: the kernel stores no slot >= pair_cap (count only)
  if (!kp.sym || (kp.pairs == nullptr && kp.pair_cap > 0) || kp.pair_count == nullptr || kp.pair_cap < 0) {
    tvbf_set_error("neighbour sweep: bad parameters");
    return TVBF_ERR_INVALID;
  }
  K1Params sweep = kp;
  sweep.tile_stride = 1;
  if (kp.wide_epilogue) {
    if (sweep.stages > Smem<2, true>::STAGES) sweep.stages = Smem<2, true>::STAGES;
    if (kp.fold) return launch_k1<4, false, 2, 11, true, false, true>(f, sweep, grid, st);
    return kp.genre_hi ? launch_k1<4, false, 2, 11, true, true>(f, sweep, grid, st)
                       : launch_k1<4, false, 2, 11, true>(f, sweep, grid, st);
  }
  if (kp.fold) return launch_k1<4, false, 2, 11, false, false, true>(f, sweep, grid, st);
  return kp.genre_hi ? launch_k1<4, false, 2, 11, false, true>(f, sweep, grid, st)
                     : launch_k1<4, false, 2, 11>(f, sweep, grid, st);
}

// histogram seed pass of an append: over the super blocks that hold new shows (from append_b0 on; the old
// shows among them are overwritten from the previous table afterwards)
static K1Params append_seed_params(const tvbf_features* f, const K1Params& kp, int grid) {
  K1Params seed = make_seed_params(kp, grid, 0);
  seed.row_begin = kp.append_b0 * 256;
  seed.rb_count = (f->n_shows - seed.row_begin + 255) / 256;
  seed.rb_per_group = grid / 2 < seed.rb_count ? grid / 2 : seed.rb_count;
  return seed;
}

void k1_append_executed_tiles(const tvbf_features* f, const K1Params& kp, int grid, long long* out) {
  out[0] = count_tiles(append_seed_params(f, kp, grid));
  K1Params sweep = kp;
  sweep.tile_stride = 1;
  long long t = 0;
  const int n_items = ((sweep.rb_count + sweep.rb_per_group - 1) / sweep.rb_per_group) * sweep.rb_per_group * sweep.splits;
  for (int item = 0; item < n_items; ++item) {
    const ItemCoord c = item_coord<true>(sweep, item);
    if (c.sb >= 0 && c.real1 > c.real0) t += c.real1 - c.real0;
  }
  out[1] = t;
}

int k1_launch_append(const tvbf_features* f, const K1Params& kp, int grid, const AppendPrev& prev,
                     cudaStream_t st) {
  if (!kp.sym || kp.n_weights > 1 || kp.sync_kb != 0) {
    tvbf_set_error("append sweep: bad parameters");
    return TVBF_ERR_INVALID;
  }
  const int n_pad = f->n_pad;
  const size_t list_bytes = static_cast<size_t>(n_pad) * kp.sym_cap * 8;
  std::lock_guard<std::mutex> lock(g_side_mutex);
  SideStream* side = nullptr;
  int rc = side_stream(&side);
  if (rc != TVBF_OK) return rc;
  // the shared lists are cleared on the side stream beside the seed pass, as in a full job
  rc = absorb_pending(side, st, true);
  if (rc != TVBF_OK) return rc;
  TVBF_CUDA_OK(cudaEventRecord(side->fork, st));
  TVBF_CUDA_OK(cudaStreamWaitEvent(side->stream, side->fork, 0));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.g_cnt, 0, static_cast<size_t>(n_pad) * 4, side->stream));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.g_list, 0, list_bytes, side->stream));
  TVBF_CUDA_OK(cudaEventRecord(side->join, side->stream));
  sym_init_kernel<<<static_cast<unsigned>((n_pad + 255) / 256), 256, 0, st>>>(kp.g_theta, f->n_shows, n_pad, n_pad,
                                                                               kp.theta_init);
  TVBF_LAUNCH_OK("sym_init_kernel");
  {
    const K1Params seed = append_seed_params(f, kp, grid);
    const int sg = seed.rb_per_group * 2;
    if (kp.wide_epilogue) {
      if (kp.fold) rc = launch_k1<4, false, 2, 3, true, false, true>(f, seed, sg, st);
      else if (kp.genre_hi != nullptr) rc = launch_k1<4, false, 2, 3, true, true>(f, seed, sg, st);
      else rc = launch_k1<4, false, 2, 3, true>(f, seed, sg, st);
    } else {
      if (kp.fold) rc = launch_k1<4, false, 2, 3, false, false, true>(f, seed, sg, st);
      else if (kp.genre_hi != nullptr) rc = launch_k1<4, false, 2, 3, false, true>(f, seed, sg, st);
      else rc = launch_k1<4, false, 2, 3>(f, seed, sg, st);
    }
    if (rc != TVBF_OK) return rc;
  }
  append_prev_kernel<<<static_cast<unsigned>((f->n_shows + 255) / 256), 256, 0, st>>>(prev, kp.g_theta, kp.theta_init,
                                                                                      f->n_shows, kp.kp);
  TVBF_LAUNCH_OK("append_prev_kernel");
  TVBF_CUDA_OK(cudaStreamWaitEvent(st, side->join, 0));
  K1Params sweep = kp;
  sweep.tile_stride = 1;
  if (kp.wide_epilogue) {
    if (sweep.stages > Smem<2, true>::STAGES) sweep.stages = Smem<2, true>::STAGES;
    if (kp.fold) return launch_k1<4, false, 2, 6, true, false, true>(f, sweep, grid, st);
    return kp.genre_hi ? launch_k1<4, false, 2, 6, true, true>(f, sweep, grid, st)
                       : launch_k1<4, false, 2, 6, true>(f, sweep, grid, st);
  }
  if (kp.fold) return launch_k1<4, false, 2, 6, false, false, true>(f, sweep, grid, st);
  return kp.genre_hi ? launch_k1<4, false, 2, 6, false, true>(f, sweep, grid, st)
                     : launch_k1<4, false, 2, 6>(f, sweep, grid, st);
}

// histogram seed pass of an update: the gathered rows against every tile_stride-th column tile
static K1Params update_seed_params(const K1Params& kp, int grid) {
  K1Params seed = make_seed_params(kp, grid, 0);
  seed.row_begin = 0;
  return seed;
}

void k1_update_executed_tiles(const K1Params& kp, int grid, long long* out) {
  out[0] = count_tiles(update_seed_params(kp, grid));
  K1Params sweep = kp;
  sweep.tile_stride = 1;
  out[1] = count_tiles(sweep);
}

int k1_launch_update(const tvbf_features* f, const tvbf_features* g, const K1Params& kp, int grid,
                     const UpdatePrev& prev, cudaStream_t st) {
  if (kp.sym || kp.n_weights > 1 || kp.sync_kb != 0 || kp.wide_epilogue || kp.upd_q < 1 || kp.upd_rows == nullptr ||
      kp.upd_bits == nullptr) {
    tvbf_set_error("update sweep: bad parameters");
    return TVBF_ERR_INVALID;
  }
  const int n_pad = f->n_pad;
  const size_t list_bytes = static_cast<size_t>(n_pad) * kp.sym_cap * 8;
  std::lock_guard<std::mutex> lock(g_side_mutex);
  SideStream* side = nullptr;
  int rc = side_stream(&side);
  if (rc != TVBF_OK) return rc;
  // the shared lists are cleared on the side stream beside the seed pass, as in a full job
  rc = absorb_pending(side, st, true);
  if (rc != TVBF_OK) return rc;
  TVBF_CUDA_OK(cudaEventRecord(side->fork, st));
  TVBF_CUDA_OK(cudaStreamWaitEvent(side->stream, side->fork, 0));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.g_cnt, 0, static_cast<size_t>(n_pad) * 4, side->stream));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.g_list, 0, list_bytes, side->stream));
  TVBF_CUDA_OK(cudaEventRecord(side->join, side->stream));
  sym_init_kernel<<<static_cast<unsigned>((n_pad + 255) / 256), 256, 0, st>>>(kp.g_theta, f->n_shows, n_pad, n_pad,
                                                                               kp.theta_init);
  TVBF_LAUNCH_OK("sym_init_kernel");
  update_prev_kernel<<<static_cast<unsigned>((f->n_shows + 255) / 256), 256, 0, st>>>(prev, kp.g_theta, kp.theta_init,
                                                                                      f->n_shows, kp.kp);
  TVBF_LAUNCH_OK("update_prev_kernel");
  {
    const K1Params seed = update_seed_params(kp, grid);
    const int sg = seed.rb_per_group * 2;
    if (kp.fold) rc = launch_k1<4, false, 2, 8, false, false, true>(f, seed, sg, st, g);
    else if (kp.genre_hi != nullptr) rc = launch_k1<4, false, 2, 8, false, true>(f, seed, sg, st, g);
    else rc = launch_k1<4, false, 2, 8>(f, seed, sg, st, g);
    if (rc != TVBF_OK) return rc;
  }
  TVBF_CUDA_OK(cudaStreamWaitEvent(st, side->join, 0));
  K1Params sweep = kp;
  sweep.tile_stride = 1;
  if (kp.fold) return launch_k1<4, false, 2, 7, false, false, true>(f, sweep, grid, st, g);
  return kp.genre_hi ? launch_k1<4, false, 2, 7, false, true>(f, sweep, grid, st, g)
                     : launch_k1<4, false, 2, 7>(f, sweep, grid, st, g);
}

// Removal: the gathered rows' thresholds move from their shows' slots (where the seed pass over the
// gathered rows wrote them) to the gathered-row slots the repair sweep and K4s index; +inf for the
// padding rows
__global__ void remove_theta_kernel(const unsigned int* theta, const int* rows, int q, int q_pad,
                                    unsigned int* gtheta) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < q_pad) gtheta[e] = e < q ? theta[rows[e]] : 0x7f800000u;
}

int k1_launch_remove(const tvbf_features* f, const tvbf_features* g, const K1Params& kp, int grid,
                     unsigned int* gtheta, cudaStream_t st) {
  if (kp.sym || kp.n_weights > 1 || kp.sync_kb != 0 || kp.wide_epilogue || kp.upd_q < 1 || kp.upd_rows == nullptr ||
      gtheta == nullptr) {
    tvbf_set_error("repair sweep: bad parameters");
    return TVBF_ERR_INVALID;
  }
  const int q_pad = kp.rb_count * 256;   // gathered rows, each with a list of its own
  const size_t list_bytes = static_cast<size_t>(q_pad) * kp.sym_cap * 8;
  std::lock_guard<std::mutex> lock(g_side_mutex);
  SideStream* side = nullptr;
  int rc = side_stream(&side);
  if (rc != TVBF_OK) return rc;
  // only the gathered rows' lists are cleared, on the side stream beside the seed pass
  rc = absorb_pending(side, st, true);
  if (rc != TVBF_OK) return rc;
  TVBF_CUDA_OK(cudaEventRecord(side->fork, st));
  TVBF_CUDA_OK(cudaStreamWaitEvent(side->stream, side->fork, 0));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.g_cnt, 0, static_cast<size_t>(q_pad) * 4, side->stream));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.g_list, 0, list_bytes, side->stream));
  TVBF_CUDA_OK(cudaEventRecord(side->join, side->stream));
  const int n_pad = f->n_pad;
  sym_init_kernel<<<static_cast<unsigned>((n_pad + 255) / 256), 256, 0, st>>>(kp.g_theta, f->n_shows, n_pad, n_pad,
                                                                               kp.theta_init);
  TVBF_LAUNCH_OK("sym_init_kernel");
  {
    const K1Params seed = update_seed_params(kp, grid);
    const int sg = seed.rb_per_group * 2;
    if (kp.fold) rc = launch_k1<4, false, 2, 8, false, false, true>(f, seed, sg, st, g);
    else if (kp.genre_hi != nullptr) rc = launch_k1<4, false, 2, 8, false, true>(f, seed, sg, st, g);
    else rc = launch_k1<4, false, 2, 8>(f, seed, sg, st, g);
    if (rc != TVBF_OK) return rc;
  }
  remove_theta_kernel<<<static_cast<unsigned>((q_pad + 255) / 256), 256, 0, st>>>(kp.g_theta, kp.upd_rows, kp.upd_q,
                                                                                   q_pad, gtheta);
  TVBF_LAUNCH_OK("remove_theta_kernel");
  TVBF_CUDA_OK(cudaStreamWaitEvent(st, side->join, 0));
  K1Params sweep = kp;
  sweep.tile_stride = 1;
  sweep.g_theta = gtheta;
  if (kp.fold) return launch_k1<4, false, 2, 9, false, false, true>(f, sweep, grid, st, g);
  return kp.genre_hi ? launch_k1<4, false, 2, 9, false, true>(f, sweep, grid, st, g)
                     : launch_k1<4, false, 2, 9>(f, sweep, grid, st, g);
}

// Refresh: as k1_launch_update, with the lists of the renumbered previous table and the refresh sweep
int k1_launch_refresh(const tvbf_features* f, const tvbf_features* g, const K1Params& kp, int grid,
                      const RefreshPrev& prev, cudaStream_t st) {
  if (kp.sym || kp.n_weights > 1 || kp.sync_kb != 0 || kp.wide_epilogue || kp.upd_q < 1 || kp.upd_rows == nullptr ||
      kp.upd_bits == nullptr || kp.upd_sbits == nullptr) {
    tvbf_set_error("refresh sweep: bad parameters");
    return TVBF_ERR_INVALID;
  }
  const int n_pad = f->n_pad;
  const size_t list_bytes = static_cast<size_t>(n_pad) * kp.sym_cap * 8;
  std::lock_guard<std::mutex> lock(g_side_mutex);
  SideStream* side = nullptr;
  int rc = side_stream(&side);
  if (rc != TVBF_OK) return rc;
  // the shared lists are cleared on the side stream beside the seed pass, as in an update
  rc = absorb_pending(side, st, true);
  if (rc != TVBF_OK) return rc;
  TVBF_CUDA_OK(cudaEventRecord(side->fork, st));
  TVBF_CUDA_OK(cudaStreamWaitEvent(side->stream, side->fork, 0));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.g_cnt, 0, static_cast<size_t>(n_pad) * 4, side->stream));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.g_list, 0, list_bytes, side->stream));
  TVBF_CUDA_OK(cudaEventRecord(side->join, side->stream));
  sym_init_kernel<<<static_cast<unsigned>((n_pad + 255) / 256), 256, 0, st>>>(kp.g_theta, f->n_shows, n_pad, n_pad,
                                                                               kp.theta_init);
  TVBF_LAUNCH_OK("sym_init_kernel");
  refresh_prev_kernel<<<static_cast<unsigned>((f->n_shows + 255) / 256), 256, 0, st>>>(prev, kp.g_theta,
                                                                                       kp.theta_init, f->n_shows, kp.kp);
  TVBF_LAUNCH_OK("refresh_prev_kernel");
  {
    const K1Params seed = update_seed_params(kp, grid);
    const int sg = seed.rb_per_group * 2;
    if (kp.fold) rc = launch_k1<4, false, 2, 8, false, false, true>(f, seed, sg, st, g);
    else if (kp.genre_hi != nullptr) rc = launch_k1<4, false, 2, 8, false, true>(f, seed, sg, st, g);
    else rc = launch_k1<4, false, 2, 8>(f, seed, sg, st, g);
    if (rc != TVBF_OK) return rc;
  }
  TVBF_CUDA_OK(cudaStreamWaitEvent(st, side->join, 0));
  K1Params sweep = kp;
  sweep.tile_stride = 1;
  if (kp.fold) return launch_k1<4, false, 2, 10, false, false, true>(f, sweep, grid, st, g);
  return kp.genre_hi ? launch_k1<4, false, 2, 10, false, true>(f, sweep, grid, st, g)
                     : launch_k1<4, false, 2, 10>(f, sweep, grid, st, g);
}

int k1_launch_dump(const tvbf_features* f, const K1Params& kp, int cta_group, cudaStream_t st) {
  return cta_group == 2 ? launch_k1<4, true, 2, 0>(f, kp, 2, st)
                        : launch_k1<4, true, 1, 0>(f, kp, 1, st);
}

int k1_launch_stats(const tvbf_features* f, const K1Params& kp, int grid, cudaStream_t st) {
  return launch_k1<4, false, 2, 2>(f, kp, grid, st);
}

int k4s_launch(const K1Params& kp, int n_rows, cudaStream_t st) {
  sym_compact_kernel<<<(n_rows + 3) / 4, 128, 0, st>>>(kp, n_rows);
  TVBF_LAUNCH_OK("sym_compact_kernel");
  return TVBF_OK;
}

}  // namespace tvbf
