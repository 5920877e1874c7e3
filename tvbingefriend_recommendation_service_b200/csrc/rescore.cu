// K5 + K6 -- exact fp64 scoring.
//
// K5 (rescore_kernel): recomputes every candidate pair the tensor-core pass kept, in float64 from
// the normalised inputs and with the reference's operation order
//   hybrid = genre_weight * genre + text_weight * text + metadata_weight * metadata
// (scripts/populate_database.py:187-192), applies the reference's selection rule -- skip self,
// drop score < min_similarity, keep top_n (populate_database.py:195-218) -- with the stated
// tie-break (score descending, column index ascending), and CERTIFIES the row: every column the
// candidate pass dropped has upper bound U <= theta, so the row is final iff theta < the k-th
// exact score (or < min_similarity when fewer than k qualify).  Rows that cannot be certified
// (tie plateaus wider than the candidate list, near-ties below the fp16 bound) go to K6.
//
// K6 (exact_rows_kernel): scores ONE source row against all N columns in fp64 and selects the
// exact top-k with a radix select over order-preserving 64-bit keys; also the engine behind the
// single-show query of services/content_based_service.py:161-236 for arbitrary n.
#include "internal.cuh"

namespace tvbf {


__device__ __forceinline__ double text_dot(const tvbf_features& f, int i, int j) {
  const int64_t bi = f.text_indptr[i], ei = f.text_indptr[i + 1];
  const int64_t bj = f.text_indptr[j], ej = f.text_indptr[j + 1];
  if (bi == ei || bj == ej) return 0.0;
  int64_t a = bi, b = bj;
  int ca = f.text_indices[a], cb = f.text_indices[b];
  double s = 0.0;
  while (true) {
    if (ca == cb) {
      s = __dadd_rn(s, __dmul_rn(f.text_values[a], f.text_values[b]));
      ++a; ++b;
      if (a >= ei || b >= ej) break;
      ca = f.text_indices[a];
      cb = f.text_indices[b];
    } else if (ca < cb) {
      if (++a >= ei) break;
      ca = f.text_indices[a];
    } else {
      if (++b >= ej) break;
      cb = f.text_indices[b];
    }
  }
  return s;
}

__device__ __forceinline__ double dense_dot(const double* x, int dim, int i, int j) {
  const double* a = x + static_cast<size_t>(i) * dim;
  const double* b = x + static_cast<size_t>(j) * dim;
  double s = 0.0;
  for (int c = 0; c < dim; ++c) s = __dadd_rn(s, __dmul_rn(a[c], b[c]));
  return s;
}

__device__ __forceinline__ double genre_score(const tvbf_features& f, int i, int j) {
  if (f.genre_mode == TVBF_GROUP_PACKED) {
    const TvbfColSide* cs = static_cast<const TvbfColSide*>(f.col_side);
    const unsigned long long bi = cs[i].genre_bits, bj = cs[j].genre_bits;
    int ni = __popcll(bi), nj = __popcll(bj), c = __popcll(bi & bj);
    if (f.genre_hi != nullptr) {   // 64 < G <= 128: second word
      const unsigned long long hi = f.genre_hi[i], hj = f.genre_hi[j];
      ni += __popcll(hi);
      nj += __popcll(hj);
      c += __popcll(hi & hj);
    }
    if (ni == 0 || nj == 0) return 0.0;
    return static_cast<double>(c) * ((1.0 / sqrt(static_cast<double>(ni))) *
                                     (1.0 / sqrt(static_cast<double>(nj))));
  }
  if (f.genre_mode == TVBF_GROUP_FOLDED) return dense_dot(f.genre_dense, f.genre_dim, i, j);
  return 0.0;
}

__device__ __forceinline__ double meta_score(const tvbf_features& f, int i, int j) {
  if (f.meta_mode == TVBF_GROUP_PACKED) {
    const TvbfColSide* cs = static_cast<const TvbfColSide*>(f.col_side);
    const uint32_t a = cs[i].meta_bits, b = cs[j].meta_bits;
    const int eq = __popc(a & b);  // groups (platform, type, language) with the same category
    if (f.meta_kind == TVBF_META_MEAN3) return static_cast<double>(eq) / 3.0;
    const int ni = __popc(a), nj = __popc(b);
    if (ni == 0 || nj == 0) return 0.0;
    return static_cast<double>(eq) * ((1.0 / sqrt(static_cast<double>(ni))) *
                                      (1.0 / sqrt(static_cast<double>(nj))));
  }
  if (f.meta_mode == TVBF_GROUP_FOLDED) {
    if (f.meta_kind == TVBF_META_MEAN3) {
      const double p = dense_dot(f.meta_dense[0], f.meta_dims[0], i, j);
      const double t = dense_dot(f.meta_dense[1], f.meta_dims[1], i, j);
      const double l = dense_dot(f.meta_dense[2], f.meta_dims[2], i, j);
      return (p + t + l) / 3;
    }
    return dense_dot(f.meta_dense[0], f.meta_dims[0], i, j);
  }
  return 0.0;
}

struct Scores {
  double h, g, t, m;
};

__device__ __forceinline__ Scores score_pair(const ScoreParams& sp, int i, int j) {
  Scores s;
  s.g = genre_score(sp.f, i, j);
  s.t = text_dot(sp.f, i, j);
  s.m = meta_score(sp.f, i, j);
  s.h = hybrid_rn(sp.wg, s.g, sp.wt, s.t, sp.wm, s.m);
  return s;
}

// (score desc, column asc) strict "a ranks before b"
__device__ __forceinline__ bool ranks_before(double ha, int ja, double hb, int jb) {
  return ha > hb || (ha == hb && ja < jb);
}

// ---------------------------------------------------------------------------------------------
// K5: one warp per source row
// ---------------------------------------------------------------------------------------------
constexpr int K5_WARPS = 4;

// the work of one warp on table row r (source row row_begin + r); n_rows sizes the flagged lists.
// kCut (update): a row with cut_index[r] >= 0 must also rank its k-th entry at or above
// (cut_score[r], cut_index[r]) to be final.
template <bool kCut = false>
__device__ __forceinline__ void rescore_row(const ScoreParams& sp, const uint2* __restrict__ cand,
                                            const int* __restrict__ cand_cnt, const float* __restrict__ cand_theta,
                                            int splits, const CandLayout& lay, int kp, int row_begin, int n_rows,
                                            const tvbf_topk_out& out, int* flagged_rows, double* flagged_floor,
                                            int max_cand, int keep, int warp, int lane, int r,
                                            const double* cut_score = nullptr, const int* cut_index = nullptr) {
  extern __shared__ __align__(16) uint8_t k5_smem[];
  const int i = row_begin + r;
  uint8_t* base = k5_smem + static_cast<size_t>(warp) * max_cand * 48;
  double* sh = reinterpret_cast<double*>(base);
  double* sg = sh + max_cand;
  double* st = sg + max_cand;
  double* sm = st + max_cand;
  int* sj = reinterpret_cast<int*>(sm + max_cand);
  uint32_t* su = reinterpret_cast<uint32_t*>(sj + max_cand);
  __shared__ double s_kth[K5_WARPS];

  // gather the candidate columns (and their upper bounds U) of all lists
  int total = 0;
  float theta = __int_as_float(0xff800000);
  for (int s = 0; s < splits; ++s) {
    const size_t slot = static_cast<size_t>(lay.slot_base + r * lay.row_stride + s * lay.list_stride);
    const uint2* list = cand + slot * (lay.packed ? kp + 1 : kp);
    int n;
    if (lay.packed) {
      const uint2 tail = list[kp];
      n = static_cast<int>(tail.x);
      theta = fmaxf(theta, __uint_as_float(tail.y));
    } else {
      n = cand_cnt[slot];
      theta = fmaxf(theta, cand_theta[slot]);
    }
    for (int e = lane; e < n; e += 32) {
      const uint2 c = list[e];
      su[total + e] = c.x;
      sj[total + e] = static_cast<int>(c.y);
    }
    total += n;
  }
  __syncwarp();
  // Several lists (column splits, or the partial lists of several GPUs): only the `keep` largest
  // upper bounds are worth an exact score -- what a single merged list would have kept.  Everything
  // cut here has exact score <= U <= the keep-th largest U, which joins the row's bound theta.
  // (selection on the order-preserving integer image of U: the one-sided sweep admits negative
  // weights and thresholds, so U may be negative.)
  if (total > keep) {
    uint32_t best = 0u;
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t t = best | (1u << bit);
      int c = 0;
      for (int e = lane; e < total; e += 32) c += (f32_orderable(__uint_as_float(su[e])) >= t);
      c = __reduce_add_sync(kFullMask, c);
      if (c >= keep) best = t;
    }
    int above = 0;
    for (int e = lane; e < total; e += 32) above += (f32_orderable(__uint_as_float(su[e])) > best);
    above = __reduce_add_sync(kFullMask, above);
    const int quota = keep - above;   // entries equal to the keep-th value that still fit
    int out_n = 0, eq_seen = 0;
    for (int c0 = 0; c0 < total; c0 += 32) {   // ordered in-place compaction (writes trail reads)
      const int e = c0 + lane;
      const uint32_t u = e < total ? su[e] : 0u;
      const uint32_t uo = f32_orderable(__uint_as_float(u));
      const int j = e < total ? sj[e] : 0;
      const unsigned lt = (1u << lane) - 1u;
      const unsigned bal_eq = __ballot_sync(kFullMask, e < total && uo == best);
      const bool take = e < total && (uo > best || (uo == best && eq_seen + __popc(bal_eq & lt) < quota));
      const unsigned bal = __ballot_sync(kFullMask, take);
      if (take) {
        su[out_n + __popc(bal & lt)] = u;
        sj[out_n + __popc(bal & lt)] = j;
      }
      out_n += __popc(bal);
      eq_seen += __popc(bal_eq);
      __syncwarp();
    }
    total = out_n;
    theta = fmaxf(theta, f32_from_orderable(best));
    __syncwarp();
  }
  // exact scores
  int valid = 0;
  for (int e = lane; e < total; e += 32) {
    const int j = sj[e];
    const Scores s = score_pair(sp, i, j);
    const bool ok = (s.h >= sp.min_similarity) && !(sp.exclude_self && j == i);
    sh[e] = ok ? s.h : -INFINITY;
    sg[e] = s.g;
    st[e] = s.t;
    sm[e] = s.m;
    valid += ok;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) valid += __shfl_xor_sync(kFullMask, valid, o);
  __syncwarp();
  const int k = sp.k;
  const int count = valid < k ? valid : k;
  if (lane == 0) s_kth[warp] = sp.min_similarity;
  __syncwarp();
  // rank by counting: position = number of entries that rank before this one
  const size_t obase = static_cast<size_t>(r) * k;
  for (int e = lane; e < total; e += 32) {
    const double he = sh[e];
    if (he == -INFINITY) continue;
    const int je = sj[e];
    int rank = 0;
    for (int o = 0; o < total; ++o) rank += ranks_before(sh[o], sj[o], he, je);
    if (rank < k) {
      out.indices[obase + rank] = je;
      out.hybrid[obase + rank] = he;
      out.genre[obase + rank] = sg[e];
      out.text[obase + rank] = st[e];
      out.metadata[obase + rank] = sm[e];
      if (rank == k - 1) s_kth[warp] = he;
    }
  }
  for (int e = count + lane; e < k; e += 32) {
    out.indices[obase + e] = -1;
    out.hybrid[obase + e] = NAN;
    out.genre[obase + e] = NAN;
    out.text[obase + e] = NAN;
    out.metadata[obase + e] = NAN;
  }
  __syncwarp();
  if (lane == 0) {
    out.counts[r] = count;
    atomicAdd(&out.stats[1], total);
    // certificate: all dropped columns have exact score <= U <= theta
    const double bound = s_kth[warp];  // k-th exact score, or min_similarity if fewer than k
    bool safe = static_cast<double>(theta) < bound;
    if constexpr (kCut) {
      // the columns list 1 left out rank below the previous k-th entry: the row is final only if its
      // k-th entry ranks at or above that (a short row does not)
      const int cj = cut_index[r];
      if (cj >= 0) {
        const double cs = cut_score[r];
        const int jk = out.indices[obase + k - 1];
        safe = safe && count == k && (bound > cs || (bound == cs && jk <= cj));
      }
    }
    if (!safe) {
      atomicAdd(&out.stats[0], 1);
      // shows with text are listed from the front, shows without (the usual tie plateaus, which
      // never need the text CSR) from the back: the exact kernel handles the two kinds separately
      const bool has_text = sp.f.text_indptr[i + 1] > sp.f.text_indptr[i];
      const int pos = has_text ? atomicAdd(&out.stats[2], 1) : n_rows - 1 - atomicAdd(&out.stats[3], 1);
      flagged_rows[pos] = r;
      // the k-th best exact score among the candidates is a lower bound of the true k-th best:
      // the exact kernel only needs to keep columns that reach it
      flagged_floor[pos] = bound;
    }
  }
}

__global__ void __launch_bounds__(K5_WARPS * 32)
rescore_kernel(const ScoreParams sp, const uint2* __restrict__ cand,
               const int* __restrict__ cand_cnt, const float* __restrict__ cand_theta, int splits,
               const CandLayout lay, int kp, int row_begin, int n_rows, tvbf_topk_out out,
               int* flagged_rows, double* flagged_floor, int max_cand, int keep) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + warp;
  if (r >= n_rows) return;
  rescore_row(sp, cand, cand_cnt, cand_theta, splits, lay, kp, row_begin, n_rows, out, flagged_rows, flagged_floor,
              max_cand, keep, warp, lane, r);
}

// K5 over the listed table rows only (rows[0 .. *n_listed)): an append rescores the new shows and the old
// shows that received new candidates; the others keep their previous rows
__global__ void __launch_bounds__(K5_WARPS * 32)
rescore_listed_kernel(const ScoreParams sp, const uint2* __restrict__ cand,
                      const int* __restrict__ cand_cnt, const float* __restrict__ cand_theta, int splits,
                      const CandLayout lay, int kp, int row_begin, int n_rows, const int* __restrict__ rows,
                      const int* __restrict__ n_listed, tvbf_topk_out out, int* flagged_rows, double* flagged_floor,
                      int max_cand, int keep) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * (blockDim.x >> 5) + warp;
  if (e >= *n_listed) return;
  rescore_row(sp, cand, cand_cnt, cand_theta, splits, lay, kp, row_begin, n_rows, out, flagged_rows, flagged_floor,
              max_cand, keep, warp, lane, rows[e]);
}

// ... where the lists of rows[e] are at row position e (the gathered rows of a removal)
__global__ void __launch_bounds__(K5_WARPS * 32)
rescore_gathered_kernel(const ScoreParams sp, const uint2* __restrict__ cand,
                        const int* __restrict__ cand_cnt, const float* __restrict__ cand_theta, int splits,
                        const CandLayout lay, int kp, int row_begin, int n_rows, const int* __restrict__ rows,
                        const int* __restrict__ n_listed, tvbf_topk_out out, int* flagged_rows, double* flagged_floor,
                        int max_cand, int keep) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * (blockDim.x >> 5) + warp;
  if (e >= *n_listed) return;
  const int r = rows[e];
  CandLayout at = lay;
  at.slot_base += static_cast<long long>(e) - static_cast<long long>(r) * lay.row_stride;   // slot of row r: e
  rescore_row(sp, cand, cand_cnt, cand_theta, splits, at, kp, row_begin, n_rows, out, flagged_rows, flagged_floor,
              max_cand, keep, warp, lane, r);
}

// ... with the rank cut of an update (rescore_row<true>)
__global__ void __launch_bounds__(K5_WARPS * 32)
rescore_cut_kernel(const ScoreParams sp, const uint2* __restrict__ cand,
                   const int* __restrict__ cand_cnt, const float* __restrict__ cand_theta, int splits,
                   const CandLayout lay, int kp, int row_begin, int n_rows, const int* __restrict__ rows,
                   const int* __restrict__ n_listed, tvbf_topk_out out, int* flagged_rows, double* flagged_floor,
                   int max_cand, int keep, const double* __restrict__ cut_score, const int* __restrict__ cut_index) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * (blockDim.x >> 5) + warp;
  if (e >= *n_listed) return;
  rescore_row<true>(sp, cand, cand_cnt, cand_theta, splits, lay, kp, row_begin, n_rows, out, flagged_rows,
                    flagged_floor, max_cand, keep, warp, lane, rows[e], cut_score, cut_index);
}

// ---------------------------------------------------------------------------------------------
// K6: exact row kernel -- one CTA per listed source row, persistent over the list
// ---------------------------------------------------------------------------------------------
constexpr int K6_THREADS = 512;
constexpr int K6_MAXK = 1024;

__device__ __forceinline__ unsigned long long f64_orderable(double d) {
  unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(d));
  return b ^ ((b >> 63) ? 0xFFFFFFFFFFFFFFFFull : 0x8000000000000000ull);
}
__device__ __forceinline__ double f64_from_orderable(unsigned long long u) {
  unsigned long long b = u ^ ((u >> 63) ? 0x8000000000000000ull : 0xFFFFFFFFFFFFFFFFull);
  return __longlong_as_double(static_cast<long long>(b));
}

// rows: shard-local row numbers when `rows_are_local`, else absolute source rows.
// count_ptr (device) overrides n_listed when non-null (flagged rows of K5).
struct FeatureScorer {
  ScoreParams sp;
  __device__ __forceinline__ Scores operator()(int i, int j) const { return score_pair(sp, i, j); }
};
// variant C: rows of precomputed N x N matrices (services/content_based_service.py:206-231)
struct MatrixScorer {
  const double* h;
  const double* g;
  const double* t;
  const double* m;
  int n;
  __device__ __forceinline__ Scores operator()(int i, int j) const {
    const size_t e = static_cast<size_t>(i) * n + j;
    Scores s;
    s.h = h[e]; s.g = g[e]; s.t = t[e]; s.m = m[e];
    return s;
  }
};

struct SelectParams {
  int n;
  int k;
  int exclude_self;
  double min_similarity;
};

// block-wide selection state (static shared memory)
struct SelectSmem {
  unsigned int hist[256];
  unsigned long long prefix;
  int rank, valid, above, taken;
  int warp_tot[32];
  unsigned long long win_key[K6_MAXK];
  int win_j[K6_MAXK];
};

// Exact top-k of one source row from its N order-preserving keys (0 = invalid): radix select of the
// count-th largest key, everything above it, then the LOWEST column indices among keys equal to
// it, finally ordered by (score desc, column asc).  Called by all threads of the block.
// `keys` has n entries; entry e is column jmap[e] (or e when jmap is null).  kOrdered: the entries
// are in ascending column order, so the tie group is cut by position; otherwise (survivor lists
// appended in arbitrary order) by a second radix select over the column numbers.
// kCg: the arrays were written by other CTAs of this launch -> read them through L2 (ld.cg).
template <bool kOrdered, bool kCg, class Scorer>
__device__ void select_and_emit(SelectSmem& sm, const unsigned long long* keys, const int* jmap, int n,
                                int k, int valid, int i, size_t orow, const Scorer& scorer,
                                const tvbf_topk_out& out) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
  auto ldk = [](const unsigned long long* p) {
    if constexpr (kCg) return __ldcg(p); else return *p;
  };
  auto ldj = [](const int* p) {
    if constexpr (kCg) return __ldcg(p); else return *p;
  };
  const int count = valid < k ? valid : k;
  const size_t obase = orow * static_cast<size_t>(k);
  __syncthreads();
  if (!kOrdered && n <= nthr) {
    // short survivor list: every thread ranks one entry against all others, no selection passes
    if (tid < n) {
      const unsigned long long ke = ldk(keys + tid);
      const int je = ldj(jmap + tid);
      int rank = 0;
      for (int o = 0; o < n; ++o) {
        const unsigned long long ko = ldk(keys + o);
        rank += (ko > ke) || (ko == ke && ldj(jmap + o) < je);
      }
      if (rank < count) {
        const Scores s = scorer(i, je);
        out.indices[obase + rank] = je;
        out.hybrid[obase + rank] = f64_from_orderable(ke);
        out.genre[obase + rank] = s.g;
        out.text[obase + rank] = s.t;
        out.metadata[obase + rank] = s.m;
      }
    }
    for (int e = count + tid; e < k; e += nthr) {
      out.indices[obase + e] = -1;
      out.hybrid[obase + e] = NAN;
      out.genre[obase + e] = NAN;
      out.text[obase + e] = NAN;
      out.metadata[obase + e] = NAN;
    }
    if (tid == 0) out.counts[orow] = count;
    __syncthreads();
    return;
  }
  if (tid == 0) { sm.above = 0; sm.taken = 0; sm.prefix = 0ull; sm.rank = count; }
  __syncthreads();
  if (count > 0) {
    for (int shift = 56; shift >= 0; shift -= 8) {
      for (int b = tid; b < 256; b += nthr) sm.hist[b] = 0u;
      __syncthreads();
      const unsigned long long prefix = sm.prefix;
      const unsigned long long hi_mask = shift == 56 ? 0ull : (~0ull << (shift + 8));
#pragma unroll 4
      for (int j = tid; j < n; j += nthr) {
        const unsigned long long key = ldk(keys + j);  // generic: global scratch or shared memory
        if (key != 0ull && (key & hi_mask) == prefix) atomicAdd(&sm.hist[(key >> shift) & 0xFFu], 1u);
      }
      __syncthreads();
      if (tid == 0) {
        int rank = sm.rank;  // rank-th largest among keys matching the prefix
        int d = 255;
        for (; d > 0; --d) {
          const int c = static_cast<int>(sm.hist[d]);
          if (rank <= c) break;
          rank -= c;
        }
        sm.prefix = prefix | (static_cast<unsigned long long>(d) << shift);
        sm.rank = rank;
      }
      __syncthreads();
    }
    const unsigned long long vstar = sm.prefix;  // count-th largest key
#pragma unroll 4
    for (int j = tid; j < n; j += nthr) {
      const unsigned long long key = ldk(keys + j);
      if (key > vstar) {
        const int pos = atomicAdd(&sm.above, 1);
        sm.win_key[pos] = key;
        sm.win_j[pos] = jmap ? ldj(jmap + j) : j;
      }
    }
    __syncthreads();
    const int above = sm.above;
    const int need = count - above;  // >= 1 : lowest column indices among keys == v*
    const int nwarps = nthr >> 5;
    if (kOrdered) {
      for (int base = 0; base < n; base += nthr) {
        const int j = base + tid;
        const bool flag = j < n && ldk(keys + j) == vstar;
        const unsigned bal = __ballot_sync(kFullMask, flag);
        if (lane == 0) sm.warp_tot[warp] = __popc(bal);
        __syncthreads();
        int before = sm.taken;
        for (int w = 0; w < warp; ++w) before += sm.warp_tot[w];
        int chunk_total = 0;
        for (int w = 0; w < nwarps; ++w) chunk_total += sm.warp_tot[w];
        const int pos = before + __popc(bal & ((1u << lane) - 1u));
        if (flag && pos < need) {
          sm.win_key[above + pos] = vstar;
          sm.win_j[above + pos] = jmap ? ldj(jmap + j) : j;
        }
        __syncthreads();
        if (tid == 0) sm.taken += chunk_total;
        __syncthreads();
        if (sm.taken >= need) break;
      }
    } else {
      // need-th smallest column among the entries equal to v* (columns are distinct)
      if (tid == 0) { sm.prefix = 0ull; sm.rank = need; }
      __syncthreads();
      for (int shift = 24; shift >= 0; shift -= 8) {
        for (int b = tid; b < 256; b += nthr) sm.hist[b] = 0u;
        __syncthreads();
        const unsigned int prefix = static_cast<unsigned int>(sm.prefix);
        const unsigned int hi_mask = shift == 24 ? 0u : (~0u << (shift + 8));
        for (int e = tid; e < n; e += nthr) {
          const unsigned int col = static_cast<unsigned int>(ldj(jmap + e));
          if (ldk(keys + e) == vstar && (col & hi_mask) == prefix) atomicAdd(&sm.hist[(col >> shift) & 0xFFu], 1u);
        }
        __syncthreads();
        if (tid == 0) {
          int rank = sm.rank;
          int d = 0;
          for (; d < 255; ++d) {
            const int c = static_cast<int>(sm.hist[d]);
            if (rank <= c) break;
            rank -= c;
          }
          sm.prefix = prefix | (static_cast<unsigned int>(d) << shift);
          sm.rank = rank;
        }
        __syncthreads();
      }
      const int jstar = static_cast<int>(sm.prefix);
      for (int e = tid; e < n; e += nthr) {
        if (ldk(keys + e) == vstar && ldj(jmap + e) <= jstar) {
          const int pos = atomicAdd(&sm.taken, 1);
          sm.win_key[above + pos] = vstar;
          sm.win_j[above + pos] = ldj(jmap + e);
        }
      }
    }
    __syncthreads();
    for (int e = tid; e < count; e += nthr) {
      const unsigned long long ke = sm.win_key[e];
      const int je = sm.win_j[e];
      int rank = 0;
      for (int o = 0; o < count; ++o)
        rank += (sm.win_key[o] > ke) || (sm.win_key[o] == ke && sm.win_j[o] < je);
      const Scores s = scorer(i, je);
      out.indices[obase + rank] = je;
      out.hybrid[obase + rank] = f64_from_orderable(ke);
      out.genre[obase + rank] = s.g;
      out.text[obase + rank] = s.t;
      out.metadata[obase + rank] = s.m;
    }
  }
  for (int e = count + tid; e < k; e += nthr) {
    out.indices[obase + e] = -1;
    out.hybrid[obase + e] = NAN;
    out.genre[obase + e] = NAN;
    out.text[obase + e] = NAN;
    out.metadata[obase + e] = NAN;
  }
  if (tid == 0) out.counts[orow] = count;
  __syncthreads();
}

// generic form: one source row per CTA pass, any scorer (used for the N x N matrix variant)
template <class Scorer>
__global__ void __launch_bounds__(K6_THREADS)
exact_rows_kernel(const Scorer scorer, const SelectParams sel, const int* __restrict__ rows,
                  int n_listed, const int* __restrict__ count_ptr, int list_cap, int row_begin,
                  int rows_are_local, unsigned long long* __restrict__ key_scratch,
                  tvbf_topk_out out) {
  __shared__ SelectSmem sm;
  const int tid = threadIdx.x, lane = tid & 31;
  const int n = sel.n;
  const int listed = count_ptr ? *count_ptr : n_listed;
  const int list0 = list_cap > 0 ? list_cap - listed : 0;
  unsigned long long* keys = key_scratch + static_cast<size_t>(blockIdx.x) * n;
  for (int t = list0 + blockIdx.x; t < list0 + listed; t += gridDim.x) {
    const int r = rows[t];
    const int i = rows_are_local ? row_begin + r : r;
    const int orow = rows_are_local ? r : t;
    if (tid == 0) sm.valid = 0;
    __syncthreads();
    int my_valid = 0;
    for (int j = tid; j < n; j += K6_THREADS) {
      const Scores s = scorer(i, j);
      const bool ok = (s.h >= sel.min_similarity) && !(sel.exclude_self && j == i);
      keys[j] = ok ? f64_orderable(s.h) : 0ull;
      my_valid += ok;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) my_valid += __shfl_xor_sync(kFullMask, my_valid, o);
    if (lane == 0 && my_valid) atomicAdd(&sm.valid, my_valid);
    __syncthreads();
    select_and_emit<true, false>(sm, keys, nullptr, n, sel.k, sm.valid, i, static_cast<size_t>(orow), scorer, out);
  }
}

// ---------------------------------------------------------------------------------------------
// K6, feature form.  Two kernels:
//   exact_rows_notext_kernel  rows known to have no text (the tie plateaus K5 flags): genre /
//                             metadata only, up to 8 rows per CTA, no CSR traffic at all
//   exact_rows_text_kernel    rows that may have text: the catalogue CSR (~12 B per text nnz, 56 MB
//                             at C3) is streamed warp-cooperatively against a shared-memory mask
//                             of the batch rows' vocabulary; when only a few rows are listed (the
//                             usual case: near-ties under the fp16 bound are rare, and the online
//                             single-show query) each row's COLUMNS are split over the CTAs and
//                             the last CTA of a row selects from the shared survivor list
// ---------------------------------------------------------------------------------------------
constexpr int K6B_THREADS = 1024;
constexpr int K6B_MAXB = 8;       // no-text kernel: batch rows per CTA (scratch is sized for this)
constexpr int K6B_TEXTB = 4;      // text kernel: batch rows
constexpr int K6B_SMALL = 4096;   // survivors that are selected from shared memory
constexpr int K6B_LIST = 16384;   // survivors listed per row (global scratch); more -> dense keys
constexpr int K6B_ROWNNZ = 192;   // text entries of a batch row staged in shared memory
constexpr size_t K6T_COUNTER_BYTES = 65536;   // text kernel: survivor counters + batch tickets

__device__ __forceinline__ double csr_lookup(const tvbf_features& f, int64_t b, int64_t e, int c) {
  // value of column c in the sorted row segment [b, e); the caller knows it is present
  while (b < e) {
    const int64_t mid = (b + e) >> 1;
    const int cm = f.text_indices[mid];
    if (cm == c) return f.text_values[mid];
    if (cm < c) b = mid + 1; else e = mid;
  }
  return 0.0;
}

// column-independent pieces of the genre / metadata scores of the batch rows (shared memory)
template <int MAXB>
struct BatchRows {
  int row[MAXB];
  double floor[MAXB];
  double gr[MAXB], mr[MAXB];          // 1/sqrt(set size) of the row's genre / metadata bits
  unsigned long long gb[MAXB], gh[MAXB];
  unsigned int mb[MAXB];
  double rs[129], m3[4];              // 1/sqrt(n), n/3
};

// hybrid score of batch row r against column show j (text part given); same expressions as
// genre_score() / meta_score() / score_pair()
template <int MAXB>
__device__ __forceinline__ double batch_hybrid(const ScoreParams& sp, const BatchRows<MAXB>& br, int r,
                                               int j, bool packed, const TvbfColSide& cj, unsigned long long hj,
                                               double g_rj, double m_rj, double text) {
  const tvbf_features& f = sp.f;
  double g = 0.0, mm = 0.0;
  if (packed) {
    if (f.genre_mode == TVBF_GROUP_PACKED)
      g = static_cast<double>(__popcll(br.gb[r] & cj.genre_bits) + __popcll(br.gh[r] & hj)) * (br.gr[r] * g_rj);
    if (f.meta_mode == TVBF_GROUP_PACKED) {
      const int eq = __popc(br.mb[r] & cj.meta_bits);
      mm = f.meta_kind == TVBF_META_MEAN3 ? br.m3[eq] : static_cast<double>(eq) * (br.mr[r] * m_rj);
    }
  } else {
    g = genre_score(f, br.row[r], j);
    mm = meta_score(f, br.row[r], j);
  }
  return hybrid_rn(sp.wg, g, sp.wt, text, sp.wm, mm);
}

template <int MAXB>
__device__ __forceinline__ void batch_rows_init(BatchRows<MAXB>& br, int tid) {
  if (tid < 129) br.rs[tid] = tid ? 1.0 / sqrt(static_cast<double>(tid)) : 0.0;
  if (tid < 4) br.m3[tid] = static_cast<double>(tid) / 3.0;
}

template <int MAXB>
__device__ __forceinline__ void batch_rows_load(BatchRows<MAXB>& br, int slot, int i, double floor_v,
                                                bool packed, const TvbfColSide* cs,
                                                const unsigned long long* genre_hi = nullptr) {
  br.row[slot] = i;
  br.floor[slot] = floor_v;
  br.gh[slot] = 0ull;
  if (packed && i >= 0) {
    const TvbfColSide ci = cs[i];
    const unsigned long long hi = genre_hi ? genre_hi[i] : 0ull;
    const int gni = __popcll(ci.genre_bits) + __popcll(hi), mni = __popc(ci.meta_bits);
    br.gb[slot] = ci.genre_bits;
    br.gh[slot] = hi;
    br.mb[slot] = ci.meta_bits;
    br.gr[slot] = gni ? 1.0 / sqrt(static_cast<double>(gni)) : 0.0;
    br.mr[slot] = mni ? 1.0 / sqrt(static_cast<double>(mni)) : 0.0;
  }
}

// Exact top-k of one batch row from what the scoring pass left behind: its survivor list (columns
// that reach the row's floor) when that holds everything, else dense keys over all N columns.
// kCg: the lists were written by other CTAs of this launch (column-split text kernel).
template <bool kCg>
__device__ void k6_select_row(SelectSmem& sm, const ScoreParams& sp, const FeatureScorer& scorer, int i,
                              double floor_i, int survivors, const unsigned long long* surv_key_r,
                              const int* surv_j_r, unsigned long long* keys_r, bool dense_written,
                              unsigned long long* small_key, int* small_j, size_t orow,
                              const tvbf_topk_out& out) {
  const int tid = threadIdx.x;
  const int n = sp.f.n_shows;
  if (survivors <= K6B_SMALL) {
    // few survivors: select from their list, staged in shared memory (instead of ~10 passes over
    // N keys)
    __syncthreads();
    for (int e = tid; e < survivors; e += K6B_THREADS) {
      small_key[e] = __ldcg(surv_key_r + e);
      small_j[e] = __ldcg(surv_j_r + e);
    }
    __syncthreads();
    select_and_emit<false, false>(sm, small_key, small_j, survivors, sp.k, survivors, i, orow, scorer, out);
  } else if (survivors <= K6B_LIST) {
    // a wide tie plateau: select over the survivor list where it lies (L2), not over N keys
    select_and_emit<false, kCg>(sm, surv_key_r, surv_j_r, survivors, sp.k, survivors, i, orow, scorer, out);
  } else {
    if (!dense_written) {
      // rare: a floor that more than K6B_LIST columns reach; the dense keys were not written
      __syncthreads();
      for (int j = tid; j < n; j += K6B_THREADS) {
        const Scores sc = scorer(i, j);
        const bool ok = (sc.h >= sp.min_similarity) && (sc.h >= floor_i) && !(sp.exclude_self && j == i);
        keys_r[j] = ok ? f64_orderable(sc.h) : 0ull;
      }
      __threadfence();
      __syncthreads();
    }
    select_and_emit<true, kCg>(sm, keys_r, nullptr, n, sp.k, survivors, i, orow, scorer, out);
  }
}

// rows / floors hold `listed` entries at [0, listed), or at [list_cap - listed, list_cap) when
// list_cap > 0 (K5 lists the shows without text from the back).
__global__ void __launch_bounds__(K6B_THREADS, 1)
exact_rows_notext_kernel(const ScoreParams sp, const int* __restrict__ rows, int n_listed,
                         const int* __restrict__ count_ptr, int list_cap,
                         const double* __restrict__ floors, int row_begin, int rows_are_local,
                         unsigned long long* __restrict__ key_scratch, tvbf_topk_out out) {
  constexpr int MAXB = K6B_MAXB;
  // dynamic smem: [small_key: K6B_SMALL u64][small_j: K6B_SMALL int]
  extern __shared__ __align__(16) unsigned long long small_key[];
  __shared__ SelectSmem sm;
  __shared__ BatchRows<MAXB> br;
  __shared__ int s_valid[MAXB];
  int* small_j = reinterpret_cast<int*>(small_key + K6B_SMALL);
  const tvbf_features& f = sp.f;
  const int tid = threadIdx.x;
  const int n = f.n_shows;
  const int listed = count_ptr ? *count_ptr : n_listed;
  if (listed <= 0) return;
  const int list0 = list_cap > 0 ? list_cap - listed : 0;
  int B = (listed + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  B = B < 1 ? 1 : (B > MAXB ? MAXB : B);
  const int n_batches = (listed + B - 1) / B;
  unsigned long long* keys0 = key_scratch + static_cast<size_t>(blockIdx.x) * MAXB * n;
  // survivor lists (columns that reach the row's floor), appended in arbitrary order while scoring
  unsigned long long* surv_key = key_scratch + static_cast<size_t>(gridDim.x) * MAXB * n +
                                 static_cast<size_t>(blockIdx.x) * MAXB * K6B_LIST;
  int* surv_j = reinterpret_cast<int*>(key_scratch + static_cast<size_t>(gridDim.x) * MAXB *
                                                         (static_cast<size_t>(n) + K6B_LIST)) +
                static_cast<size_t>(blockIdx.x) * MAXB * K6B_LIST;
  const bool packed = f.genre_mode != TVBF_GROUP_FOLDED && f.meta_mode != TVBF_GROUP_FOLDED;
  const TvbfColSide* cs = static_cast<const TvbfColSide*>(f.col_side);
  const unsigned long long* ghi = reinterpret_cast<const unsigned long long*>(f.genre_hi);
  // without floors every column is a survivor and the selection runs over dense keys; with floors
  // the survivor lists almost always suffice and the dense keys are not written at all
  const bool dense = floors == nullptr;
  batch_rows_init(br, tid);

  for (int batch = blockIdx.x; batch < n_batches; batch += gridDim.x) {
    const int nb = (listed - batch * B) < B ? (listed - batch * B) : B;
    __syncthreads();
    if (tid < MAXB) {
      s_valid[tid] = 0;
      if (tid < nb) {
        const int r = rows[list0 + batch * B + tid];
        batch_rows_load(br, tid, rows_are_local ? row_begin + r : r,
                        floors ? floors[list0 + batch * B + tid] : -INFINITY, packed, cs, ghi);
      } else {
        batch_rows_load(br, tid, -1, INFINITY, packed, cs, ghi);
      }
    }
    __syncthreads();
    for (int j = tid; j < n; j += K6B_THREADS) {
      TvbfColSide cj;
      unsigned long long hj = 0ull;
      double g_rj = 0.0, m_rj = 0.0;
      if (packed) {
        cj = cs[j];
        if (ghi) hj = ghi[j];
        g_rj = br.rs[__popcll(cj.genre_bits) + __popcll(hj)];
        m_rj = br.rs[__popc(cj.meta_bits)];
      }
#pragma unroll
      for (int r = 0; r < MAXB; ++r) {
        if (r < nb) {
          const double h = batch_hybrid(sp, br, r, j, packed, cj, hj, g_rj, m_rj, 0.0);
          // only columns that reach the row's floor (a lower bound of its k-th best score) can
          // matter; everything else is "invalid"
          const bool ok = (h >= sp.min_similarity) && (h >= br.floor[r]) && !(sp.exclude_self && j == br.row[r]);
          const unsigned long long key = ok ? f64_orderable(h) : 0ull;
          if (dense) keys0[static_cast<size_t>(r) * n + j] = key;
          if (ok) {
            const int pos = atomicAdd(&s_valid[r], 1);
            if (pos < K6B_LIST) {
              surv_key[r * K6B_LIST + pos] = key;
              surv_j[r * K6B_LIST + pos] = j;
            }
          }
        }
      }
    }
    __syncthreads();
    const FeatureScorer scorer{sp};
    for (int r = 0; r < nb; ++r) {
      const int t = list0 + batch * B + r;
      const int orow = rows_are_local ? rows[t] : t;
      k6_select_row<false>(sm, sp, scorer, br.row[r], br.floor[r], s_valid[r], surv_key + r * K6B_LIST,
                           surv_j + r * K6B_LIST, keys0 + static_cast<size_t>(r) * n, dense, small_key, small_j,
                           static_cast<size_t>(orow), out);
    }
  }
}

// Text form.  scratch (key_scratch): [counters: K6T_COUNTER_BYTES][surv_key: cap_rows x K6B_LIST u64]
// [surv_j: cap_rows x K6B_LIST int][dense keys: cap_rows x n u64].  Row slots: the listed position
// when listed <= cap_rows (column-split mode, counters zeroed by the launcher), else per-CTA slots.
__global__ void __launch_bounds__(K6B_THREADS, 1)
exact_rows_text_kernel(const ScoreParams sp, const int* __restrict__ rows, int n_listed,
                       const int* __restrict__ count_ptr, int list_cap,
                       const double* __restrict__ floors, int row_begin, int rows_are_local,
                       int mask_bytes, unsigned long long* __restrict__ key_scratch, int cap_rows,
                       tvbf_topk_out out) {
  constexpr int MAXB = K6B_TEXTB;
  // dynamic smem: [mask: vocab bytes][small_key: K6B_SMALL u64][small_j: K6B_SMALL int]
  extern __shared__ __align__(16) unsigned int mask_words[];
  __shared__ SelectSmem sm;
  __shared__ BatchRows<MAXB> br;
  __shared__ long long s_b[MAXB], s_e[MAXB];
  __shared__ int s_last;
  // the batch rows' own (column, value) lists, staged so that a mask hit is resolved by a binary
  // search in shared memory (rows with more than K6B_ROWNNZ entries are searched in global memory)
  __shared__ int s_cols[MAXB][K6B_ROWNNZ];
  __shared__ double s_vals[MAXB][K6B_ROWNNZ];
  unsigned long long* small_key =
      reinterpret_cast<unsigned long long*>(reinterpret_cast<unsigned char*>(mask_words) + mask_bytes);
  int* small_j = reinterpret_cast<int*>(small_key + K6B_SMALL);
  const tvbf_features& f = sp.f;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = f.n_shows;
  const int listed = count_ptr ? *count_ptr : n_listed;
  if (listed <= 0) return;
  const int list0 = list_cap > 0 ? list_cap - listed : 0;
  const int G = static_cast<int>(gridDim.x);
  int B = (listed + G - 1) / G;
  B = B < 1 ? 1 : (B > MAXB ? MAXB : B);
  const int n_batches = (listed + B - 1) / B;
  const bool split = listed <= cap_rows;          // one scratch slot per listed row
  const int S = split && n_batches < G ? G / n_batches : 1;   // column slices per batch
  const int items = n_batches * S;
  const int chunks = (n + 31) / 32;
  const int words = (f.vocab + 3) / 4;
  const unsigned char* mask = reinterpret_cast<const unsigned char*>(mask_words);
  int* cnt = reinterpret_cast<int*>(key_scratch);
  int* ticket = cnt + 8192;
  unsigned long long* surv_key = key_scratch + K6T_COUNTER_BYTES / 8;
  int* surv_j = reinterpret_cast<int*>(surv_key + static_cast<size_t>(cap_rows) * K6B_LIST);
  unsigned long long* dense_keys = surv_key + static_cast<size_t>(cap_rows) * K6B_LIST * 3 / 2;
  const bool packed = f.genre_mode != TVBF_GROUP_FOLDED && f.meta_mode != TVBF_GROUP_FOLDED;
  const TvbfColSide* cs = static_cast<const TvbfColSide*>(f.col_side);
  const unsigned long long* ghi = reinterpret_cast<const unsigned long long*>(f.genre_hi);
  const bool dense = floors == nullptr;
  batch_rows_init(br, tid);

  for (int item = blockIdx.x; item < items; item += G) {
    const int batch = item / S, slice = item % S;
    const int nb = (listed - batch * B) < B ? (listed - batch * B) : B;
    const int slot0 = split ? batch * B : static_cast<int>(blockIdx.x) * MAXB;
    __syncthreads();
    for (int w = tid; w < words; w += K6B_THREADS) mask_words[w] = 0u;
    if (tid < MAXB) {
      if (tid < nb) {
        const int r = rows[list0 + batch * B + tid];
        const int i = rows_are_local ? row_begin + r : r;
        batch_rows_load(br, tid, i, floors ? floors[list0 + batch * B + tid] : -INFINITY, packed, cs, ghi);
        s_b[tid] = f.text_indptr[i];
        s_e[tid] = f.text_indptr[i + 1];
        if (!split) cnt[slot0 + tid] = 0;   // per-CTA slots are reused from batch to batch
      } else {
        batch_rows_load(br, tid, -1, INFINITY, packed, cs, ghi);
        s_b[tid] = 0; s_e[tid] = 0;
      }
    }
    __syncthreads();
    bool any_text = false;
    for (int r = 0; r < nb; ++r) {
      any_text |= s_e[r] > s_b[r];
      const bool staged = (s_e[r] - s_b[r]) <= K6B_ROWNNZ;
      for (long long e = s_b[r] + tid; e < s_e[r]; e += K6B_THREADS) {
        const int c = f.text_indices[e];
        atomicOr(&mask_words[c >> 2], (1u << r) << (8 * (c & 3)));
        if (staged) {
          s_cols[r][e - s_b[r]] = c;
          s_vals[r][e - s_b[r]] = f.text_values[e];
        }
      }
    }
    __syncthreads();

    // Each warp takes 32 consecutive column shows per step (lane = column).  Their CSR segments
    // are one contiguous span, streamed with coalesced loads (lane = entry) and tested against
    // the mask.  Every hit lane looks its product up in parallel; the products then go to the
    // lane that owns the entry's column one by one in ascending entry order, so each pair's sum
    // runs over ascending column index with one rounding per product and per add, like text_dot.
    const int ch0 = static_cast<int>(static_cast<long long>(chunks) * slice / S);
    const int ch1 = static_cast<int>(static_cast<long long>(chunks) * (slice + 1) / S);
    for (int ch = ch0 + warp; ch < ch1; ch += K6B_THREADS / 32) {
      const int j0 = ch * 32;
      const int j = j0 + lane;
      double acc[MAXB];
#pragma unroll
      for (int r = 0; r < MAXB; ++r) acc[r] = 0.0;
      if (any_text) {
        const long long ip = f.text_indptr[j < n ? j : n];   // first entry of this lane's column
        const long long span_b = __shfl_sync(kFullMask, ip, 0);
        const long long span_e = f.text_indptr[j0 + 32 < n ? j0 + 32 : n];
        // four 32-entry groups (8 loads) are always in flight: a slot is refilled with the group
        // 128 entries ahead as soon as it has been consumed
        int c[4];
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const long long e = span_b + u * 32 + lane;
          c[u] = e < span_e ? f.text_indices[e] : -1;
          v[u] = e < span_e ? f.text_values[e] : 0.0;
        }
        for (long long off = span_b; off < span_e; off += 128) {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const long long e = off + u * 32 + lane;
            const int cu = c[u];
            const double vu = v[u];
            {
              const long long en = e + 128;
              c[u] = en < span_e ? f.text_indices[en] : -1;
              v[u] = en < span_e ? f.text_values[en] : 0.0;
            }
            const unsigned mu = cu >= 0 ? mask[cu] : 0u;
            if (__ballot_sync(kFullMask, mu != 0u) == 0u) continue;
            // lane that owns this lane's entry: the last one whose column starts at or before it
            int owner = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
              const long long ipc = __shfl_sync(kFullMask, ip, (owner + step) & 31);
              if (ipc <= e) owner += step;
            }
#pragma unroll
            for (int r = 0; r < MAXB; ++r) {
              const bool mine = (mu >> r) & 1u;
              unsigned hits = __ballot_sync(kFullMask, mine);
              if (hits == 0u) continue;
              double prod = 0.0;
              if (mine) {
                const int len = static_cast<int>(s_e[r] - s_b[r]);
                double xv = 0.0;
                if (len <= K6B_ROWNNZ) {
                  int lo = 0, hi = len;
                  while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    const int cm = s_cols[r][mid];
                    if (cm == cu) { xv = s_vals[r][mid]; break; }
                    if (cm < cu) lo = mid + 1; else hi = mid;
                  }
                } else {
                  xv = csr_lookup(f, s_b[r], s_e[r], cu);
                }
                prod = __dmul_rn(xv, vu);
              }
              while (hits) {
                const int hl = __ffs(hits) - 1;
                hits &= hits - 1;
                const int o = __shfl_sync(kFullMask, owner, hl);
                const double pp = __shfl_sync(kFullMask, prod, hl);
                if (lane == o) acc[r] = __dadd_rn(acc[r], pp);
              }
            }
          }
        }
      }
      // genre / metadata parts and the survivor test (all lanes stay in: ballots below)
      const bool in = j < n;
      TvbfColSide cj{0ull, 0.0f, 0u};
      unsigned long long hj = 0ull;
      double g_rj = 0.0, m_rj = 0.0;
      if (packed && in) {
        cj = cs[j];
        if (ghi) hj = ghi[j];
        g_rj = br.rs[__popcll(cj.genre_bits) + __popcll(hj)];
        m_rj = br.rs[__popc(cj.meta_bits)];
      }
#pragma unroll
      for (int r = 0; r < MAXB; ++r) {
        if (r < nb) {
          bool ok = false;
          unsigned long long key = 0ull;
          if (in) {
            const double h = batch_hybrid(sp, br, r, j, packed, cj, hj, g_rj, m_rj, acc[r]);
            ok = (h >= sp.min_similarity) && (h >= br.floor[r]) && !(sp.exclude_self && j == br.row[r]);
            key = ok ? f64_orderable(h) : 0ull;
            if (dense) dense_keys[static_cast<size_t>(slot0 + r) * n + j] = key;
          }
          const unsigned okb = __ballot_sync(kFullMask, ok);
          if (okb) {   // one counter update per warp: the row's survivor list may be shared by many CTAs
            const int leader = __ffs(okb) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(&cnt[slot0 + r], __popc(okb));
            base = __shfl_sync(kFullMask, base, leader);
            const int pos = base + __popc(okb & ((1u << lane) - 1u));
            if (ok && pos < K6B_LIST) {
              surv_key[static_cast<size_t>(slot0 + r) * K6B_LIST + pos] = key;
              surv_j[static_cast<size_t>(slot0 + r) * K6B_LIST + pos] = j;
            }
          }
        }
      }
    }
    // the last CTA to finish a batch selects its rows (no waiting: everybody else just leaves)
    __threadfence();
    __syncthreads();
    if (S > 1) {
      if (tid == 0) s_last = atomicAdd(&ticket[batch], 1) == S - 1;
      __syncthreads();
      if (!s_last) continue;
      __threadfence();
    }
    const FeatureScorer scorer{sp};
    for (int r = 0; r < nb; ++r) {
      const int t = list0 + batch * B + r;
      const int orow = rows_are_local ? rows[t] : t;
      const size_t slot = static_cast<size_t>(slot0 + r);
      k6_select_row<true>(sm, sp, scorer, br.row[r], br.floor[r], __ldcg(cnt + slot), surv_key + slot * K6B_LIST,
                          surv_j + slot * K6B_LIST, dense_keys + slot * n, dense, small_key, small_j,
                          static_cast<size_t>(orow), out);
    }
  }
}

// exact fp64 scores of explicit (i, j) pairs: out[p] = {hybrid, genre, text, metadata}
__global__ void score_pairs_kernel(const ScoreParams sp, const int* __restrict__ pairs, int n_pairs,
                                   double* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_pairs) return;
  const int i = pairs[2 * t], j = pairs[2 * t + 1];
  Scores s{0.0, 0.0, 0.0, 0.0};
  if (i >= 0 && j >= 0 && i < sp.f.n_shows && j < sp.f.n_shows) s = score_pair(sp, i, j);
  out[4 * t + 0] = s.h;
  out[4 * t + 1] = s.g;
  out[4 * t + 2] = s.t;
  out[4 * t + 3] = s.m;
}

int score_pairs_launch(const ScoreParams& sp, const int* pairs, int n_pairs, double* out,
                       cudaStream_t st) {
  score_pairs_kernel<<<(n_pairs + 127) / 128, 128, 0, st>>>(sp, pairs, n_pairs, out);
  TVBF_LAUNCH_OK("score_pairs_kernel");
  return TVBF_OK;
}

// ---------------------------------------------------------------------------------------------
// host-side launchers used by api.cu
// ---------------------------------------------------------------------------------------------
int k5_launch(const ScoreParams& sp, const uint2* cand, const int* cand_cnt,
              const float* cand_theta, int splits, CandLayout lay, int kp, int row_begin, int n_rows,
              const tvbf_topk_out& out, int* flagged_rows, double* flagged_floor, cudaStream_t st) {
  const int max_cand = splits * kp;
  int warps = K5_WARPS;
  while (warps > 1 && static_cast<size_t>(warps) * max_cand * 48 > 200 * 1024) warps >>= 1;
  const size_t smem = static_cast<size_t>(warps) * max_cand * 48;
  if (smem > 200 * 1024) {
    tvbf_set_error("rescore: lists*candidates = %d is too large", max_cand);
    return TVBF_ERR_INVALID;
  }
  TVBF_CUDA_OK(cudaFuncSetAttribute(rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(smem)));
  const int grid = (n_rows + warps - 1) / warps;
  rescore_kernel<<<grid, warps * 32, smem, st>>>(sp, cand, cand_cnt, cand_theta, splits, lay, kp,
                                                 row_begin, n_rows, out, flagged_rows, flagged_floor,
                                                 max_cand, 2 * kp);
  TVBF_LAUNCH_OK("rescore_kernel");
  return TVBF_OK;
}

int k5_launch_listed(const ScoreParams& sp, const uint2* cand, const int* cand_cnt, const float* cand_theta,
                     int splits, CandLayout lay, int kp, int row_begin, int n_rows, const int* rows,
                     const int* n_listed, const tvbf_topk_out& out, int* flagged_rows, double* flagged_floor,
                     cudaStream_t st, const double* cut_score, const int* cut_index) {
  const int max_cand = splits * kp;
  int warps = K5_WARPS;
  while (warps > 1 && static_cast<size_t>(warps) * max_cand * 48 > 200 * 1024) warps >>= 1;
  const size_t smem = static_cast<size_t>(warps) * max_cand * 48;
  if (smem > 200 * 1024) {
    tvbf_set_error("rescore: lists*candidates = %d is too large", max_cand);
    return TVBF_ERR_INVALID;
  }
  const int grid = (n_rows + warps - 1) / warps;   // at most n_rows listed; the count is on the device
  if (lay.gathered) {
    if (cut_index != nullptr) {
      tvbf_set_error("rescore: gathered lists take no rank cut");
      return TVBF_ERR_INVALID;
    }
    TVBF_CUDA_OK(cudaFuncSetAttribute(rescore_gathered_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
    rescore_gathered_kernel<<<grid, warps * 32, smem, st>>>(sp, cand, cand_cnt, cand_theta, splits, lay, kp,
                                                            row_begin, n_rows, rows, n_listed, out, flagged_rows,
                                                            flagged_floor, max_cand, 2 * kp);
    TVBF_LAUNCH_OK("rescore_gathered_kernel");
    return TVBF_OK;
  }
  if (cut_index != nullptr) {
    TVBF_CUDA_OK(cudaFuncSetAttribute(rescore_cut_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
    rescore_cut_kernel<<<grid, warps * 32, smem, st>>>(sp, cand, cand_cnt, cand_theta, splits, lay, kp, row_begin,
                                                       n_rows, rows, n_listed, out, flagged_rows, flagged_floor,
                                                       max_cand, 2 * kp, cut_score, cut_index);
    TVBF_LAUNCH_OK("rescore_cut_kernel");
    return TVBF_OK;
  }
  TVBF_CUDA_OK(cudaFuncSetAttribute(rescore_listed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    static_cast<int>(smem)));
  rescore_listed_kernel<<<grid, warps * 32, smem, st>>>(sp, cand, cand_cnt, cand_theta, splits, lay, kp, row_begin,
                                                        n_rows, rows, n_listed, out, flagged_rows, flagged_floor,
                                                        max_cand, 2 * kp);
  TVBF_LAUNCH_OK("rescore_listed_kernel");
  return TVBF_OK;
}

static int k6_cap_rows(int sm_count) { return sm_count * K6B_MAXB; }

size_t k6_scratch_bytes(int n_shows, int sm_count) {
  // no-text kernel: one CTA per SM, up to K6B_MAXB rows each: dense keys + survivor lists of
  // K6B_LIST (key, column) entries per row; the text kernel lays the same bytes out per listed row
  // behind its counters
  return K6T_COUNTER_BYTES + static_cast<size_t>(k6_cap_rows(sm_count)) *
                                 (static_cast<size_t>(n_shows) * 8 + K6B_LIST * 12);
}

int k6_launch(const ScoreParams& sp, const int* rows, int n_listed, const int* count_ptr,
              const double* floors, int row_begin, int rows_are_local, unsigned long long* key_scratch,
              int grid, const tvbf_topk_out& out, cudaStream_t st, int no_text, int list_cap) {
  if (sp.k > K6_MAXK) {
    tvbf_set_error("exact rows: k=%d exceeds %d", sp.k, K6_MAXK);
    return TVBF_ERR_INVALID;
  }
  const size_t mask_bytes = (static_cast<size_t>(sp.f.vocab) + 15) / 16 * 16;
  if (no_text) {
    // rows known to have no text: no mask, no CSR
    const size_t smem = static_cast<size_t>(K6B_SMALL) * 12;
    TVBF_CUDA_OK(cudaFuncSetAttribute(exact_rows_notext_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
    exact_rows_notext_kernel<<<grid, K6B_THREADS, smem, st>>>(sp, rows, n_listed, count_ptr, list_cap, floors,
                                                              row_begin, rows_are_local, key_scratch, out);
    TVBF_LAUNCH_OK("exact_rows_notext_kernel");
    return TVBF_OK;
  }
  const size_t smem = mask_bytes + static_cast<size_t>(K6B_SMALL) * 12;
  if (k6_cap_rows(grid) > 8192) {   // counters and tickets: two int arrays of 8192 in K6T_COUNTER_BYTES
    tvbf_set_error("exact rows: grid of %d CTAs exceeds the counter area", grid);
    return TVBF_ERR_INVALID;
  }
  if (smem <= 160 * 1024) {
    TVBF_CUDA_OK(cudaFuncSetAttribute(exact_rows_text_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
    TVBF_CUDA_OK(cudaMemsetAsync(key_scratch, 0, K6T_COUNTER_BYTES, st));
    exact_rows_text_kernel<<<grid, K6B_THREADS, smem, st>>>(sp, rows, n_listed, count_ptr, list_cap, floors,
                                                            row_begin, rows_are_local,
                                                            static_cast<int>(mask_bytes), key_scratch,
                                                            k6_cap_rows(grid), out);
    TVBF_LAUNCH_OK("exact_rows_text_kernel");
    return TVBF_OK;
  }
  // vocabulary too wide for the shared-memory mask: one row per CTA pass
  FeatureScorer sc{sp};
  SelectParams sel{sp.f.n_shows, sp.k, sp.exclude_self, sp.min_similarity};
  exact_rows_kernel<FeatureScorer><<<grid, K6_THREADS, 0, st>>>(
      sc, sel, rows, n_listed, count_ptr, list_cap, row_begin, rows_are_local, key_scratch, out);
  TVBF_LAUNCH_OK("exact_rows_kernel");
  return TVBF_OK;
}

int k6_launch_flagged(const ScoreParams& sp, const int* flagged, const double* floors, int n_rows,
                      int row_begin, unsigned long long* key_scratch, int grid, const tvbf_topk_out& out,
                      cudaStream_t st) {
  int rc = k6_launch(sp, flagged, 0, out.stats + 2, floors, row_begin, 1, key_scratch, grid, out, st, 0, 0);
  if (rc != TVBF_OK) return rc;
  return k6_launch(sp, flagged, 0, out.stats + 3, floors, row_begin, 1, key_scratch, grid, out, st, 1, n_rows);
}

int k6_launch_matrix(const double* h, const double* g, const double* t, const double* m, int n,
                     int k, int exclude_self, double min_similarity, const int* rows, int n_listed,
                     unsigned long long* key_scratch, int grid, const tvbf_topk_out& out,
                     cudaStream_t st) {
  if (k > K6_MAXK) {
    tvbf_set_error("matrix rows: k=%d exceeds %d", k, K6_MAXK);
    return TVBF_ERR_INVALID;
  }
  MatrixScorer sc{h, g, t, m, n};
  SelectParams sel{n, k, exclude_self, min_similarity};
  exact_rows_kernel<MatrixScorer><<<grid, K6_THREADS, 0, st>>>(sc, sel, rows, n_listed, nullptr, 0, 0,
                                                               0, key_scratch, out);
  TVBF_LAUNCH_OK("exact_rows_kernel<matrix>");
  return TVBF_OK;
}

}  // namespace tvbf
