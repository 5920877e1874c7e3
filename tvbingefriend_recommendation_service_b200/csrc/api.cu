// C ABI of libtvbf (see include/tvbf.h): argument validation, workspace carving and the launch
// sequence K1 (tcgen05 candidate pass) -> K5 (fp64 rescore + certificate) -> K6 (exact repair).
#include "internal.cuh"

#include <atomic>
#include <cmath>
#include <cstdarg>

static thread_local char g_last_error[512] = "";
static std::atomic<unsigned long long> g_launches{0};

static std::atomic<unsigned long long> g_coop_fallbacks{0};

void tvbf_count_launch(void) { g_launches.fetch_add(1, std::memory_order_relaxed); }
void tvbf_count_coop_fallback(void) { g_coop_fallbacks.fetch_add(1, std::memory_order_relaxed); }

void tvbf_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
  va_end(ap);
}

namespace {

__global__ void iota_kernel(int* dst, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = i;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int sm_count_cached(int* out) {
  int dev = 0;
  TVBF_CUDA_OK(cudaGetDevice(&dev));
  int sms = 0, major = 0;
  TVBF_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  TVBF_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) {
    tvbf_set_error("libtvbf needs an sm_100 device (B200); found compute capability %d.x", major);
    return TVBF_ERR_UNSUPPORTED;
  }
  *out = sms;
  return TVBF_OK;
}

struct Plan {
  int rows, cg, sb_count, col_tiles, splits, sb_per_group, grid, entries, kp, k6_grid;
  int tiles_per_split, sync_kb, sync_slack, stages, sym, sym_cap, cand_lists;
  size_t off_scratch, off_cand, off_cnt, off_theta, off_flag, off_floor, off_keys, off_count, off_gtheta, off_gcnt,
      off_glist, total;
};

int validate_features(const tvbf_features* f) {
  TVBF_REQUIRE(f != nullptr, "features is NULL");
  TVBF_REQUIRE(f->n_shows > 0, "n_shows must be positive");
  TVBF_REQUIRE(f->n_pad >= f->n_shows && f->n_pad % 256 == 0, "n_pad must be a multiple of 256 >= n_shows");
  TVBF_REQUIRE(f->k_pad > 0 && f->k_pad % 64 == 0, "k_pad must be a positive multiple of 64");
  TVBF_REQUIRE(f->operand && f->col_side && f->meta_scale, "operand / col_side / meta_scale missing");
  TVBF_REQUIRE(f->text_indptr && f->text_indices && f->text_values, "text CSR missing");
  TVBF_REQUIRE(f->text_dtype == TVBF_TEXT_FP16 || f->text_dtype == TVBF_TEXT_BF16, "bad text_dtype");
  TVBF_REQUIRE((reinterpret_cast<uintptr_t>(f->operand) & 127) == 0, "operand must be 128-byte aligned");
  TVBF_REQUIRE((reinterpret_cast<uintptr_t>(f->col_side) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(f->meta_scale) & 15) == 0,
               "col_side / meta_scale must be 16-byte aligned");
  if (f->genre_mode == TVBF_GROUP_FOLDED)
    TVBF_REQUIRE(f->genre_dense && f->genre_dim > 0, "folded genre needs genre_dense");
  if (f->genre_mode == TVBF_GROUP_PACKED) {
    TVBF_REQUIRE(f->genre_dim >= 1 && f->genre_dim <= 128, "packed genre: %d columns outside 1..128", f->genre_dim);
    TVBF_REQUIRE((f->genre_dim > 64) == (f->genre_hi != nullptr),
                 "packed genre: genre_hi must be given exactly when there are more than 64 columns");
    if (f->genre_hi) TVBF_REQUIRE((reinterpret_cast<uintptr_t>(f->genre_hi) & 15) == 0, "genre_hi must be 16-byte aligned");
  }
  TVBF_REQUIRE(f->text_cols >= 0 && f->text_cols <= f->vocab && f->text_cols <= f->k_pad,
               "text_cols %d outside [0, min(vocab %d, k_pad %d)]", f->text_cols, f->vocab, f->k_pad);
  if (f->text_cols > 0)
    TVBF_REQUIRE(!f->text_signed, "a merged text operand (text_cols > 0) needs non-negative text");
  TVBF_REQUIRE(f->text_nnz >= 0 && f->text_nnz < INT32_MAX, "text_nnz %lld outside [0, 2^31 - 1)",
               static_cast<long long>(f->text_nnz));
  if (f->bits_folded) {
    TVBF_REQUIRE(f->genre_mode == TVBF_GROUP_PACKED && f->meta_mode == TVBF_GROUP_PACKED && !f->text_signed,
                 "bits_folded needs packed genre and metadata groups and non-negative text");
    const int text_end = f->text_cols > 0 ? f->text_cols : f->vocab;
    TVBF_REQUIRE(f->fold_col0 >= text_end && f->fold_col0 + f->genre_dim + 32 <= f->k_pad,
                 "bits_folded: columns [%d, %d) do not fit k_pad %d", f->fold_col0, f->fold_col0 + f->genre_dim + 32,
                 f->k_pad);
    TVBF_REQUIRE(f->fold_weights[1] > 0.0 && f->fold_weights[0] >= 0.0 && f->fold_weights[2] >= 0.0,
                 "bits_folded needs text_weight > 0 and non-negative genre / metadata weights");
  }
  if (f->meta_mode == TVBF_GROUP_FOLDED) {
    TVBF_REQUIRE(f->meta_groups == (f->meta_kind == TVBF_META_MEAN3 ? 3 : 1), "bad meta_groups");
    for (int g = 0; g < f->meta_groups; ++g)
      TVBF_REQUIRE(f->meta_dense[g] && f->meta_dims[g] > 0, "folded metadata group %d missing", g);
  }
  return TVBF_OK;
}

int validate_params(const tvbf_features* f, const tvbf_params* p) {
  TVBF_REQUIRE(p != nullptr, "params is NULL");
  TVBF_REQUIRE(p->k >= 1, "k must be >= 1");
  TVBF_REQUIRE(p->row_begin >= 0 && p->row_begin % 128 == 0, "row_begin must be a multiple of 128");
  TVBF_REQUIRE(p->row_end > p->row_begin && p->row_end <= f->n_shows, "bad row range [%d, %d)",
               p->row_begin, p->row_end);
  TVBF_REQUIRE(std::isfinite(p->genre_weight) && std::isfinite(p->text_weight) &&
                   std::isfinite(p->metadata_weight),
               "weights must be finite");
  return TVBF_OK;
}

// sweep > 1: a weight sweep -- every list-shaped region holds `sweep` slices of n_pad virtual shows
int make_plan(const tvbf_features* f, const tvbf_params* p, Plan* pl, int sweep = 1) {
  int sms = 0;
  int rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  pl->rows = p->row_end - p->row_begin;
  // tuning: bits 0-3 cta_group (0 = 2), bits 4-11 pacing chunk in k-blocks (0 = 16, 255 = off),
  // bits 12-15 pacing slack in chunks (0 = 2)
  const int tune = p->tuning;
  pl->cg = (tune & 0xF) == 1 && f->genre_hi == nullptr ? 1 : 2;   // two-word genre masks: CTA pairs only
  pl->sync_kb = ((tune >> 4) & 0xFF) == 0 ? 16 : (((tune >> 4) & 0xFF) == 255 ? 0 : ((tune >> 4) & 0xFF));
  // an operand that stays in L2 whatever the CTAs do (126 MB) needs no pacing: the lockstep only costs
  // (P80k, 92 MB: K1 5.01 ms paced, 4.79 ms free-running)
  if (((tune >> 4) & 0xFF) == 0 && static_cast<size_t>(f->n_pad) * f->k_pad * 2 <= (static_cast<size_t>(96) << 20))
    pl->sync_kb = 0;
  pl->sync_slack = ((tune >> 12) & 0xF) == 0 ? 2 : ((tune >> 12) & 0xF);
  // bits 16-19 ring stages (0 = all); bits 20-21 symmetric mode (0 = auto, 1 = off, 2 = on)
  const int max_stages = pl->cg == 2 ? 6 : 4;
  pl->stages = ((tune >> 16) & 0xF) == 0 ? max_stages : ((tune >> 16) & 0xF);
  if (pl->stages > max_stages) pl->stages = max_stages;
  if (pl->stages < 2) pl->stages = 2;
  pl->sym = 0;
  pl->sym_cap = 1024;   // entries per shared list; 4096 once more than 64 candidates are kept (set below)
  const int sb_rows = 128 * pl->cg;
  pl->sb_count = (pl->rows + sb_rows - 1) / sb_rows;
  pl->col_tiles = (f->n_shows + 255) / 256;
  pl->entries = tvbf::k1_entries_per_lane(p->k);
  pl->kp = 0;
  pl->splits = 1;
  pl->sb_per_group = 1;
  pl->grid = pl->cg;
  pl->tiles_per_split = pl->col_tiles;
  const bool use_k1 = !p->force_exact && pl->entries != 0;
  if (use_k1) {
    pl->kp = p->candidates > 0 ? p->candidates : tvbf::k1_default_candidates(p->k);
    const int cap = 32 * pl->entries;
    TVBF_REQUIRE(pl->kp >= p->k && pl->kp <= cap - 64, "candidates=%d must lie in [k, %d]", pl->kp,
                 cap - 64);
    const int clusters = sms / pl->cg;
    pl->splits = p->splits > 0 ? p->splits : tvbf::k1_choose_splits(pl->sb_count, pl->col_tiles, clusters);
    if (pl->splits > pl->col_tiles) pl->splits = pl->col_tiles;
    if (pl->splits > clusters) pl->splits = clusters;
    while (pl->splits > 1 && pl->splits * pl->kp > 1024) --pl->splits;
    TVBF_REQUIRE(pl->splits >= 1, "bad splits %d", pl->splits);
    pl->sb_per_group = clusters / pl->splits;
    if (pl->sb_per_group > pl->sb_count) pl->sb_per_group = pl->sb_count;
    pl->grid = pl->sb_per_group * pl->splits * pl->cg;
    pl->tiles_per_split = (pl->col_tiles + pl->splits - 1) / pl->splits;
    // Symmetric mode: hybrid(i,j) == hybrid(j,i), so only tiles on or above the diagonal are
    // computed and each score is offered to both shows.  Needs the whole catalogue in one shard,
    // CTA pairs (256-row super block == 256-column tile), packed groups with non-negative weights,
    // and thresholds that are positive floats (the shared thresholds are raised with atomicMax on
    // their raw bits): a positive min_similarity, or -- for min_similarity <= 0 -- non-negative text,
    // so that every upper bound U is > 0 and the initial threshold can be +0 ("everything passes").
    if (pl->kp > 64) pl->sym_cap = 4096;
    const int sym_req = (tune >> 20) & 0x3;
    const bool eligible = pl->cg == 2 && p->row_begin == 0 && p->row_end == f->n_shows &&
                          f->genre_mode != TVBF_GROUP_FOLDED && f->meta_mode != TVBF_GROUP_FOLDED &&
                          p->genre_weight >= 0.0 && p->text_weight >= 0.0 && p->metadata_weight >= 0.0 &&
                          (p->min_similarity > 1e-30 || !f->text_signed) && pl->kp <= 128 && p->exclude_self;
    if (sym_req == 2) TVBF_REQUIRE(eligible, "symmetric mode requested but the job is not eligible");
    // auto: worth it once the triangle is large (measured: C2, 79 tiles, is 15 % slower; C3, 391
    // tiles, 1.5x faster)
    pl->sym = (sym_req == 2 || (sym_req == 0 && eligible && pl->col_tiles >= 160)) ? 1 : 0;
    if (pl->sym && p->splits <= 0) {
      // the symmetric sweep keeps ONE shared list per show, so rescoring does not grow with the
      // split count; more splits = fewer phantom tiles under the diagonal
      pl->splits = 8;
      while (pl->splits > 1 && (clusters / pl->splits < 1 || pl->col_tiles / pl->splits < 8)) --pl->splits;
      pl->sb_per_group = clusters / pl->splits;
      if (pl->sb_per_group > pl->sb_count) pl->sb_per_group = pl->sb_count;
      pl->grid = pl->sb_per_group * pl->splits * pl->cg;
      pl->tiles_per_split = (pl->col_tiles + pl->splits - 1) / pl->splits;
    }
  }
  pl->cand_lists = pl->sym ? 1 : pl->splits;
  pl->k6_grid = sms;
  size_t off = 0;
  pl->off_scratch = off; off = align_up(off + (use_k1 ? static_cast<size_t>(pl->grid) * 128 * 32 * pl->entries * 8 : 0), 256);
  const size_t list_rows = sweep > 1 ? static_cast<size_t>(sweep) * f->n_pad : static_cast<size_t>(pl->rows);
  const size_t sym_rows = static_cast<size_t>(sweep > 1 ? sweep : 1) * f->n_pad;
  pl->off_cand = off;    off = align_up(off + (use_k1 ? list_rows * pl->cand_lists * pl->kp * 8 : 0), 256);
  pl->off_cnt = off;     off = align_up(off + list_rows * pl->cand_lists * 4, 256);
  pl->off_theta = off;   off = align_up(off + list_rows * pl->cand_lists * 4, 256);
  pl->off_gtheta = off;  off = align_up(off + (pl->sym ? sym_rows * 4 : 0), 256);
  pl->off_gcnt = off;    off = align_up(off + (pl->sym ? sym_rows * 4 : 0), 256);
  pl->off_glist = off;   off = align_up(off + (pl->sym ? sym_rows * pl->sym_cap * 8 : 0), 256);
  pl->off_flag = off;    off = align_up(off + static_cast<size_t>(pl->rows) * 4, 256);
  pl->off_floor = off;   off = align_up(off + static_cast<size_t>(pl->rows) * 8, 256);
  pl->off_count = off;   off = align_up(off + 256, 256);
  pl->off_keys = off;    off = align_up(off + tvbf::k6_scratch_bytes(*f, sms), 256);
  pl->total = off;
  return TVBF_OK;
}

tvbf::ScoreParams score_params(const tvbf_features* f, const tvbf_params* p) {
  tvbf::ScoreParams sp;
  sp.f = *f;
  sp.wg = p->genre_weight;
  sp.wt = p->text_weight;
  sp.wm = p->metadata_weight;
  sp.min_similarity = p->min_similarity;
  sp.k = p->k;
  sp.exclude_self = p->exclude_self;
  return sp;
}

// ---- slack of the upper bound U >= exact hybrid -------------------------------------------------
// (1) operand rounding: the product of two fp16/bf16-rounded NORMAL numbers differs from the exact
//     product by at most (2u + u^2) relative, u = unit roundoff.
// (2) fp16 subnormal operands (x * 2^s < 2^-14) carry an ABSOLUTE error <= 2^-25 instead; against an
//     operand of magnitude <= op_max * 2^s that is <= 2^-25 * op_max * 2^s per product.
// (3) accumulation inside the tensor core: products of two 11-bit significands are exact in fp32;
//     model of one tcgen05.mma K=16 step: the non-zero addends (products and the running sum) are
//     aligned to the largest exponent keeping >= 24 significant bits, truncated, summed, and the
//     sum rounded to fp32 -- each non-zero addend loses < 2^-23 of the largest magnitude, zero
//     addends lose nothing (adding zeros is exact).  With at most T non-zero products in a pair
//     (T = non-zero operand entries of the row) the total loss is < (2T + T) * 2^-23 * sum|a_k b_k|.
//     kAccUnit budgets 4 * 2^-23 per term.  tests/test_gpu_parity.py::test_fp16_error_bound_*
//     measure the three parts against float64 on sparse and on dense 50k-wide text.
// Non-negative text (TF-IDF): sum|a_k b_k| == acc, all three are taken relative to |acc| per row.
// Signed text or folded float groups: cancellation breaks that, so the bound is absolute via
// Cauchy-Schwarz on the unit rows: sum|a_k b_k| <= ||a|| ||b|| = 2^2s * (w_text + folded weights) / w_text.
double operand_rel_err(int dtype) {
  const double u = dtype == TVBF_TEXT_BF16 ? 1.0 / 256.0 : 1.0 / 2048.0;  // unit roundoff
  return (2.0 * u + u * u) * 1.01;
}
constexpr double kAccUnit = 4.0 / 8388608.0 * 1.01;       // 4 * 2^-23 per term
constexpr double kSubnormalUnit = 2.0 / 8589934592.0;     // 2 * 2^-33 per term (score units, x <= 1)

struct Slack {
  float w_text, w_text_err, w_text_acc, eps, eps_term;
};

Slack make_slack(const tvbf_features* f, double wg, double wt, double wm, double rel_override) {
  const double inv_scale2 = std::ldexp(1.0, -2 * f->text_scale_log2);
  const double rel = rel_override > 0 ? rel_override : operand_rel_err(f->text_dtype);
  double folded_w = 0.0, op_max = 1.0;
  if (f->genre_mode == TVBF_GROUP_FOLDED) {
    folded_w += std::fabs(wg);
    if (wt > 0) op_max = std::fmax(op_max, std::sqrt(std::fabs(wg) / wt));
  }
  if (f->meta_mode == TVBF_GROUP_FOLDED) {
    folded_w += std::fabs(wm);
    const double per_group = f->meta_kind == TVBF_META_MEAN3 ? std::fabs(wm) / 3.0 : std::fabs(wm);
    if (wt > 0) op_max = std::fmax(op_max, std::sqrt(per_group / wt));
  }
  if (f->bits_folded && wt > 0) {
    // packed groups carried as operand columns (non-negative, so the relative bound below holds for
    // the whole accumulator): largest operand magnitude relative to a text entry (<= 1)
    op_max = std::fmax(op_max, std::sqrt(std::fabs(wg) / wt));
    op_max = std::fmax(op_max, std::sqrt(std::fabs(wm) / wt));
  }
  if (f->text_cols > 0) {
    // merged text: an entry sums at most vocab - text_cols + 1 entries of a unit row, so it is at most
    // the square root of that (Cauchy-Schwarz); only the subnormal term needs the largest operand
    op_max = std::fmax(op_max, std::sqrt(static_cast<double>(f->vocab - f->text_cols + 1)));
  }
  const double wsum = std::fabs(wg) + std::fabs(wt) + std::fabs(wm);
  const double eps0 = 4e-6 * (wsum + 1.0);   // fp32 rounding of the epilogue's four FMAs
  Slack s;
  s.w_text = static_cast<float>(wt * inv_scale2);
  const double sub = f->text_dtype == TVBF_TEXT_FP16 ? kSubnormalUnit * std::fabs(wt) * op_max : 0.0;
  if (folded_w > 0.0 || f->text_signed) {
    const double mass = std::fabs(wt) + folded_w;      // bound of sum|a_k b_k| in score units
    s.w_text_err = 0.0f;
    s.w_text_acc = 0.0f;
    s.eps = static_cast<float>(eps0 + rel * mass);
    s.eps_term = static_cast<float>(kAccUnit * mass + sub);
  } else {
    s.w_text_err = static_cast<float>(std::fabs(wt) * inv_scale2 * rel);
    s.w_text_acc = static_cast<float>(std::fabs(wt) * inv_scale2 * kAccUnit);
    s.eps = static_cast<float>(eps0);
    s.eps_term = static_cast<float>(sub);
  }
  return s;
}

// Everything the candidate kernel needs besides the launch geometry: pointers into the workspace,
// the fp32 weights of the epilogue and the slack terms of the upper bound U.
int fill_k1_params(const tvbf_features* f, const tvbf_params* p, const Plan& pl, uint8_t* ws,
                   tvbf::K1Params* out_kp, int n_sweep = 1) {
  const bool any_folded = f->genre_mode == TVBF_GROUP_FOLDED || f->meta_mode == TVBF_GROUP_FOLDED;
  if (any_folded) {
    TVBF_REQUIRE(p->text_weight > 0.0, "folded feature groups need text_weight > 0");
    TVBF_REQUIRE(p->genre_weight >= 0.0 && p->metadata_weight >= 0.0,
                 "folded feature groups need non-negative weights");
  }

  if (f->bits_folded) {
    TVBF_REQUIRE(n_sweep == 1, "a weight sweep needs the plain operand (bits_folded catalogues bake one triple)");
    TVBF_REQUIRE(p->genre_weight == f->fold_weights[0] && p->text_weight == f->fold_weights[1] &&
                     p->metadata_weight == f->fold_weights[2],
                 "this operand carries the genre / metadata columns for weights (%g, %g, %g), not (%g, %g, %g)",
                 f->fold_weights[0], f->fold_weights[1], f->fold_weights[2], p->genre_weight, p->text_weight,
                 p->metadata_weight);
  }

  tvbf::K1Params& kp = *out_kp;
  memset(&kp, 0, sizeof(kp));
  kp.col_side = static_cast<const TvbfColSide*>(f->col_side);
  kp.meta_scale = f->meta_scale;
  kp.genre_hi = f->genre_mode == TVBF_GROUP_PACKED ? reinterpret_cast<const unsigned long long*>(f->genre_hi) : nullptr;
  kp.scratch = reinterpret_cast<uint2*>(ws + pl.off_scratch);
  kp.cand = reinterpret_cast<uint2*>(ws + pl.off_cand);
  kp.cand_cnt = reinterpret_cast<int*>(ws + pl.off_cnt);
  kp.cand_theta = reinterpret_cast<float*>(ws + pl.off_theta);
  kp.n_shows = f->n_shows;
  kp.row_begin = p->row_begin;
  kp.row_end = p->row_end;
  kp.k_blocks = f->k_pad / 64;
  kp.col_tiles = pl.col_tiles;
  kp.splits = pl.splits;
  kp.rb_count = pl.sb_count;
  kp.rb_per_group = pl.sb_per_group;
  kp.tiles_per_split = pl.tiles_per_split;
  kp.sync_kb = pl.sync_kb;
  kp.sync_slack = pl.sync_slack;
  kp.stages = pl.stages;
  kp.sym = pl.sym;
  kp.deal_groups = 0;   // single GPU: local super block == global super block
  kp.deal_r = 1;
  kp.tile_stride = 1;
  kp.seed_theta = 0;
  if (pl.sym) {
    // bits 22-27 of tuning: column-tile stride of the threshold seed pass (0 = auto, 63 = no seeding)
    // (values above 48 step by 8: 50 -> 64, 54 -> 96, 58 -> 128, 62 -> 160)
    const int st_req = (p->tuning >> 22) & 0x3F;
    // default: every 96th tile but at least 4 sampled tiles (measured on C3: stride 48 62.2 ms per
    // step, 64 61.1, 96 61.0, 128 61.6, 160 61.5)
    int st_auto = pl.col_tiles / 4;
    st_auto = st_auto > 96 ? 96 : (st_auto < 8 ? 8 : st_auto);
    kp.tile_stride = st_req == 0 ? st_auto : (st_req == 63 ? 1 : (st_req <= 48 ? st_req : 48 + (st_req - 48) * 8));
    if (kp.tile_stride > pl.col_tiles) kp.tile_stride = pl.col_tiles > 1 ? pl.col_tiles : 1;
  }
  kp.sym_cap = pl.sym_cap;
  kp.g_theta = reinterpret_cast<unsigned int*>(ws + pl.off_gtheta);
  kp.g_cnt = reinterpret_cast<unsigned int*>(ws + pl.off_gcnt);
  kp.g_list = reinterpret_cast<uint2*>(ws + pl.off_glist);
  kp.cooperative = ((p->tuning >> 30) & 1) ? 0 : 1;  // bit 30: plain launch (profilers that patch SASS)
  {
    // experiment knobs (environment, read once): TVBF_REFRESH_PERIOD (0 = doubling schedule),
    // TVBF_WAIT_NS (first sleep of the backed-off waits)
    static const int env_period = [] { const char* e = getenv("TVBF_REFRESH_PERIOD"); return e ? atoi(e) : -1; }();
    static const int env_wait = [] { const char* e = getenv("TVBF_WAIT_NS"); return e ? atoi(e) : -1; }();
    // default: the doubling schedule.  Measured on P80k / C3: refreshing every 32 appends leaves 24 %
    // fewer list entries (19.1 M against 25.2 M / 24.9 M against 33.5 M) but the extra refreshes cost
    // more than the appends they save (K1 9.5 against 8.9 ms / 56.7 against 56.9 ms)
    kp.refresh_period = env_period >= 0 ? env_period : 0;
    kp.wait_ns = env_wait >= 0 ? env_wait : 64;
  }
  // 16 epilogue warps when the tile's MMAs (~0.27 us per 64-wide k-block) cannot hide the epilogue
  // (~30 us per tile with 8 warps); bits 28-29 of tuning: 0 auto, 1 off, 2 on
  {
    const int wide_req = (p->tuning >> 28) & 0x3;
    kp.wide_epilogue = (wide_req == 2 || (wide_req == 0 && f->k_pad / 64 <= 96)) && pl.kp <= 64 ? 1 : 0;
  }
  kp.progress = reinterpret_cast<unsigned int*>(ws + pl.off_count);
  kp.kp = pl.kp;
  kp.exclude_self = p->exclude_self;
  {
    // folded groups: operand columns were scaled by 2^s * sqrt(w_group / text_weight), so
    // acc * text_weight * 2^-2s is the whole folded part of the hybrid
    const Slack sl = make_slack(f, p->genre_weight, p->text_weight, p->metadata_weight, p->text_rel_err);
    kp.w_text = sl.w_text;
    kp.w_text_err = sl.w_text_err;
    kp.w_text_acc = sl.w_text_acc;
    kp.eps = sl.eps;
    kp.eps_term = sl.eps_term;
  }
  kp.text_indptr = f->text_indptr;
  {
    int folded = 0;
    if (f->genre_mode == TVBF_GROUP_FOLDED) folded += f->genre_dim;
    if (f->meta_mode == TVBF_GROUP_FOLDED)
      for (int g = 0; g < f->meta_groups; ++g) folded += f->meta_dims[g];
    if (f->bits_folded) folded = f->genre_dim + 3;   // non-zero folded entries of a row: its genres + 3 one-hots
    kp.folded_cols = folded;
  }
  kp.fold = f->bits_folded ? 1 : 0;
  kp.w_genre = f->genre_mode == TVBF_GROUP_PACKED && !f->bits_folded ? static_cast<float>(p->genre_weight) : 0.0f;
  kp.w_meta = f->meta_mode == TVBF_GROUP_PACKED && !f->bits_folded ? static_cast<float>(p->metadata_weight) : 0.0f;
  if (f->bits_folded) kp.genre_hi = nullptr;   // the second mask word is in the operand as well
  kp.meta_hstack = f->meta_kind == TVBF_META_HSTACK ? 1 : 0;
  {
    // strictly below min_similarity in fp32 so that U >= min_similarity always passes "U > theta"
    const double ms = p->min_similarity;
    float th = static_cast<float>(ms);
    if (!(ms > -3.0e38)) th = -3.0e38f;
    th = std::nextafterf(th, -INFINITY);
    if (static_cast<double>(th) >= ms) th = std::nextafterf(th, -INFINITY);
    // symmetric sweep with min_similarity <= 0: every U is > 0 (non-negative weights and features,
    // eps > 0), so +0 drops nothing and keeps the thresholds' raw bits ordered like unsigned integers
    if (pl.sym && th < 0.0f) th = 0.0f;
    kp.theta_init = th;
  }
  kp.n_weights = 1;
  kp.n_pad = f->n_pad;
  // no upper bound U exceeds the sum of the weights by more than its (relative) slack
  auto score_hi = [](const tvbf_params& q) {
    return static_cast<float>((std::fabs(q.genre_weight) + std::fabs(q.text_weight) + std::fabs(q.metadata_weight)) * 1.02 + 1e-3);
  };
  kp.score_hi = score_hi(*p);
  if (n_sweep > 1) {
    // weight sweep over the triples p[0 .. n_sweep) (packed groups only, checked by the caller):
    // the epilogue constants of every triple, same formulas as above
    kp.n_weights = n_sweep;
    for (int w = 0; w < n_sweep; ++w) {
      const tvbf_params& q = p[w];
      const Slack sl = make_slack(f, q.genre_weight, q.text_weight, q.metadata_weight, q.text_rel_err);
      kp.mw_text[w] = sl.w_text;
      kp.mw_text_err[w] = sl.w_text_err;
      kp.mw_text_acc[w] = sl.w_text_acc;
      kp.mw_eps[w] = sl.eps;
      kp.mw_eps_term[w] = sl.eps_term;
      kp.mw_genre[w] = static_cast<float>(q.genre_weight);
      kp.mw_meta[w] = static_cast<float>(q.metadata_weight);
      kp.mw_score_hi[w] = score_hi(q);
    }
  }
  return TVBF_OK;
}

}  // namespace

extern "C" {

int tvbf_version(void) { return TVBF_VERSION; }

const char* tvbf_last_error(void) { return g_last_error; }

uint64_t tvbf_kernel_launches(void) { return g_launches.load(std::memory_order_relaxed); }

uint64_t tvbf_noncooperative_fallbacks(void) { return g_coop_fallbacks.load(std::memory_order_relaxed); }

int tvbf_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor) {
  int dev = 0;
  TVBF_CUDA_OK(cudaGetDevice(&dev));
  int sms = 0, major = 0, minor = 0;
  TVBF_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  TVBF_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  TVBF_CUDA_OK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  if (sm_count) *sm_count = sms;
  if (cc_major) *cc_major = major;
  if (cc_minor) *cc_minor = minor;
  if (major != 10) {
    tvbf_set_error("libtvbf needs an sm_100 device (B200); found compute capability %d.%d", major,
                   minor);
    return TVBF_ERR_UNSUPPORTED;
  }
  return TVBF_OK;
}

size_t tvbf_topk_workspace_bytes(const tvbf_features* f, const tvbf_params* p) {
  if (validate_features(f) != TVBF_OK || validate_params(f, p) != TVBF_OK) return 0;
  Plan pl;
  if (make_plan(f, p, &pl) != TVBF_OK) return 0;
  return pl.total;
}

int tvbf_hybrid_topk(const tvbf_features* f, const tvbf_params* p, const tvbf_topk_out* out,
                     void* workspace, size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  rc = validate_params(f, p);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(out && out->indices && out->counts && out->hybrid && out->genre && out->text &&
                   out->metadata && out->stats,
               "output table has NULL members");
  TVBF_REQUIRE(workspace != nullptr, "workspace is NULL");
  Plan pl;
  rc = make_plan(f, p, &pl);
  if (rc != TVBF_OK) return rc;
  if (workspace_bytes < pl.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int* flagged = reinterpret_cast<int*>(ws + pl.off_flag);
  double* floors = reinterpret_cast<double*>(ws + pl.off_floor);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + pl.off_keys);
  const int phases = p->phases == 0 ? 7 : p->phases;
  if (phases & 1) TVBF_CUDA_OK(cudaMemsetAsync(out->stats, 0, 8 * sizeof(int32_t), st));
  const tvbf::ScoreParams sp = score_params(f, p);

  const bool use_k1 = !p->force_exact && pl.entries != 0;
  if (!use_k1) {
    // every row through the exact kernel
    iota_kernel<<<(pl.rows + 255) / 256, 256, 0, st>>>(flagged, pl.rows);
    TVBF_LAUNCH_OK("iota_kernel");
    rc = tvbf::k6_launch(sp, flagged, pl.rows, nullptr, nullptr, p->row_begin, 1, keys, pl.k6_grid, *out, st);
    if (rc != TVBF_OK) return rc;
    return TVBF_OK;
  }

  tvbf::K1Params kp;
  rc = fill_k1_params(f, p, pl, ws, &kp);
  if (rc != TVBF_OK) return rc;
  if (phases & 1) {
    TVBF_CUDA_OK(cudaMemsetAsync(kp.progress, 0, 256, st));
    rc = tvbf::k1_launch(f, kp, pl.entries, pl.cg, pl.grid, st);
    if (rc != TVBF_OK) return rc;
  }
  if ((phases & 2) && pl.sym) {
    static const bool dbg_counts = getenv("TVBF_DEBUG_COUNTS") != nullptr;
    if (dbg_counts) kp.dbg_entries = out->stats + 4;
    rc = tvbf::k4s_launch(kp, pl.rows, st);
    if (rc != TVBF_OK) return rc;
  }
  if (phases & 2) {
    const tvbf::CandLayout lay{0, pl.cand_lists, 1, 0};
    rc = tvbf::k5_launch(sp, kp.cand, kp.cand_cnt, kp.cand_theta, pl.cand_lists, lay, pl.kp,
                         p->row_begin, pl.rows, *out, flagged, floors, st);
    if (rc != TVBF_OK) return rc;
  }
  if ((phases & 4) && !p->skip_fallback) {
    rc = tvbf::k6_launch_flagged(sp, flagged, floors, pl.rows, p->row_begin, keys, pl.k6_grid, *out, st);
    if (rc != TVBF_OK) return rc;
  }
  return TVBF_OK;
}

// ---- weight sweep: several weight triples share ONE symmetric tensor-core sweep ----------------
namespace {
int sweep_plan(const tvbf_features* f, const tvbf_params* p, int n, tvbf_params* q, Plan* pl) {
  TVBF_REQUIRE(p != nullptr && n >= 1 && n <= tvbf::kMaxSweep, "weight sweep: 1..%d triples per call",
               tvbf::kMaxSweep);
  TVBF_REQUIRE(n == 1 || f->genre_hi == nullptr, "the shared weight sweep supports at most 64 genre columns");
  for (int w = 0; w < n; ++w) {
    int rc = validate_params(f, &p[w]);
    if (rc != TVBF_OK) return rc;
    TVBF_REQUIRE(p[w].k == p[0].k && p[w].min_similarity == p[0].min_similarity &&
                     p[w].exclude_self == p[0].exclude_self && p[w].row_begin == 0 &&
                     p[w].row_end == f->n_shows && !p[w].force_exact && p[w].phases == 0,
                 "weight sweep: triple %d differs from triple 0 in more than the weights (whole catalogue only)", w);
    // every triple must be eligible for the symmetric sweep on its own
    tvbf_params t = p[w];
    t.tuning = (t.tuning & ~(0x3 << 20)) | (2 << 20);
    t.tuning = (t.tuning & ~0xF) | 2;
    Plan tmp;
    rc = make_plan(f, &t, &tmp);
    if (rc != TVBF_OK) return rc;
  }
  *q = p[0];
  q->tuning = (q->tuning & ~(0x3 << 20)) | (2 << 20);
  q->tuning = (q->tuning & ~0xF) | 2;
  return make_plan(f, q, pl, n);
}
}  // namespace

size_t tvbf_topk_sweep_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_weights) {
  if (validate_features(f) != TVBF_OK) return 0;
  tvbf_params q;
  Plan pl;
  if (sweep_plan(f, p, n_weights, &q, &pl) != TVBF_OK) return 0;
  return pl.total;
}

int tvbf_hybrid_topk_sweep(const tvbf_features* f, const tvbf_params* p, int32_t n_weights,
                           const tvbf_topk_out* out, void* workspace, size_t workspace_bytes,
                           void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(out != nullptr && workspace != nullptr, "tvbf_hybrid_topk_sweep: NULL argument");
  tvbf_params q;
  Plan pl;
  rc = sweep_plan(f, p, n_weights, &q, &pl);
  if (rc != TVBF_OK) return rc;
  for (int w = 0; w < n_weights; ++w)
    TVBF_REQUIRE(out[w].indices && out[w].counts && out[w].hybrid && out[w].genre && out[w].text &&
                     out[w].metadata && out[w].stats,
                 "output table %d has NULL members", w);
  if (workspace_bytes < pl.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int* flagged = reinterpret_cast<int*>(ws + pl.off_flag);
  double* floors = reinterpret_cast<double*>(ws + pl.off_floor);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + pl.off_keys);
  tvbf::K1Params kp;
  rc = fill_k1_params(f, n_weights > 1 ? p : &q, pl, ws, &kp, n_weights);
  if (rc != TVBF_OK) return rc;
  TVBF_CUDA_OK(cudaMemsetAsync(kp.progress, 0, 256, st));
  rc = tvbf::k1_launch(f, kp, pl.entries, pl.cg, pl.grid, st);
  if (rc != TVBF_OK) return rc;
  // compaction of all n_weights * n_pad shared lists into the candidate tables [triple][show][kp]
  rc = tvbf::k4s_launch(kp, (n_weights > 1 ? n_weights : 1) * (n_weights > 1 ? f->n_pad : pl.rows), st);
  if (rc != TVBF_OK) return rc;
  for (int w = 0; w < n_weights; ++w) {
    TVBF_CUDA_OK(cudaMemsetAsync(out[w].stats, 0, 8 * sizeof(int32_t), st));
    const tvbf::ScoreParams sp = score_params(f, &p[w]);
    const tvbf::CandLayout lay{static_cast<long long>(w) * (n_weights > 1 ? f->n_pad : 0), 1, 1, 0};
    rc = tvbf::k5_launch(sp, kp.cand, kp.cand_cnt, kp.cand_theta, 1, lay, pl.kp, 0, pl.rows, out[w], flagged,
                         floors, st);
    if (rc != TVBF_OK) return rc;
    if (!q.skip_fallback) {
      rc = tvbf::k6_launch_flagged(sp, flagged, floors, pl.rows, 0, keys, pl.k6_grid, out[w], st);
      if (rc != TVBF_OK) return rc;
    }
  }
  return TVBF_OK;
}

// ---- symmetric sweep over several GPUs ---------------------------------------------------------
// Tile sharding instead of row sharding: GPU `rank` of `world` owns the 256-row super blocks dealt
// to it in zigzag order and sweeps their tiles on/above the diagonal, feeding the candidate lists of
// BOTH shows of every score, so it ends up with partial lists for ALL shows.  Three calls with one
// small collective between each (done by the caller, e.g. NCCL through torch.distributed):
//   tvbf_sym_seed   -> all_reduce(MAX) of theta[n_pad] (uint32)
//   tvbf_sym_sweep  -> all_gather of cand / cand_cnt / cand_bound
//   tvbf_rescore_lists (own row shard) -> gather of the result tables
namespace {

struct SymPlan {
  Plan pl;            // geometry of a full-catalogue symmetric job
  int local_sb;       // super blocks owned by this rank
  int deal_groups;    // ... in this many dealt groups of pl.sb_per_group consecutive blocks
  unsigned short gid[tvbf::kMaxDealGroups];
  size_t off_prog, off_scratch, off_gcnt, off_glist, off_flag, off_floor, off_keys, total;
};

int make_sym_plan(const tvbf_features* f, const tvbf_params* p, int rank, int world, SymPlan* sp) {
  TVBF_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank %d / world %d", rank, world);
  tvbf_params q = *p;
  q.row_begin = 0;
  q.row_end = f->n_shows;
  q.tuning = (q.tuning & ~(0x3 << 20)) | (2 << 20);   // symmetric mode on (or fail if ineligible)
  q.tuning = (q.tuning & ~0xF) | 2;                   // CTA pairs
  int rc = validate_params(f, &q);
  if (rc != TVBF_OK) return rc;
  rc = make_plan(f, &q, &sp->pl);
  if (rc != TVBF_OK) return rc;
  Plan& pl = sp->pl;
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  const int clusters = sms / 2;
  if (p->splits <= 0 && world >= 4) {
    // 12 column splits x 6 super blocks per wave: the per-GPU walks differ by < 1 % on C3 at 8 GPUs
    // (8 x 9: 3.5 %); the symmetric sweep keeps one list per show, so more splits cost nothing later
    pl.splits = 12;
    while (pl.splits > 1 && (clusters / pl.splits < 1 || pl.col_tiles / pl.splits < 8)) --pl.splits;
  }
  // One launch wave = one dealt group of R consecutive super blocks x S column splits: the blocks of
  // a wave then differ by < R diagonal tiles (the phantom tiles every item walks for the pacing).
  pl.sb_per_group = clusters / pl.splits;
  if (pl.sb_per_group > pl.sb_count) pl.sb_per_group = pl.sb_count;
  if (pl.sb_per_group < 1) pl.sb_per_group = 1;
  if (world == 1) {
    sp->deal_groups = 0;
    sp->local_sb = pl.sb_count;
  } else {
    sp->deal_groups = tvbf::k1_deal_groups(pl.sb_count, pl.sb_per_group, world, rank, sp->gid, &sp->local_sb);
    TVBF_REQUIRE(sp->deal_groups >= 0, "catalogue too large for the tile-sharded symmetric sweep on %d GPUs", world);
  }
  pl.grid = pl.sb_per_group * pl.splits * 2;
  size_t off = 0;
  sp->off_prog = off;    off = align_up(off + 256, 256);
  sp->off_scratch = off; off = align_up(off + static_cast<size_t>(sms) * 128 * 32 * pl.entries * 8, 256);
  sp->off_gcnt = off;    off = align_up(off + static_cast<size_t>(f->n_pad) * 4, 256);
  sp->off_glist = off;   off = align_up(off + static_cast<size_t>(f->n_pad) * pl.sym_cap * 8, 256);
  sp->off_flag = off;    off = align_up(off + static_cast<size_t>(f->n_shows) * 4, 256);
  sp->off_floor = off;   off = align_up(off + static_cast<size_t>(f->n_shows) * 8, 256);
  sp->off_keys = off;    off = align_up(off + tvbf::k6_scratch_bytes(*f, sms), 256);
  sp->total = off;
  return TVBF_OK;
}

int fill_sym_params(const tvbf_features* f, const tvbf_params* p, const SymPlan& sp, int rank, int world,
                    uint8_t* ws, uint32_t* theta, tvbf::K1Params* kp) {
  tvbf_params q = *p;
  q.row_begin = 0;
  q.row_end = f->n_shows;
  int rc = fill_k1_params(f, &q, sp.pl, ws, kp);
  if (rc != TVBF_OK) return rc;
  kp->scratch = reinterpret_cast<uint2*>(ws + sp.off_scratch);
  kp->progress = reinterpret_cast<unsigned int*>(ws + sp.off_prog);
  kp->g_theta = theta;
  kp->g_cnt = reinterpret_cast<unsigned int*>(ws + sp.off_gcnt);
  kp->g_list = reinterpret_cast<uint2*>(ws + sp.off_glist);
  kp->cand = nullptr;
  kp->cand_cnt = nullptr;
  kp->cand_theta = nullptr;
  kp->rb_count = sp.local_sb;
  kp->rb_per_group = sp.pl.sb_per_group;
  kp->seed_world = world;
  kp->seed_rank = rank;
  {
    int sms = 0;
    rc = sm_count_cached(&sms);
    if (rc != TVBF_OK) return rc;
    kp->seed_clusters = sms / 2;
  }
  kp->deal_groups = sp.deal_groups;
  kp->deal_r = sp.pl.sb_per_group;
  for (int g = 0; g < sp.deal_groups; ++g) kp->deal_gid[g] = sp.gid[g];
  // a rank that sweeps 1/world of the tiles gets fewer threshold refreshes: seed more densely
  // (measured at world = 8 on C3: stride 48 -> 0.6 + 8.0 ms per rank, stride 96 -> 0.4 + 8.5 ms)
  if (world >= 4 && ((p->tuning >> 22) & 0x3F) == 0 && kp->tile_stride > 48) kp->tile_stride = 48;
  return TVBF_OK;
}

}  // namespace

int tvbf_sym_eligible(const tvbf_features* f, const tvbf_params* p) {
  if (validate_features(f) != TVBF_OK || p == nullptr) return 0;
  SymPlan sp;
  return make_sym_plan(f, p, 0, 1, &sp) == TVBF_OK ? 1 : 0;
}

int32_t tvbf_sym_list_len(const tvbf_features* f, const tvbf_params* p) {
  SymPlan sp;
  if (validate_features(f) != TVBF_OK || make_sym_plan(f, p, 0, 1, &sp) != TVBF_OK) return 0;
  return sp.pl.kp;
}

size_t tvbf_sym_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t world) {
  SymPlan sp;
  if (validate_features(f) != TVBF_OK || make_sym_plan(f, p, 0, world, &sp) != TVBF_OK) return 0;
  return sp.total;
}

static int sym_seed_impl(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                         uint32_t* theta, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(theta && workspace, "tvbf_sym_seed: NULL buffer");
  SymPlan sp;
  rc = make_sym_plan(f, p, rank, world, &sp);
  if (rc != TVBF_OK) return rc;
  if (workspace_bytes < sp.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, sp.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  tvbf::K1Params kp;
  rc = fill_sym_params(f, p, sp, rank, world, ws, theta, &kp);
  if (rc != TVBF_OK) return rc;
  kp.sym_phase = 1;
  TVBF_CUDA_OK(cudaMemsetAsync(kp.progress, 0, 256, st));
  return tvbf::k1_launch(f, kp, sp.pl.entries, 2, sp.pl.grid, st);
}

int tvbf_sym_seed(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                  uint32_t* theta, void* workspace, size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  const int rc = sym_seed_impl(f, p, rank, world, theta, workspace, workspace_bytes, stream);
  if (rc != TVBF_OK) tvbf_absorb_pending_clear(stream);   // no sweep may trust a failed seed's clear
  return rc;
}

static int sym_sweep_phase(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                           uint32_t* theta, void* cand, int32_t* cand_cnt, float* cand_bound,
                           const uint64_t* peer_ptrs, int32_t shard_rows, void* workspace, size_t workspace_bytes,
                           void* stream) {
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(theta && workspace && (cand || peer_ptrs), "tvbf_sym_sweep: NULL buffer");
  TVBF_REQUIRE((cand_cnt == nullptr) == (cand_bound == nullptr),
               "tvbf_sym_sweep: pass both cand_cnt and cand_bound, or neither (packed rows)");
  SymPlan sp;
  rc = make_sym_plan(f, p, rank, world, &sp);
  if (rc != TVBF_OK) return rc;
  if (workspace_bytes < sp.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, sp.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  tvbf::K1Params kp;
  rc = fill_sym_params(f, p, sp, rank, world, ws, theta, &kp);
  if (rc != TVBF_OK) return rc;
  kp.sym_phase = 2;
  kp.cand = static_cast<uint2*>(cand);
  kp.cand_cnt = cand_cnt;
  kp.cand_theta = cand_bound;
  kp.cand_packed = cand_cnt == nullptr ? 1 : 0;
  if (peer_ptrs != nullptr) {
    TVBF_REQUIRE(world <= tvbf::kMaxPeers, "peer exchange supports at most %d GPUs", tvbf::kMaxPeers);
    TVBF_REQUIRE(shard_rows > 0 && static_cast<int64_t>(shard_rows) * world >= f->n_shows,
                 "tvbf_sym_sweep_peer: shard_rows * world must cover the catalogue");
    kp.cand_packed = 2;
    kp.peer_shard_rows = shard_rows;
    kp.peer_rank = rank;
    for (int r = 0; r < world; ++r) {
      TVBF_REQUIRE(peer_ptrs[r] != 0, "tvbf_sym_sweep_peer: NULL peer buffer %d", r);
      kp.peer_cand[r] = reinterpret_cast<uint2*>(static_cast<uintptr_t>(peer_ptrs[r]));
    }
  }
  TVBF_CUDA_OK(cudaMemsetAsync(kp.progress, 0, 256, st));
  if (sp.local_sb > 0) {
    rc = tvbf::k1_launch(f, kp, sp.pl.entries, 2, sp.pl.grid, st);
    if (rc != TVBF_OK) return rc;
  } else {
    rc = tvbf_absorb_pending_clear(stream);
    if (rc != TVBF_OK) return rc;
    TVBF_CUDA_OK(cudaMemsetAsync(kp.g_cnt, 0, static_cast<size_t>(f->n_pad) * 4, st));
  }
  return tvbf::k4s_launch(kp, f->n_shows, st);
}

static int sym_sweep_impl(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                          uint32_t* theta, void* cand, int32_t* cand_cnt, float* cand_bound,
                          const uint64_t* peer_ptrs, int32_t shard_rows, void* workspace, size_t workspace_bytes,
                          void* stream) {
  int rc = tvbf_enter_call(stream, 1);
  if (rc != TVBF_OK) return rc;
  rc = sym_sweep_phase(f, p, rank, world, theta, cand, cand_cnt, cand_bound, peer_ptrs, shard_rows, workspace,
                       workspace_bytes, stream);
  if (rc != TVBF_OK) tvbf_absorb_pending_clear(stream);
  return rc;
}

int tvbf_sym_sweep(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                   uint32_t* theta, void* cand, int32_t* cand_cnt, float* cand_bound,
                   void* workspace, size_t workspace_bytes, void* stream) {
  TVBF_REQUIRE(cand != nullptr, "tvbf_sym_sweep: NULL buffer");
  return sym_sweep_impl(f, p, rank, world, theta, cand, cand_cnt, cand_bound, nullptr, 0, workspace,
                        workspace_bytes, stream);
}

int tvbf_sym_sweep_peer(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                        uint32_t* theta, const uint64_t* peer_ptrs, int32_t shard_rows, void* workspace,
                        size_t workspace_bytes, void* stream) {
  TVBF_REQUIRE(peer_ptrs != nullptr, "tvbf_sym_sweep_peer: NULL peer pointer array");
  return sym_sweep_impl(f, p, rank, world, theta, nullptr, nullptr, nullptr, peer_ptrs, shard_rows, workspace,
                        workspace_bytes, stream);
}

int tvbf_rescore_lists(const tvbf_features* f, const tvbf_params* p, const void* cand_all,
                       const int32_t* cnt_all, const float* bound_all, int32_t lists,
                       int32_t table_row0, int32_t table_rows, const tvbf_topk_out* out,
                       void* workspace, size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  rc = validate_params(f, p);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(cand_all && lists >= 1 && (cnt_all == nullptr) == (bound_all == nullptr),
               "tvbf_rescore_lists: bad candidate tables");
  TVBF_REQUIRE(table_row0 >= 0 && table_row0 <= p->row_begin &&
                   static_cast<int64_t>(table_row0) + table_rows >= p->row_end,
               "tvbf_rescore_lists: the candidate tables do not cover rows [row_begin, row_end)");
  TVBF_REQUIRE(out && out->indices && out->counts && out->hybrid && out->genre && out->text &&
                   out->metadata && out->stats,
               "output table has NULL members");
  SymPlan sp;
  rc = make_sym_plan(f, p, 0, lists, &sp);
  if (rc != TVBF_OK) return rc;
  if (workspace == nullptr || workspace_bytes < sp.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, sp.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int* flagged = reinterpret_cast<int*>(ws + sp.off_flag);
  double* floors = reinterpret_cast<double*>(ws + sp.off_floor);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + sp.off_keys);
  TVBF_CUDA_OK(cudaMemsetAsync(out->stats, 0, 8 * sizeof(int32_t), st));
  const tvbf::ScoreParams scp = score_params(f, p);
  const int rows = p->row_end - p->row_begin;
  // table layout: [lists][table_rows][kp]
  const tvbf::CandLayout lay{p->row_begin - table_row0, 1, table_rows, cnt_all == nullptr ? 1 : 0};
  rc = tvbf::k5_launch(scp, static_cast<const uint2*>(cand_all), cnt_all, bound_all, lists, lay, sp.pl.kp,
                       p->row_begin, rows, *out, flagged, floors, st);
  if (rc != TVBF_OK) return rc;
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  return tvbf::k6_launch_flagged(scp, flagged, floors, rows, p->row_begin, keys, sms, *out, st);
}

// ---- append shows to a catalogue whose table exists --------------------------------------------
// The append sweep (K1 kMode 6) computes only the tiles that hold a new show and feeds both shows of
// every pair with at least one new show; K4s compacts the lists; K5 merges, per show, that list with
// the show's previous row (list 1, bound -inf) and certifies; K6 repairs over all columns.
namespace {

__global__ void append_changed_kernel(const int* prev_idx, const int* prev_cnt, const int* idx, const int* cnt,
                                      int n_old, int k, int* changed) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_old) return;
  int c = prev_cnt[r] != cnt[r];
  const size_t base = static_cast<size_t>(r) * k;
  for (int e = 0; e < k && !c; ++e) c = prev_idx[base + e] != idx[base + e];
  changed[r] = c;
}

// After K4s: an old show whose append list is empty received no new column above its threshold, which
// lies strictly below its previous k-th score (or below min_similarity for a short row), so no new
// column can enter and its row IS the previous row: copied, no rescoring.  Every other show (the new
// ones and the old ones with new candidates) is listed for K5.
__global__ void append_select_kernel(tvbf_topk_out prev, tvbf_topk_out out, const int* list0_cnt, int n_old, int n_shows,
                                     int k, int* rows, int* n_listed) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_shows) return;
  if (r >= n_old || list0_cnt[r] != 0) {
    rows[atomicAdd(n_listed, 1)] = r;
    return;
  }
  const size_t base = static_cast<size_t>(r) * k;
  for (int e = 0; e < k; ++e) {
    out.indices[base + e] = prev.indices[base + e];
    out.hybrid[base + e] = prev.hybrid[base + e];
    out.genre[base + e] = prev.genre[base + e];
    out.text[base + e] = prev.text[base + e];
    out.metadata[base + e] = prev.metadata[base + e];
  }
  out.counts[r] = prev.counts[r];
}

struct AppendPlan {
  Plan pl;             // a whole-catalogue symmetric job over all shows
  tvbf::K1Params geo;  // tile schedule of the append sweep
  int grid;
  size_t off_cand, off_cnt, off_bound;   // two candidate lists per show: [2][n_shows]
  size_t off_rows, off_listed, total;    // shows K5 rescores and their count
};

int make_append_plan(const tvbf_features* f, const tvbf_params* p, int n_old, AppendPlan* ap, tvbf_params* q) {
  TVBF_REQUIRE(n_old >= 1 && n_old < f->n_shows, "append: n_old %d must lie in [1, n_shows %d)", n_old, f->n_shows);
  TVBF_REQUIRE(!f->text_signed, "append: signed text needs the whole job");
  *q = *p;
  q->row_begin = 0;
  q->row_end = f->n_shows;
  q->tuning = (q->tuning & ~(0x3 << 20)) | (2 << 20);   // symmetric job (or fail if ineligible)
  q->tuning = (q->tuning & ~0xF) | 2;                   // CTA pairs
  int rc = validate_params(f, q);
  if (rc != TVBF_OK) return rc;
  rc = make_plan(f, q, &ap->pl);
  if (rc != TVBF_OK) return rc;
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  memset(&ap->geo, 0, sizeof(ap->geo));
  tvbf::k1_append_geometry(n_old, f->n_shows, sms / 2, &ap->geo);
  const int items = (ap->geo.rb_count + ap->geo.rb_per_group - 1) / ap->geo.rb_per_group * ap->geo.rb_per_group *
                    ap->geo.splits;
  ap->grid = 2 * (items < sms / 2 ? items : sms / 2);
  const size_t rows = static_cast<size_t>(f->n_shows);
  size_t off = ap->pl.total;
  ap->off_cand = off;  off = align_up(off + 2 * rows * ap->pl.kp * 8, 256);
  ap->off_cnt = off;   off = align_up(off + 2 * rows * 4, 256);
  ap->off_bound = off; off = align_up(off + 2 * rows * 4, 256);
  ap->off_rows = off;  off = align_up(off + rows * 4, 256);
  ap->off_listed = off; off = align_up(off + 4, 256);
  ap->total = off;
  return TVBF_OK;
}

// the candidate-kernel parameters of an append: a whole-catalogue symmetric job on the append geometry
int fill_append_params(const tvbf_features* f, const tvbf_params* q, const AppendPlan& ap, uint8_t* ws,
                       tvbf::K1Params* kp) {
  int rc = fill_k1_params(f, q, ap.pl, ws, kp);
  if (rc != TVBF_OK) return rc;
  kp->sync_kb = 0;
  kp->col_tiles = ap.geo.col_tiles;
  kp->rb_count = ap.geo.rb_count;
  kp->splits = ap.geo.splits;
  kp->rb_per_group = ap.geo.rb_per_group;
  kp->tiles_per_split = ap.geo.tiles_per_split;
  kp->append_n_old = ap.geo.append_n_old;
  kp->append_b0 = ap.geo.append_b0;
  kp->cand = reinterpret_cast<uint2*>(ws + ap.off_cand);   // list 0: what the append sweep found
  kp->cand_cnt = reinterpret_cast<int*>(ws + ap.off_cnt);
  kp->cand_theta = reinterpret_cast<float*>(ws + ap.off_bound);
  return TVBF_OK;
}

}  // namespace

size_t tvbf_append_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_old) {
  if (validate_features(f) != TVBF_OK || p == nullptr) return 0;
  AppendPlan ap;
  tvbf_params q;
  if (make_append_plan(f, p, n_old, &ap, &q) != TVBF_OK) return 0;
  return ap.total;
}

int tvbf_append_topk(const tvbf_features* f, const tvbf_params* p, int32_t n_old, const tvbf_topk_out* prev,
                     const tvbf_topk_out* out, int32_t* changed, void* workspace, size_t workspace_bytes,
                     void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p != nullptr, "params is NULL");
  TVBF_REQUIRE(prev && prev->indices && prev->counts && prev->hybrid && prev->genre && prev->text && prev->metadata,
               "previous table has NULL members");
  TVBF_REQUIRE(out && out->indices && out->counts && out->hybrid && out->genre && out->text && out->metadata &&
                   out->stats,
               "output table has NULL members");
  TVBF_REQUIRE(changed != nullptr && workspace != nullptr, "tvbf_append_topk: NULL argument");
  AppendPlan ap;
  tvbf_params q;
  rc = make_append_plan(f, p, n_old, &ap, &q);
  if (rc != TVBF_OK) return rc;
  if (workspace_bytes < ap.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, ap.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const Plan& pl = ap.pl;
  const int rows = f->n_shows;
  int* flagged = reinterpret_cast<int*>(ws + pl.off_flag);
  double* floors = reinterpret_cast<double*>(ws + pl.off_floor);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + pl.off_keys);
  int* listed_rows = reinterpret_cast<int*>(ws + ap.off_rows);
  int* n_listed = reinterpret_cast<int*>(ws + ap.off_listed);
  tvbf::K1Params kp;
  rc = fill_append_params(f, &q, ap, ws, &kp);
  if (rc != TVBF_OK) return rc;
  uint2* cand = kp.cand;
  int* cnt = kp.cand_cnt;
  float* bound = kp.cand_theta;
  const tvbf::AppendPrev pv{prev->indices, prev->counts, prev->hybrid, n_old, p->k,
                            cand + static_cast<size_t>(rows) * pl.kp, cnt + rows, bound + rows};
  TVBF_CUDA_OK(cudaMemsetAsync(out->stats, 0, 8 * sizeof(int32_t), st));
  rc = tvbf::k1_launch_append(f, kp, ap.grid, pv, st);
  if (rc != TVBF_OK) return rc;
  rc = tvbf::k4s_launch(kp, rows, st);
  if (rc != TVBF_OK) return rc;
  TVBF_CUDA_OK(cudaMemsetAsync(n_listed, 0, 4, st));
  append_select_kernel<<<(rows + 255) / 256, 256, 0, st>>>(*prev, *out, cnt, n_old, rows, p->k, listed_rows, n_listed);
  TVBF_LAUNCH_OK("append_select_kernel");
  const tvbf::ScoreParams sp = score_params(f, &q);
  const tvbf::CandLayout lay{0, 1, rows, 0};   // list s of show r: slot r + s * rows
  rc = tvbf::k5_launch_listed(sp, cand, cnt, bound, 2, lay, pl.kp, 0, rows, listed_rows, n_listed, *out, flagged,
                              floors, st);
  if (rc != TVBF_OK) return rc;
  rc = tvbf::k6_launch_flagged(sp, flagged, floors, rows, 0, keys, pl.k6_grid, *out, st);
  if (rc != TVBF_OK) return rc;
  append_changed_kernel<<<(n_old + 255) / 256, 256, 0, st>>>(prev->indices, prev->counts, out->indices, out->counts,
                                                             n_old, p->k, changed);
  TVBF_LAUNCH_OK("append_changed_kernel");
  return TVBF_OK;
}

int tvbf_append_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t n_old, int64_t* out2) {
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p && out2, "tvbf_append_plan_tiles: NULL argument");
  AppendPlan ap;
  tvbf_params q;
  rc = make_append_plan(f, p, n_old, &ap, &q);
  if (rc != TVBF_OK) return rc;
  uint8_t* fake_ws = reinterpret_cast<uint8_t*>(static_cast<uintptr_t>(4096));   // offsets only, never dereferenced
  tvbf::K1Params kp;
  rc = fill_append_params(f, &q, ap, fake_ws, &kp);
  if (rc != TVBF_OK) return rc;
  long long t[2];
  tvbf::k1_append_executed_tiles(f, kp, ap.grid, t);
  out2[0] = t[0];
  out2[1] = t[1];
  return TVBF_OK;
}

int32_t tvbf_debug_append_schedule(int32_t n_old, int32_t n_shows, int32_t sm_count, int32_t* out,
                                   int32_t max_items) {
  if (n_old < 1 || n_old >= n_shows || sm_count < 2 || out == nullptr || max_items < 0) {
    tvbf_set_error("tvbf_debug_append_schedule: bad arguments");
    return TVBF_ERR_INVALID;
  }
  tvbf::K1Params kp;
  memset(&kp, 0, sizeof(kp));
  tvbf::k1_append_geometry(n_old, n_shows, sm_count / 2, &kp);
  return tvbf::k1_debug_append_schedule(kp, out, max_items);
}

// ---- update the features of shows in a catalogue whose table exists ----------------------------
// The updated shows' operand rows are gathered into a [q_pad, k_pad] operand.  The update sweep (K1
// kMode 7) runs those rows against every column tile and offers each score to the row's show and to
// the column's show unless that one was updated too (it has a gathered row of its own): every ordered
// pair with an updated show reaches its list once.  K4s compacts the lists; K5 merges them with the
// previous rows minus the updated shows (list 1) under the rank cut; K6 repairs over all columns.
namespace {

__global__ void update_bits_kernel(const int* rows, int q, unsigned int* bits) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < q) atomicOr(bits + (rows[r] >> 5), 1u << (rows[r] & 31));
}

// dst row r = operand row rows[r] (r < q), zero for the padding rows up to q_pad
__global__ void update_gather_kernel(const uint4* operand, const int* rows, int q, int q_pad, int row_vec,
                                     uint4* dst) {
  const size_t n = static_cast<size_t>(q_pad) * row_vec;
  for (size_t e = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; e < n;
       e += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(e / row_vec), c = static_cast<int>(e % row_vec);
    dst[e] = r < q ? operand[static_cast<size_t>(rows[r]) * row_vec + c] : make_uint4(0u, 0u, 0u, 0u);
  }
}

// After K4s: a show that was not updated, received no candidate from an updated one above its threshold
// (strictly below its previous k-th score, or below min_similarity for a short row) and names no
// updated show in its previous row keeps that row: the scores of all its other columns are unchanged.
// It is copied, no rescoring.  Every other show is listed for K5.
__global__ void update_select_kernel(tvbf_topk_out prev, tvbf_topk_out out, const int* list0_cnt,
                                     const unsigned int* bits, int n_shows, int k, int* rows, int* n_listed) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_shows) return;
  const size_t base = static_cast<size_t>(r) * k;
  bool listed = ((bits[r >> 5] >> (r & 31)) & 1u) != 0u || list0_cnt[r] != 0;
  for (int e = 0; e < prev.counts[r] && !listed; ++e) {
    const int j = prev.indices[base + e];
    listed = ((bits[j >> 5] >> (j & 31)) & 1u) != 0u;
  }
  if (listed) {
    rows[atomicAdd(n_listed, 1)] = r;
    return;
  }
  for (int e = 0; e < k; ++e) {
    out.indices[base + e] = prev.indices[base + e];
    out.hybrid[base + e] = prev.hybrid[base + e];
    out.genre[base + e] = prev.genre[base + e];
    out.text[base + e] = prev.text[base + e];
    out.metadata[base + e] = prev.metadata[base + e];
  }
  out.counts[r] = prev.counts[r];
}

__device__ __forceinline__ bool same_bits(double a, double b) { return __double_as_longlong(a) == __double_as_longlong(b); }

// changed[r] = 1 when row r differs from the previous row in any of the six fields (bit for bit)
__global__ void update_changed_kernel(tvbf_topk_out prev, tvbf_topk_out out, int n_shows, int k, int* changed) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_shows) return;
  int c = prev.counts[r] != out.counts[r];
  const size_t base = static_cast<size_t>(r) * k;
  for (int e = 0; e < k && !c; ++e)
    c = prev.indices[base + e] != out.indices[base + e] || !same_bits(prev.hybrid[base + e], out.hybrid[base + e]) ||
        !same_bits(prev.genre[base + e], out.genre[base + e]) || !same_bits(prev.text[base + e], out.text[base + e]) ||
        !same_bits(prev.metadata[base + e], out.metadata[base + e]);
  changed[r] = c;
}

struct UpdatePlan {
  Plan pl;             // a whole-catalogue symmetric job over all shows
  tvbf::K1Params geo;  // tile schedule of the update sweep
  int grid, q_pad;
  size_t off_cand, off_cnt, off_bound;   // two candidate lists per show: [2][n_shows]
  size_t off_rows, off_listed;           // shows K5 rescores and their count
  size_t off_gather, off_bits, off_cut_s, off_cut_j, total;
};

int make_update_plan(const tvbf_features* f, const tvbf_params* p, int n_rows, UpdatePlan* up, tvbf_params* q) {
  TVBF_REQUIRE(n_rows >= 1 && n_rows <= f->n_shows, "update: %d rows outside [1, n_shows %d]", n_rows, f->n_shows);
  TVBF_REQUIRE(!f->text_signed, "update: signed text needs the whole job");
  *q = *p;
  q->row_begin = 0;
  q->row_end = f->n_shows;
  q->tuning = (q->tuning & ~(0x3 << 20)) | (2 << 20);   // symmetric job (or fail if ineligible)
  q->tuning = (q->tuning & ~0xF) | 2;                   // CTA pairs
  int rc = validate_params(f, q);
  if (rc != TVBF_OK) return rc;
  rc = make_plan(f, q, &up->pl);
  if (rc != TVBF_OK) return rc;
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  memset(&up->geo, 0, sizeof(up->geo));
  tvbf::k1_update_geometry(n_rows, f->n_shows, sms / 2, &up->geo);
  const int items = (up->geo.rb_count + up->geo.rb_per_group - 1) / up->geo.rb_per_group * up->geo.rb_per_group *
                    up->geo.splits;
  up->grid = 2 * (items < sms / 2 ? items : sms / 2);
  up->q_pad = up->geo.rb_count * 256;
  const size_t rows = static_cast<size_t>(f->n_shows);
  size_t off = up->pl.total;
  up->off_cand = off;   off = align_up(off + 2 * rows * up->pl.kp * 8, 256);
  up->off_cnt = off;    off = align_up(off + 2 * rows * 4, 256);
  up->off_bound = off;  off = align_up(off + 2 * rows * 4, 256);
  up->off_rows = off;   off = align_up(off + rows * 4, 256);
  up->off_listed = off; off = align_up(off + 4, 256);
  up->off_gather = off; off = align_up(off + static_cast<size_t>(up->q_pad) * f->k_pad * 2, 256);
  up->off_bits = off;   off = align_up(off + static_cast<size_t>(f->n_pad) / 32 * 4, 256);
  up->off_cut_s = off;  off = align_up(off + rows * 8, 256);
  up->off_cut_j = off;  off = align_up(off + rows * 4, 256);
  up->total = off;
  return TVBF_OK;
}

// the candidate-kernel parameters of an update: a whole-catalogue symmetric job on the update geometry
int fill_update_params(const tvbf_features* f, const tvbf_params* q, const UpdatePlan& up, uint8_t* ws,
                       const int* rows, int n_rows, tvbf::K1Params* kp) {
  int rc = fill_k1_params(f, q, up.pl, ws, kp);
  if (rc != TVBF_OK) return rc;
  kp->sync_kb = 0;
  kp->sym = 0;   // the one-sided schedule: a rectangle (the epilogue of kMode 7 still feeds both lists)
  // 8 epilogue warps whatever the vocabulary: the 16-warp epilogue spills under its register cap, and
  // the sweep covers few tiles
  kp->wide_epilogue = 0;
  kp->col_tiles = up.geo.col_tiles;
  kp->rb_count = up.geo.rb_count;
  kp->splits = up.geo.splits;
  kp->rb_per_group = up.geo.rb_per_group;
  kp->tiles_per_split = up.geo.tiles_per_split;
  kp->upd_rows = rows;
  kp->upd_q = n_rows;
  kp->upd_bits = reinterpret_cast<const unsigned int*>(ws + up.off_bits);
  kp->cand = reinterpret_cast<uint2*>(ws + up.off_cand);   // list 0: what the update sweep found
  kp->cand_cnt = reinterpret_cast<int*>(ws + up.off_cnt);
  kp->cand_theta = reinterpret_cast<float*>(ws + up.off_bound);
  return TVBF_OK;
}

}  // namespace

size_t tvbf_update_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_rows) {
  if (validate_features(f) != TVBF_OK || p == nullptr) return 0;
  UpdatePlan up;
  tvbf_params q;
  if (make_update_plan(f, p, n_rows, &up, &q) != TVBF_OK) return 0;
  return up.total;
}

int tvbf_update_topk(const tvbf_features* f, const tvbf_params* p, const int32_t* rows, int32_t n_rows,
                     const tvbf_topk_out* prev, const tvbf_topk_out* out, int32_t* changed, void* workspace,
                     size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p != nullptr, "params is NULL");
  TVBF_REQUIRE(prev && prev->indices && prev->counts && prev->hybrid && prev->genre && prev->text && prev->metadata,
               "previous table has NULL members");
  TVBF_REQUIRE(out && out->indices && out->counts && out->hybrid && out->genre && out->text && out->metadata &&
                   out->stats,
               "output table has NULL members");
  TVBF_REQUIRE(rows != nullptr && changed != nullptr && workspace != nullptr, "tvbf_update_topk: NULL argument");
  UpdatePlan up;
  tvbf_params q;
  rc = make_update_plan(f, p, n_rows, &up, &q);
  if (rc != TVBF_OK) return rc;
  if (workspace_bytes < up.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, up.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const Plan& pl = up.pl;
  const int n = f->n_shows;
  int* flagged = reinterpret_cast<int*>(ws + pl.off_flag);
  double* floors = reinterpret_cast<double*>(ws + pl.off_floor);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + pl.off_keys);
  int* listed_rows = reinterpret_cast<int*>(ws + up.off_rows);
  int* n_listed = reinterpret_cast<int*>(ws + up.off_listed);
  unsigned int* bits = reinterpret_cast<unsigned int*>(ws + up.off_bits);
  double* cut_s = reinterpret_cast<double*>(ws + up.off_cut_s);
  int* cut_j = reinterpret_cast<int*>(ws + up.off_cut_j);
  tvbf::K1Params kp;
  rc = fill_update_params(f, &q, up, ws, rows, n_rows, &kp);
  if (rc != TVBF_OK) return rc;
  TVBF_CUDA_OK(cudaMemsetAsync(bits, 0, static_cast<size_t>(f->n_pad) / 32 * 4, st));
  update_bits_kernel<<<(n_rows + 255) / 256, 256, 0, st>>>(rows, n_rows, bits);
  TVBF_LAUNCH_OK("update_bits_kernel");
  const int row_vec = f->k_pad / 8;   // 16-byte vectors per operand row
  update_gather_kernel<<<1024, 256, 0, st>>>(static_cast<const uint4*>(f->operand), rows, n_rows, up.q_pad, row_vec,
                                             reinterpret_cast<uint4*>(ws + up.off_gather));
  TVBF_LAUNCH_OK("update_gather_kernel");
  tvbf_features g = *f;   // the gathered rows as the A operand
  g.operand = ws + up.off_gather;
  g.n_pad = up.q_pad;
  uint2* cand = kp.cand;
  int* cnt = kp.cand_cnt;
  float* bound = kp.cand_theta;
  const tvbf::UpdatePrev pv{prev->indices, prev->counts, prev->hybrid, p->k, bits,
                            cand + static_cast<size_t>(n) * pl.kp, cnt + n, bound + n, cut_s, cut_j};
  TVBF_CUDA_OK(cudaMemsetAsync(out->stats, 0, 8 * sizeof(int32_t), st));
  rc = tvbf::k1_launch_update(f, &g, kp, up.grid, pv, st);
  if (rc != TVBF_OK) return rc;
  rc = tvbf::k4s_launch(kp, n, st);
  if (rc != TVBF_OK) return rc;
  TVBF_CUDA_OK(cudaMemsetAsync(n_listed, 0, 4, st));
  update_select_kernel<<<(n + 255) / 256, 256, 0, st>>>(*prev, *out, cnt, bits, n, p->k, listed_rows, n_listed);
  TVBF_LAUNCH_OK("update_select_kernel");
  const tvbf::ScoreParams sp = score_params(f, &q);
  const tvbf::CandLayout lay{0, 1, n, 0};   // list s of show r: slot r + s * n
  rc = tvbf::k5_launch_listed(sp, cand, cnt, bound, 2, lay, pl.kp, 0, n, listed_rows, n_listed, *out, flagged, floors,
                              st, cut_s, cut_j);
  if (rc != TVBF_OK) return rc;
  rc = tvbf::k6_launch_flagged(sp, flagged, floors, n, 0, keys, pl.k6_grid, *out, st);
  if (rc != TVBF_OK) return rc;
  update_changed_kernel<<<(n + 255) / 256, 256, 0, st>>>(*prev, *out, n, p->k, changed);
  TVBF_LAUNCH_OK("update_changed_kernel");
  return TVBF_OK;
}

int tvbf_update_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t n_rows, int64_t* out2) {
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p && out2, "tvbf_update_plan_tiles: NULL argument");
  UpdatePlan up;
  tvbf_params q;
  rc = make_update_plan(f, p, n_rows, &up, &q);
  if (rc != TVBF_OK) return rc;
  uint8_t* fake_ws = reinterpret_cast<uint8_t*>(static_cast<uintptr_t>(4096));   // offsets only, never dereferenced
  tvbf::K1Params kp;
  rc = fill_update_params(f, &q, up, fake_ws, nullptr, n_rows, &kp);
  if (rc != TVBF_OK) return rc;
  long long t[2];
  tvbf::k1_update_executed_tiles(kp, up.grid, t);
  out2[0] = t[0];
  out2[1] = t[1];
  return TVBF_OK;
}

int32_t tvbf_debug_update_schedule(int32_t q, int32_t n_shows, int32_t sm_count, int32_t* out, int32_t max_items) {
  if (q < 1 || q > n_shows || sm_count < 2 || out == nullptr || max_items < 0) {
    tvbf_set_error("tvbf_debug_update_schedule: bad arguments");
    return TVBF_ERR_INVALID;
  }
  tvbf::K1Params kp;
  memset(&kp, 0, sizeof(kp));
  tvbf::k1_update_geometry(q, n_shows, sm_count / 2, &kp);
  return tvbf::k1_debug_schedule(kp, out, max_items);
}

// ---- remove shows from a catalogue whose table exists -------------------------------------------
// No pair score changes.  A remaining show whose previous row names no removed show keeps that row with
// its indices renumbered: removing columns cannot bring a new one in.  The other remaining shows (A)
// are swept against every column as gathered rows (K1 kMode 9: each score goes to the gathered row's
// own list only), compacted (K4s over |A| lists), rescored (K5 on those lists alone, plain
// certificate) and repaired (K6).
namespace {

// map[o] = new row of old row o, or -1 when o is removed (removed: sorted, distinct)
__global__ void remove_map_kernel(const int* removed, int q, int n_old, int* map) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_old) return;
  int lo = 0, hi = q;   // removed rows below o
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (removed[mid] < o) lo = mid + 1;
    else hi = mid;
  }
  map[o] = lo < q && removed[lo] == o ? -1 : o - lo;
}

// Remaining old row o becomes new row r = map[o].  in_a[r] = 1 when its previous row names a removed
// show (row r is in A, K5 and K6 write it); otherwise the previous row is copied with its indices
// renumbered, the -1 padding and the scores as they are.
__global__ void remove_rows_kernel(tvbf_topk_out prev, tvbf_topk_out out, const int* map, int n_old, int k,
                                   int* in_a) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_old) return;
  const int r = map[o];
  if (r < 0) return;
  const int n = prev.counts[o];
  const size_t src = static_cast<size_t>(o) * k, dst = static_cast<size_t>(r) * k;
  bool named = false;
  for (int e = 0; e < n && !named; ++e) named = map[prev.indices[src + e]] < 0;
  in_a[r] = named;
  if (named) return;
  for (int e = 0; e < k; ++e) {
    const int j = prev.indices[src + e];
    out.indices[dst + e] = e < n ? map[j] : j;
    out.hybrid[dst + e] = prev.hybrid[src + e];
    out.genre[dst + e] = prev.genre[src + e];
    out.text[dst + e] = prev.text[src + e];
    out.metadata[dst + e] = prev.metadata[src + e];
  }
  out.counts[r] = n;
}

// rows[0 .. *n_rows) = the rows r with in_a[r] = 1, ascending (one block: a chunk per thread, then a
// scan of the chunk counts)
constexpr int kCompactThreads = 1024;
__global__ void __launch_bounds__(kCompactThreads) remove_compact_kernel(const int* in_a, int n, int* rows,
                                                                          int* n_rows) {
  __shared__ int sums[kCompactThreads];
  const int t = threadIdx.x;
  const int chunk = (n + kCompactThreads - 1) / kCompactThreads;
  const int b = min(n, t * chunk), e = min(n, b + chunk);
  int c = 0;
  for (int r = b; r < e; ++r) c += in_a[r] != 0;
  sums[t] = c;
  __syncthreads();
  for (int off = 1; off < kCompactThreads; off <<= 1) {   // inclusive scan
    const int v = t >= off ? sums[t - off] : 0;
    __syncthreads();
    sums[t] += v;
    __syncthreads();
  }
  int pos = sums[t] - c;
  for (int r = b; r < e; ++r)
    if (in_a[r] != 0) rows[pos++] = r;
  if (t == kCompactThreads - 1) *n_rows = sums[t];
}

struct RemovePlan {
  Plan pl;             // a whole-catalogue symmetric job over the remaining shows
  tvbf::K1Params geo;  // tile schedule of the repair sweep (the update geometry over |A| gathered rows)
  int grid, q_pad;
  size_t off_map, off_in_a, off_rows, off_count, off_gather, off_gtheta, total;
};

// n_a: rows of A (the geometry of the sweep; 0 sizes the workspace only, which holds |A| up to every
// remaining show)
int make_remove_plan(const tvbf_features* f, const tvbf_params* p, int n_removed, int n_a, RemovePlan* rp,
                     tvbf_params* q) {
  TVBF_REQUIRE(n_removed >= 1 && n_removed <= INT32_MAX - f->n_shows, "remove: %d removed shows", n_removed);
  TVBF_REQUIRE(n_a >= 0 && n_a <= f->n_shows, "remove: %d repaired rows outside [0, n_shows %d]", n_a, f->n_shows);
  TVBF_REQUIRE(!f->text_signed, "remove: signed text needs the whole job");
  *q = *p;
  q->row_begin = 0;
  q->row_end = f->n_shows;
  q->tuning = (q->tuning & ~(0x3 << 20)) | (2 << 20);   // symmetric job (or fail if ineligible)
  q->tuning = (q->tuning & ~0xF) | 2;                   // CTA pairs
  int rc = validate_params(f, q);
  if (rc != TVBF_OK) return rc;
  rc = make_plan(f, q, &rp->pl);
  if (rc != TVBF_OK) return rc;
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  memset(&rp->geo, 0, sizeof(rp->geo));
  rp->grid = 0;
  rp->q_pad = 0;
  if (n_a > 0) {
    tvbf::k1_update_geometry(n_a, f->n_shows, sms / 2, &rp->geo);
    const int items = (rp->geo.rb_count + rp->geo.rb_per_group - 1) / rp->geo.rb_per_group * rp->geo.rb_per_group *
                      rp->geo.splits;
    rp->grid = 2 * (items < sms / 2 ? items : sms / 2);
    rp->q_pad = rp->geo.rb_count * 256;
  }
  const size_t rows = static_cast<size_t>(f->n_shows);
  size_t off = rp->pl.total;
  rp->off_map = off;    off = align_up(off + (rows + n_removed) * 4, 256);
  rp->off_in_a = off;   off = align_up(off + rows * 4, 256);
  rp->off_rows = off;   off = align_up(off + rows * 4, 256);
  rp->off_count = off;  off = align_up(off + 4, 256);
  rp->off_gather = off; off = align_up(off + static_cast<size_t>(f->n_pad) * f->k_pad * 2, 256);
  rp->off_gtheta = off; off = align_up(off + static_cast<size_t>(f->n_pad) * 4, 256);
  rp->total = off;
  return TVBF_OK;
}

// the candidate-kernel parameters of the repair sweep: a whole-catalogue symmetric job on the update
// geometry, one list per gathered row (the plan's lists and candidate table, indexed by gathered row)
int fill_remove_params(const tvbf_features* f, const tvbf_params* q, const RemovePlan& rp, uint8_t* ws,
                       const int* rows, int n_a, tvbf::K1Params* kp) {
  int rc = fill_k1_params(f, q, rp.pl, ws, kp);
  if (rc != TVBF_OK) return rc;
  kp->sync_kb = 0;
  kp->sym = 0;   // the one-sided schedule: a rectangle
  kp->wide_epilogue = 0;   // 8 epilogue warps, as the update sweep
  kp->col_tiles = rp.geo.col_tiles;
  kp->rb_count = rp.geo.rb_count;
  kp->splits = rp.geo.splits;
  kp->rb_per_group = rp.geo.rb_per_group;
  kp->tiles_per_split = rp.geo.tiles_per_split;
  kp->upd_rows = rows;
  kp->upd_q = n_a;
  kp->upd_bits = nullptr;
  return TVBF_OK;
}

}  // namespace

size_t tvbf_remove_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_removed) {
  if (validate_features(f) != TVBF_OK || p == nullptr) return 0;
  RemovePlan rp;
  tvbf_params q;
  if (make_remove_plan(f, p, n_removed, 0, &rp, &q) != TVBF_OK) return 0;
  return rp.total;
}

int tvbf_remove_topk(const tvbf_features* f, const tvbf_params* p, const int32_t* removed, int32_t n_removed,
                     const tvbf_topk_out* prev, const tvbf_topk_out* out, int32_t* changed, void* workspace,
                     size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p != nullptr, "params is NULL");
  TVBF_REQUIRE(prev && prev->indices && prev->counts && prev->hybrid && prev->genre && prev->text && prev->metadata,
               "previous table has NULL members");
  TVBF_REQUIRE(out && out->indices && out->counts && out->hybrid && out->genre && out->text && out->metadata &&
                   out->stats,
               "output table has NULL members");
  TVBF_REQUIRE(removed != nullptr && changed != nullptr && workspace != nullptr, "tvbf_remove_topk: NULL argument");
  RemovePlan rp;
  tvbf_params q;
  rc = make_remove_plan(f, p, n_removed, 0, &rp, &q);
  if (rc != TVBF_OK) return rc;
  if (workspace_bytes < rp.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, rp.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const int n = f->n_shows, n_old = n + n_removed;
  int* map = reinterpret_cast<int*>(ws + rp.off_map);
  int* in_a = reinterpret_cast<int*>(ws + rp.off_in_a);
  int* a_rows = reinterpret_cast<int*>(ws + rp.off_rows);
  int* a_count = reinterpret_cast<int*>(ws + rp.off_count);
  TVBF_CUDA_OK(cudaMemsetAsync(out->stats, 0, 8 * sizeof(int32_t), st));
  remove_map_kernel<<<(n_old + 255) / 256, 256, 0, st>>>(removed, n_removed, n_old, map);
  TVBF_LAUNCH_OK("remove_map_kernel");
  remove_rows_kernel<<<(n_old + 255) / 256, 256, 0, st>>>(*prev, *out, map, n_old, p->k, in_a);
  TVBF_LAUNCH_OK("remove_rows_kernel");
  remove_compact_kernel<<<1, kCompactThreads, 0, st>>>(in_a, n, a_rows, a_count);
  TVBF_LAUNCH_OK("remove_compact_kernel");
  TVBF_CUDA_OK(cudaMemcpyAsync(changed, in_a, static_cast<size_t>(n) * 4, cudaMemcpyDeviceToDevice, st));
  // the sweep's geometry depends on |A|
  int n_a = 0;
  TVBF_CUDA_OK(cudaMemcpyAsync(&n_a, a_count, 4, cudaMemcpyDeviceToHost, st));
  TVBF_CUDA_OK(cudaStreamSynchronize(st));
  if (n_a == 0) return TVBF_OK;
  rc = make_remove_plan(f, p, n_removed, n_a, &rp, &q);
  if (rc != TVBF_OK) return rc;
  const Plan& pl = rp.pl;
  tvbf::K1Params kp;
  rc = fill_remove_params(f, &q, rp, ws, a_rows, n_a, &kp);
  if (rc != TVBF_OK) return rc;
  const int row_vec = f->k_pad / 8;   // 16-byte vectors per operand row
  update_gather_kernel<<<1024, 256, 0, st>>>(static_cast<const uint4*>(f->operand), a_rows, n_a, rp.q_pad, row_vec,
                                             reinterpret_cast<uint4*>(ws + rp.off_gather));
  TVBF_LAUNCH_OK("update_gather_kernel");
  tvbf_features g = *f;   // the gathered rows as the A operand
  g.operand = ws + rp.off_gather;
  g.n_pad = rp.q_pad;
  unsigned int* gtheta = reinterpret_cast<unsigned int*>(ws + rp.off_gtheta);
  rc = tvbf::k1_launch_remove(f, &g, kp, rp.grid, gtheta, st);
  if (rc != TVBF_OK) return rc;
  kp.g_theta = gtheta;   // K4s: the gathered rows' lists under their thresholds
  rc = tvbf::k4s_launch(kp, n_a, st);
  if (rc != TVBF_OK) return rc;
  const tvbf::ScoreParams sp = score_params(f, &q);
  const tvbf::CandLayout lay{0, 1, 0, 0, 1};   // the list of rows[e] is slot e
  int* flagged = reinterpret_cast<int*>(ws + pl.off_flag);
  double* floors = reinterpret_cast<double*>(ws + pl.off_floor);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + pl.off_keys);
  rc = tvbf::k5_launch_listed(sp, kp.cand, kp.cand_cnt, kp.cand_theta, 1, lay, pl.kp, 0, n, a_rows, a_count, *out,
                              flagged, floors, st);
  if (rc != TVBF_OK) return rc;
  return tvbf::k6_launch_flagged(sp, flagged, floors, n, 0, keys, pl.k6_grid, *out, st);
}

int tvbf_remove_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t n_rows, int64_t* out2) {
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p && out2, "tvbf_remove_plan_tiles: NULL argument");
  TVBF_REQUIRE(n_rows >= 1, "tvbf_remove_plan_tiles: %d repaired rows", n_rows);
  RemovePlan rp;
  tvbf_params q;
  rc = make_remove_plan(f, p, 1, n_rows, &rp, &q);
  if (rc != TVBF_OK) return rc;
  uint8_t* fake_ws = reinterpret_cast<uint8_t*>(static_cast<uintptr_t>(4096));   // offsets only, never dereferenced
  tvbf::K1Params kp;
  rc = fill_remove_params(f, &q, rp, fake_ws, nullptr, n_rows, &kp);
  if (rc != TVBF_OK) return rc;
  long long t[2];
  tvbf::k1_update_executed_tiles(kp, rp.grid, t);
  out2[0] = t[0];
  out2[1] = t[1];
  return TVBF_OK;
}

// ---- refresh a catalogue whose table exists: removed, updated and appended shows in one call ------
// New numbering: the remaining shows in their old order, then the appended ones.  S = updated and
// appended shows (their pair scores changed or are new); A = the other remaining shows whose previous
// row names a removed show; G = S + A.  Stage 1 sweeps the gathered rows of G against every column (K1
// kMode 10): a row of G scores its whole row into its own list, and a row of S also offers each score to
// the column's list unless that column is in G.  A show outside G merges the renumbered previous row T'
// without S (list 1, with the rank cut at its previous k-th entry) with what S offered it (list 0); one
// that was offered nothing and names no show of S in T' keeps T'.  K5 rescores the rest.  Stage 2
// repairs the rows outside G that K5 rejects -- mostly rows that lost a neighbour of S below their
// previous k-th entry, which no list can refill -- on the tensor cores as the removal repairs A (kMode 8
// seed, kMode 9 sweep, K5 on the gathered lists).  K6 takes the rows of G that K5 rejects (tie plateaus,
// overflowed lists: a second sweep would reject them again) and what stage 2 rejects.
namespace {

// S bits: the new rows of the updated shows (old rows updated[0 .. n_upd)) and of the n_app appended ones
__global__ void refresh_sbits_kernel(const int* updated, int n_upd, const int* map, int n, int n_app,
                                     unsigned int* s_bits) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_upd + n_app) return;
  const int r = t < n_upd ? map[updated[t]] : n - n_app + (t - n_upd);
  atomicOr(s_bits + (r >> 5), 1u << (r & 31));
}

// Thread t < n_old: old row t, remaining as new row r = map[t]; thread n_old + a: appended new row
// n - n_app + a.  old_row[r] = its old row (-1 appended); in_g[r] = 1 and the G bit for S and for a
// remaining show whose previous row names a removed show (A).
__global__ void refresh_rows_kernel(tvbf_topk_out prev, const int* map, int n_old, int n, int n_app, int k,
                                    const unsigned int* s_bits, int* old_row, int* in_g, unsigned int* g_bits) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_old + n_app) return;
  int r = n - n_app + (t - n_old), o = -1;
  bool g = true;
  if (t < n_old) {
    o = t;
    r = map[o];
    if (r < 0) return;
    g = ((s_bits[r >> 5] >> (r & 31)) & 1u) != 0u;
    const int c = prev.counts[o];
    const size_t src = static_cast<size_t>(o) * k;
    for (int e = 0; e < c && !g; ++e) g = map[prev.indices[src + e]] < 0;
  }
  old_row[r] = o;
  in_g[r] = g;
  if (g) atomicOr(g_bits + (r >> 5), 1u << (r & 31));
}

__device__ __forceinline__ bool refresh_bit(const unsigned int* bits, int j) { return ((bits[j >> 5] >> (j & 31)) & 1u) != 0u; }

// After K4s: a show outside G that received no candidate from S above its threshold and whose T' names no
// show of S keeps T' (the scores of all its columns are unchanged): copied with the indices renumbered,
// no rescoring.  Every other show is listed for K5.
__global__ void refresh_select_kernel(tvbf_topk_out prev, tvbf_topk_out out, const int* list0_cnt, const int* map,
                                      const int* old_row, const unsigned int* s_bits, const unsigned int* g_bits,
                                      int n, int k, int* rows, int* n_listed) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  bool listed = refresh_bit(g_bits, r) || list0_cnt[r] != 0;
  const int o = old_row[r];
  const size_t src = static_cast<size_t>(o) * k, dst = static_cast<size_t>(r) * k;
  const int c = listed ? 0 : prev.counts[o];
  for (int e = 0; e < c && !listed; ++e) listed = refresh_bit(s_bits, map[prev.indices[src + e]]);
  if (listed) {
    rows[atomicAdd(n_listed, 1)] = r;
    return;
  }
  for (int e = 0; e < k; ++e) {
    const int j = prev.indices[src + e];
    out.indices[dst + e] = e < c ? map[j] : j;
    out.hybrid[dst + e] = prev.hybrid[src + e];
    out.genre[dst + e] = prev.genre[src + e];
    out.text[dst + e] = prev.text[src + e];
    out.metadata[dst + e] = prev.metadata[src + e];
  }
  out.counts[r] = c;
}

// After K5 (one block): of the rows K5 flagged, those in G move to the second flagged arrays (flag2 /
// floor2, counts c2[2] / c2[3], with text at the front as K5 lays them out) for K6; the others are marked
// in in2 for the second sweep, leave stats[0] (they are not the exact kernel's) and are counted in
// stats[5].  The first flagged arrays are then empty for the K5 of the second stage.
constexpr int kSplitThreads = 1024;
__global__ void __launch_bounds__(kSplitThreads) refresh_split_kernel(const int* flagged, const double* floors,
                                                                       const unsigned int* g_bits, int n, int* stats,
                                                                       int* in2, int* flag2, double* floor2, int* c2) {
  __shared__ int front, back, moved;
  if (threadIdx.x == 0) front = back = moved = 0;
  const int n_front = stats[2], n_back = stats[3];
  __syncthreads();
  for (int i = threadIdx.x; i < n_front + n_back; i += kSplitThreads) {
    const int pos = i < n_front ? i : n - 1 - (i - n_front);
    const int r = flagged[pos];
    if (refresh_bit(g_bits, r)) {
      const int at = i < n_front ? atomicAdd(&front, 1) : n - 1 - atomicAdd(&back, 1);
      flag2[at] = r;
      floor2[at] = floors[pos];
    } else {
      in2[r] = 1;
      atomicAdd(&moved, 1);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    c2[2] = front;
    c2[3] = back;
    stats[0] -= moved;
    stats[2] = 0;
    stats[3] = 0;
    stats[5] = moved;
  }
}

// changed[r] = 1 for an appended row and for a row that differs from T'_r in any of the six fields (bit
// for bit)
__global__ void refresh_changed_kernel(tvbf_topk_out prev, tvbf_topk_out out, const int* map, const int* old_row,
                                       int n, int k, int* changed) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int o = old_row[r];
  if (o < 0) {
    changed[r] = 1;
    return;
  }
  const int cnt = prev.counts[o];
  int c = cnt != out.counts[r];
  const size_t src = static_cast<size_t>(o) * k, dst = static_cast<size_t>(r) * k;
  for (int e = 0; e < k && !c; ++e) {
    const int j = prev.indices[src + e];
    c = (e < cnt ? map[j] : j) != out.indices[dst + e] || !same_bits(prev.hybrid[src + e], out.hybrid[dst + e]) ||
        !same_bits(prev.genre[src + e], out.genre[dst + e]) || !same_bits(prev.text[src + e], out.text[dst + e]) ||
        !same_bits(prev.metadata[src + e], out.metadata[dst + e]);
  }
  changed[r] = c;
}

struct RefreshPlan {
  Plan pl;                // a whole-catalogue symmetric job over the shows after the refresh
  tvbf::K1Params geo[2];  // tile schedules of the refresh sweep (|G| rows) and the repair sweep (stage 2)
  int grid[2], q_pad[2];
  size_t off_cand, off_cnt, off_bound;   // stage 1: two candidate lists per show, [2][n_shows]
  size_t off_rows, off_listed;           // shows K5 rescores and their count
  size_t off_gather;                     // gathered operand rows of either stage: [n_pad, k_pad]
  size_t off_sbits, off_gbits, off_cut_s, off_cut_j, off_map, off_old_row, off_in_g, off_grows, off_gcount;
  size_t off_in2, off_rows2, off_count2, off_flag2, off_floor2, off_c2, off_gtheta2, total;
};

int refresh_counts_ok(const tvbf_features* f, int n_removed, int n_updated, int n_appended) {
  TVBF_REQUIRE(n_removed >= 0 && n_updated >= 0 && n_appended >= 0, "refresh: negative count (%d, %d, %d)",
               n_removed, n_updated, n_appended);
  TVBF_REQUIRE(n_appended < f->n_shows && n_updated <= f->n_shows - n_appended,
               "refresh: %d updated and %d appended shows in a catalogue of %d (at least one show must remain)",
               n_updated, n_appended, f->n_shows);
  TVBF_REQUIRE(n_removed <= INT32_MAX - f->n_shows, "refresh: %d removed shows", n_removed);
  return TVBF_OK;
}

// n_rows[0] = |G|, n_rows[1] = rows of the second stage (the sweep geometries; 0 sizes the workspace
// only, which holds either up to every show)
int make_refresh_plan(const tvbf_features* f, const tvbf_params* p, int n_removed, int n_updated, int n_appended,
                      const int* n_rows, RefreshPlan* rp, tvbf_params* q) {
  int rc = refresh_counts_ok(f, n_removed, n_updated, n_appended);
  if (rc != TVBF_OK) return rc;
  for (int s = 0; s < 2; ++s)
    TVBF_REQUIRE(n_rows[s] >= 0 && n_rows[s] <= f->n_shows, "refresh: %d swept rows outside [0, n_shows %d]",
                 n_rows[s], f->n_shows);
  TVBF_REQUIRE(!f->text_signed, "refresh: signed text needs the whole job");
  *q = *p;
  q->row_begin = 0;
  q->row_end = f->n_shows;
  q->tuning = (q->tuning & ~(0x3 << 20)) | (2 << 20);   // symmetric job (or fail if ineligible)
  q->tuning = (q->tuning & ~0xF) | 2;                   // CTA pairs
  rc = validate_params(f, q);
  if (rc != TVBF_OK) return rc;
  rc = make_plan(f, q, &rp->pl);
  if (rc != TVBF_OK) return rc;
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  for (int s = 0; s < 2; ++s) {
    memset(&rp->geo[s], 0, sizeof(rp->geo[s]));
    rp->grid[s] = 0;
    rp->q_pad[s] = 0;
    if (n_rows[s] == 0) continue;
    tvbf::k1_update_geometry(n_rows[s], f->n_shows, sms / 2, &rp->geo[s]);
    const tvbf::K1Params& g = rp->geo[s];
    const int items = (g.rb_count + g.rb_per_group - 1) / g.rb_per_group * g.rb_per_group * g.splits;
    rp->grid[s] = 2 * (items < sms / 2 ? items : sms / 2);
    rp->q_pad[s] = g.rb_count * 256;
  }
  const size_t rows = static_cast<size_t>(f->n_shows);
  const size_t words = static_cast<size_t>(f->n_pad) / 32 * 4;
  size_t off = rp->pl.total;
  rp->off_cand = off;    off = align_up(off + 2 * rows * rp->pl.kp * 8, 256);
  rp->off_cnt = off;     off = align_up(off + 2 * rows * 4, 256);
  rp->off_bound = off;   off = align_up(off + 2 * rows * 4, 256);
  rp->off_rows = off;    off = align_up(off + rows * 4, 256);
  rp->off_listed = off;  off = align_up(off + 4, 256);
  rp->off_gather = off;  off = align_up(off + static_cast<size_t>(f->n_pad) * f->k_pad * 2, 256);
  rp->off_sbits = off;   off = align_up(off + words, 256);
  rp->off_gbits = off;   off = align_up(off + words, 256);
  rp->off_cut_s = off;   off = align_up(off + rows * 8, 256);
  rp->off_cut_j = off;   off = align_up(off + rows * 4, 256);
  rp->off_map = off;     off = align_up(off + (rows - n_appended + n_removed) * 4, 256);
  rp->off_old_row = off; off = align_up(off + rows * 4, 256);
  rp->off_in_g = off;    off = align_up(off + rows * 4, 256);
  rp->off_grows = off;   off = align_up(off + rows * 4, 256);
  rp->off_gcount = off;  off = align_up(off + 4, 256);
  rp->off_in2 = off;     off = align_up(off + rows * 4, 256);
  rp->off_rows2 = off;   off = align_up(off + rows * 4, 256);
  rp->off_count2 = off;  off = align_up(off + 4, 256);
  rp->off_flag2 = off;   off = align_up(off + rows * 4, 256);
  rp->off_floor2 = off;  off = align_up(off + rows * 8, 256);
  rp->off_c2 = off;      off = align_up(off + 8 * 4, 256);
  rp->off_gtheta2 = off; off = align_up(off + static_cast<size_t>(f->n_pad) * 4, 256);
  rp->total = off;
  return TVBF_OK;
}

// the candidate-kernel parameters of stage s: a whole-catalogue symmetric job on the sweep geometry.
// Stage 0, the refresh sweep: lists by show, list 0 of the two-list table.  Stage 1, the repair sweep:
// lists by gathered row (the plan's lists and candidate table), as the removal.
int fill_refresh_params(const tvbf_features* f, const tvbf_params* q, const RefreshPlan& rp, uint8_t* ws, int s,
                        const int* rows, int n_rows, tvbf::K1Params* kp) {
  int rc = fill_k1_params(f, q, rp.pl, ws, kp);
  if (rc != TVBF_OK) return rc;
  kp->sync_kb = 0;
  kp->sym = 0;              // the one-sided schedule: a rectangle
  kp->wide_epilogue = 0;    // 8 epilogue warps, as the update sweep
  kp->col_tiles = rp.geo[s].col_tiles;
  kp->rb_count = rp.geo[s].rb_count;
  kp->splits = rp.geo[s].splits;
  kp->rb_per_group = rp.geo[s].rb_per_group;
  kp->tiles_per_split = rp.geo[s].tiles_per_split;
  kp->upd_rows = rows;
  kp->upd_q = n_rows;
  kp->upd_bits = nullptr;
  kp->upd_sbits = nullptr;
  if (s == 0) {
    kp->upd_bits = reinterpret_cast<const unsigned int*>(ws + rp.off_gbits);
    kp->upd_sbits = reinterpret_cast<const unsigned int*>(ws + rp.off_sbits);
    kp->cand = reinterpret_cast<uint2*>(ws + rp.off_cand);
    kp->cand_cnt = reinterpret_cast<int*>(ws + rp.off_cnt);
    kp->cand_theta = reinterpret_cast<float*>(ws + rp.off_bound);
  }
  return TVBF_OK;
}

}  // namespace

size_t tvbf_refresh_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_removed,
                                    int32_t n_updated, int32_t n_appended) {
  if (validate_features(f) != TVBF_OK || p == nullptr) return 0;
  RefreshPlan rp;
  tvbf_params q;
  const int none[2] = {0, 0};
  if (make_refresh_plan(f, p, n_removed, n_updated, n_appended, none, &rp, &q) != TVBF_OK) return 0;
  return rp.total;
}

int tvbf_refresh_topk(const tvbf_features* f, const tvbf_params* p, const int32_t* removed, int32_t n_removed,
                      const int32_t* updated, int32_t n_updated, int32_t n_appended, const tvbf_topk_out* prev,
                      const tvbf_topk_out* out, int32_t* changed, void* workspace, size_t workspace_bytes,
                      void* stream) {
  // the arguments first: these checks need no device
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p != nullptr, "params is NULL");
  TVBF_REQUIRE(prev && prev->indices && prev->counts && prev->hybrid && prev->genre && prev->text && prev->metadata,
               "previous table has NULL members");
  TVBF_REQUIRE(out && out->indices && out->counts && out->hybrid && out->genre && out->text && out->metadata &&
                   out->stats,
               "output table has NULL members");
  {
    const void* po[6] = {prev->indices, prev->counts, prev->hybrid, prev->genre, prev->text, prev->metadata};
    const void* oo[6] = {out->indices, out->counts, out->hybrid, out->genre, out->text, out->metadata};
    for (int a = 0; a < 6; ++a)
      for (int b = 0; b < 6; ++b) TVBF_REQUIRE(po[a] != oo[b], "tvbf_refresh_topk: the output table aliases the previous one");
  }
  TVBF_REQUIRE(changed != nullptr && workspace != nullptr, "tvbf_refresh_topk: NULL argument");
  TVBF_REQUIRE((removed != nullptr || n_removed == 0) && (updated != nullptr || n_updated == 0),
               "tvbf_refresh_topk: NULL row list");
  rc = refresh_counts_ok(f, n_removed, n_updated, n_appended);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(!f->text_signed, "refresh: signed text needs the whole job");
  TVBF_ENTER_CALL(stream);
  RefreshPlan rp;
  tvbf_params q;
  int n_rows[2] = {0, 0};
  rc = make_refresh_plan(f, p, n_removed, n_updated, n_appended, n_rows, &rp, &q);
  if (rc != TVBF_OK) return rc;
  if (workspace_bytes < rp.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, rp.total);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const Plan& pl = rp.pl;
  const int n = f->n_shows, k = p->k, n_old = n - n_appended + n_removed;
  const size_t words = static_cast<size_t>(f->n_pad) / 32 * 4;
  auto at = [&](size_t off) { return reinterpret_cast<int*>(ws + off); };
  int *map = at(rp.off_map), *old_row = at(rp.off_old_row), *in_g = at(rp.off_in_g), *g_rows = at(rp.off_grows);
  int *g_count = at(rp.off_gcount), *listed_rows = at(rp.off_rows), *n_listed = at(rp.off_listed);
  int *in2 = at(rp.off_in2), *rows2 = at(rp.off_rows2), *count2 = at(rp.off_count2), *flag2 = at(rp.off_flag2);
  int *c2 = at(rp.off_c2), *cut_j = at(rp.off_cut_j), *flagged = at(pl.off_flag);
  unsigned int* s_bits = reinterpret_cast<unsigned int*>(ws + rp.off_sbits);
  unsigned int* g_bits = reinterpret_cast<unsigned int*>(ws + rp.off_gbits);
  double* cut_s = reinterpret_cast<double*>(ws + rp.off_cut_s);
  double* floors = reinterpret_cast<double*>(ws + pl.off_floor);
  double* floor2 = reinterpret_cast<double*>(ws + rp.off_floor2);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + pl.off_keys);
  int* cnt = reinterpret_cast<int*>(ws + rp.off_cnt);
  // 1. map and classify
  TVBF_CUDA_OK(cudaMemsetAsync(out->stats, 0, 8 * sizeof(int32_t), st));
  TVBF_CUDA_OK(cudaMemsetAsync(s_bits, 0, words, st));
  TVBF_CUDA_OK(cudaMemsetAsync(g_bits, 0, words, st));
  remove_map_kernel<<<(n_old + 255) / 256, 256, 0, st>>>(removed, n_removed, n_old, map);
  TVBF_LAUNCH_OK("remove_map_kernel");
  if (n_updated + n_appended > 0) {
    refresh_sbits_kernel<<<(n_updated + n_appended + 255) / 256, 256, 0, st>>>(updated, n_updated, map, n, n_appended,
                                                                              s_bits);
    TVBF_LAUNCH_OK("refresh_sbits_kernel");
  }
  refresh_rows_kernel<<<(n_old + n_appended + 255) / 256, 256, 0, st>>>(*prev, map, n_old, n, n_appended, k, s_bits,
                                                                         old_row, in_g, g_bits);
  TVBF_LAUNCH_OK("refresh_rows_kernel");
  remove_compact_kernel<<<1, kCompactThreads, 0, st>>>(in_g, n, g_rows, g_count);
  TVBF_LAUNCH_OK("remove_compact_kernel");
  // the sweep's geometry depends on |G|
  TVBF_CUDA_OK(cudaMemcpyAsync(&n_rows[0], g_count, 4, cudaMemcpyDeviceToHost, st));
  TVBF_CUDA_OK(cudaStreamSynchronize(st));
  const tvbf::ScoreParams sp = score_params(f, &q);
  if (n_rows[0] == 0) {   // nothing was swept: every row keeps T'
    TVBF_CUDA_OK(cudaMemsetAsync(cnt, 0, static_cast<size_t>(n) * 4, st));
  } else {
    // 2.-4. the refresh sweep over G, K4s, select, K5 with the rank cut
    rc = make_refresh_plan(f, p, n_removed, n_updated, n_appended, n_rows, &rp, &q);
    if (rc != TVBF_OK) return rc;
    tvbf::K1Params kp;
    rc = fill_refresh_params(f, &q, rp, ws, 0, g_rows, n_rows[0], &kp);
    if (rc != TVBF_OK) return rc;
    const int row_vec = f->k_pad / 8;   // 16-byte vectors per operand row
    update_gather_kernel<<<1024, 256, 0, st>>>(static_cast<const uint4*>(f->operand), g_rows, n_rows[0], rp.q_pad[0],
                                               row_vec, reinterpret_cast<uint4*>(ws + rp.off_gather));
    TVBF_LAUNCH_OK("update_gather_kernel");
    tvbf_features g = *f;   // the gathered rows as the A operand
    g.operand = ws + rp.off_gather;
    g.n_pad = rp.q_pad[0];
    const tvbf::RefreshPrev pv{prev->indices, prev->counts, prev->hybrid, k, old_row, map, s_bits, g_bits,
                               kp.cand + static_cast<size_t>(n) * pl.kp, cnt + n, kp.cand_theta + n, cut_s, cut_j};
    rc = tvbf::k1_launch_refresh(f, &g, kp, rp.grid[0], pv, st);
    if (rc != TVBF_OK) return rc;
    rc = tvbf::k4s_launch(kp, n, st);
    if (rc != TVBF_OK) return rc;
  }
  TVBF_CUDA_OK(cudaMemsetAsync(n_listed, 0, 4, st));
  refresh_select_kernel<<<(n + 255) / 256, 256, 0, st>>>(*prev, *out, cnt, map, old_row, s_bits, g_bits, n, k,
                                                          listed_rows, n_listed);
  TVBF_LAUNCH_OK("refresh_select_kernel");
  if (n_rows[0] > 0) {
    const tvbf::CandLayout lay{0, 1, n, 0};   // list s of show r: slot r + s * n
    rc = tvbf::k5_launch_listed(sp, reinterpret_cast<uint2*>(ws + rp.off_cand), cnt,
                                reinterpret_cast<float*>(ws + rp.off_bound), 2, lay, pl.kp, 0, n, listed_rows, n_listed,
                                *out, flagged, floors, st, cut_s, cut_j);
    if (rc != TVBF_OK) return rc;
    // 5. rejected rows of G to K6 now, the others to the second stage
    TVBF_CUDA_OK(cudaMemsetAsync(in2, 0, static_cast<size_t>(n) * 4, st));
    refresh_split_kernel<<<1, kSplitThreads, 0, st>>>(flagged, floors, g_bits, n, out->stats, in2, flag2, floor2, c2);
    TVBF_LAUNCH_OK("refresh_split_kernel");
    tvbf_topk_out o2 = *out;
    o2.stats = c2;   // the counts of the second flagged arrays, at the slots K6 reads
    rc = tvbf::k6_launch_flagged(sp, flag2, floor2, n, 0, keys, pl.k6_grid, o2, st);
    if (rc != TVBF_OK) return rc;
    remove_compact_kernel<<<1, kCompactThreads, 0, st>>>(in2, n, rows2, count2);
    TVBF_LAUNCH_OK("remove_compact_kernel");
    TVBF_CUDA_OK(cudaMemcpyAsync(&n_rows[1], count2, 4, cudaMemcpyDeviceToHost, st));
    TVBF_CUDA_OK(cudaStreamSynchronize(st));
  }
  if (n_rows[1] > 0) {
    // the second stage: the rejected rows outside G against every column, lists by gathered row
    rc = make_refresh_plan(f, p, n_removed, n_updated, n_appended, n_rows, &rp, &q);
    if (rc != TVBF_OK) return rc;
    tvbf::K1Params kp;
    rc = fill_refresh_params(f, &q, rp, ws, 1, rows2, n_rows[1], &kp);
    if (rc != TVBF_OK) return rc;
    const int row_vec = f->k_pad / 8;
    update_gather_kernel<<<1024, 256, 0, st>>>(static_cast<const uint4*>(f->operand), rows2, n_rows[1], rp.q_pad[1],
                                               row_vec, reinterpret_cast<uint4*>(ws + rp.off_gather));
    TVBF_LAUNCH_OK("update_gather_kernel");
    tvbf_features g = *f;
    g.operand = ws + rp.off_gather;
    g.n_pad = rp.q_pad[1];
    unsigned int* gtheta = reinterpret_cast<unsigned int*>(ws + rp.off_gtheta2);
    rc = tvbf::k1_launch_remove(f, &g, kp, rp.grid[1], gtheta, st);
    if (rc != TVBF_OK) return rc;
    kp.g_theta = gtheta;   // K4s: the gathered rows' lists under their thresholds
    rc = tvbf::k4s_launch(kp, n_rows[1], st);
    if (rc != TVBF_OK) return rc;
    const tvbf::CandLayout lay{0, 1, 0, 0, 1};   // the list of rows2[e] is slot e
    rc = tvbf::k5_launch_listed(sp, kp.cand, kp.cand_cnt, kp.cand_theta, 1, lay, pl.kp, 0, n, rows2, count2, *out,
                                flagged, floors, st);
    if (rc != TVBF_OK) return rc;
  }
  if (n_rows[0] > 0) {
    rc = tvbf::k6_launch_flagged(sp, flagged, floors, n, 0, keys, pl.k6_grid, *out, st);
    if (rc != TVBF_OK) return rc;
  }
  // 6. changed flags against T'
  refresh_changed_kernel<<<(n + 255) / 256, 256, 0, st>>>(*prev, *out, map, old_row, n, k, changed);
  TVBF_LAUNCH_OK("refresh_changed_kernel");
  return TVBF_OK;
}

int tvbf_refresh_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t n_gathered, int32_t n_repaired,
                            int64_t* out4) {
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p && out4, "tvbf_refresh_plan_tiles: NULL argument");
  TVBF_REQUIRE(n_gathered >= 1 || n_repaired == 0, "tvbf_refresh_plan_tiles: %d gathered and %d repaired rows",
               n_gathered, n_repaired);
  RefreshPlan rp;
  tvbf_params q;
  const int n_rows[2] = {n_gathered, n_repaired};
  rc = make_refresh_plan(f, p, 0, 0, 0, n_rows, &rp, &q);
  if (rc != TVBF_OK) return rc;
  uint8_t* fake_ws = reinterpret_cast<uint8_t*>(static_cast<uintptr_t>(4096));   // offsets only, never dereferenced
  for (int s = 0; s < 2; ++s) {
    out4[2 * s] = out4[2 * s + 1] = 0;
    if (n_rows[s] == 0) continue;
    tvbf::K1Params kp;
    rc = fill_refresh_params(f, &q, rp, fake_ws, s, nullptr, n_rows[s], &kp);
    if (rc != TVBF_OK) return rc;
    long long t[2];
    tvbf::k1_update_executed_tiles(kp, rp.grid[s], t);
    out4[2 * s] = t[0];
    out4[2 * s + 1] = t[1];
  }
  return TVBF_OK;
}

// ---- streaming statistics of the four similarity matrices (no N x N) --------------------------
size_t tvbf_stats_accum_bytes(void) { return sizeof(tvbf::StatsAccum); }

int tvbf_similarity_stats(const tvbf_features* f, const tvbf_params* p, void* accum, void* workspace,
                          size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p && accum && workspace, "tvbf_similarity_stats: NULL argument");
  TVBF_REQUIRE(f->genre_mode != TVBF_GROUP_FOLDED && f->meta_mode != TVBF_GROUP_FOLDED && f->genre_hi == nullptr,
               "streaming statistics need binary genre (at most 64 columns) / one-hot metadata features");
  TVBF_REQUIRE(!f->bits_folded, "streaming statistics need the plain text operand (bits_folded is set)");
  TVBF_REQUIRE(f->text_cols == 0, "streaming statistics need the plain text operand (text_cols is set)");
  TVBF_REQUIRE(p->genre_weight >= 0.0 && p->text_weight >= 0.0 && p->metadata_weight >= 0.0,
               "streaming statistics need non-negative weights");
  tvbf_params q = *p;
  q.row_begin = 0;
  q.row_end = f->n_shows;
  q.k = 20;
  q.min_similarity = 0.5;
  q.exclude_self = 1;
  q.splits = 0;
  q.tuning = (p->tuning & (1 << 30)) | 2 | (1 << 20);   // CTA pairs, plan as a one-sided job
  Plan pl;
  rc = make_plan(f, &q, &pl);
  if (rc != TVBF_OK) return rc;
  if (workspace_bytes < pl.total) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return TVBF_ERR_WORKSPACE;
  }
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  tvbf::K1Params kp;
  rc = fill_k1_params(f, &q, pl, ws, &kp);
  if (rc != TVBF_OK) return rc;
  // symmetric schedule, 8 splits, one ring stage given up for the shared-memory histogram
  const int clusters = sms / 2;
  kp.sym = 1;
  kp.splits = 8;
  while (kp.splits > 1 && (clusters / kp.splits < 1 || pl.col_tiles / kp.splits < 8)) --kp.splits;
  kp.rb_count = pl.sb_count;
  kp.rb_per_group = clusters / kp.splits;
  if (kp.rb_per_group > pl.sb_count) kp.rb_per_group = pl.sb_count;
  kp.tiles_per_split = (pl.col_tiles + kp.splits - 1) / kp.splits;
  kp.stages = 5;
  kp.stats = static_cast<tvbf::StatsAccum*>(accum);
  kp.inv_scale2 = static_cast<float>(std::ldexp(1.0, -2 * f->text_scale_log2));
  kp.w_text_plain = static_cast<float>(p->text_weight);
  kp.w_genre = static_cast<float>(p->genre_weight);
  kp.w_meta = static_cast<float>(p->metadata_weight);
  static thread_local tvbf::StatsAccum init;   // 80 KB: keep it off the stack
  memset(&init, 0, sizeof(init));
  const double wsum = p->genre_weight + p->text_weight + p->metadata_weight;
  for (int qi = 0; qi < 4; ++qi) {
    init.min_bits[qi] = 0x7f800000u;
    init.max_bits[qi] = 0u;
    init.hi[qi] = static_cast<float>((qi == 3 ? (wsum > 0 ? wsum : 1.0) : 1.0) * 1.002);
  }
  for (int qi = 0; qi < 2; ++qi)
    for (int c = 0; c < tvbf::kStatsCand; ++c) { init.cand_val[qi][c] = -1.0f; init.cand_ij[qi][c][0] = -1; init.cand_ij[qi][c][1] = -1; }
  // staged through pageable host memory: small (80 KB) and synchronous with respect to the host
  TVBF_CUDA_OK(cudaMemcpyAsync(accum, &init, sizeof(init), cudaMemcpyHostToDevice, st));
  TVBF_CUDA_OK(cudaStreamSynchronize(st));
  TVBF_CUDA_OK(cudaMemsetAsync(kp.progress, 0, 256, st));
  return tvbf::k1_launch_stats(f, kp, kp.rb_per_group * kp.splits * 2, st);
}

int tvbf_score_pairs(const tvbf_features* f, const tvbf_params* p, const int32_t* pairs,
                     int32_t n_pairs, double* out4, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p && pairs && out4 && n_pairs > 0, "tvbf_score_pairs: bad arguments");
  const tvbf::ScoreParams sp = score_params(f, p);
  return tvbf::score_pairs_launch(sp, pairs, n_pairs, out4, static_cast<cudaStream_t>(stream));
}

// ---- every pair above a threshold (tvbf_neighbours_*) ------------------------------------------
// The sweep walks the tiles of the symmetric top-k sweep of the same job with kMode 11 of the candidate
// kernel: no lists, no thresholds, no seed pass.  Every pair i < j whose upper bound U (which is >= its
// exact hybrid) exceeds theta_init (an fp32 below min_similarity, fill_k1_params) is emitted, so every pair whose exact
// score reaches min_similarity is among the candidates; the finish rescores them in float64.
namespace {

// the job as the symmetric top-k sweep would take it: k and the candidate knobs do not apply, the
// diagonal is added by the finish
int neighbours_plan(const tvbf_features* f, const tvbf_params* p, SymPlan* sp, tvbf_params* q) {
  TVBF_REQUIRE(p != nullptr, "params is NULL");
  TVBF_REQUIRE(p->min_similarity > 0.0,
               "neighbour sweep: min_similarity must be > 0 (got %g); a threshold at or below 0 selects every pair",
               p->min_similarity);
  TVBF_REQUIRE(f->genre_mode != TVBF_GROUP_FOLDED && f->meta_mode != TVBF_GROUP_FOLDED,
               "neighbour sweep: float (folded) genre / metadata groups are not supported, only packed ones");
  TVBF_REQUIRE(p->genre_weight >= 0.0 && p->text_weight >= 0.0 && p->metadata_weight >= 0.0,
               "neighbour sweep: the weights must be non-negative (got %g, %g, %g)", p->genre_weight,
               p->text_weight, p->metadata_weight);
  *q = *p;
  q->k = 1;
  q->exclude_self = 1;
  q->candidates = 0;
  q->force_exact = 0;
  q->row_begin = 0;
  q->row_end = f->n_shows;
  const int rc = make_sym_plan(f, q, 0, 1, sp);
  if (rc != TVBF_OK) {
    char why[512];
    snprintf(why, sizeof(why), "%s", g_last_error);
    tvbf_set_error("neighbour sweep: the symmetric sweep does not take this job (%s)", why);
  }
  return rc;
}

int neighbours_sizes_ok(const tvbf_features* f, int64_t n_pairs) {
  TVBF_REQUIRE(n_pairs >= 0 && 2 * n_pairs + f->n_shows <= INT32_MAX,
               "neighbour finish: %lld candidate pairs are more than one call takes", static_cast<long long>(n_pairs));
  return TVBF_OK;
}

}  // namespace

size_t tvbf_neighbours_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int64_t capacity) {
  if (validate_features(f) != TVBF_OK || capacity < 0 || neighbours_sizes_ok(f, capacity) != TVBF_OK) return 0;
  SymPlan sp;
  tvbf_params q;
  if (neighbours_plan(f, p, &sp, &q) != TVBF_OK) return 0;
  const size_t finish = tvbf::neighbours_finish_bytes(f->n_shows, capacity, p->exclude_self);
  return finish > 256 ? finish : 256;
}

int tvbf_neighbours_sweep(const tvbf_features* f, const tvbf_params* p, int32_t* pairs, int64_t capacity,
                          int64_t* n_candidates, void* workspace, size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(n_candidates && workspace && capacity >= 0 && (pairs || capacity == 0),
               "tvbf_neighbours_sweep: bad arguments");
  SymPlan sp;
  tvbf_params q;
  rc = neighbours_plan(f, p, &sp, &q);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(workspace_bytes >= 256, "workspace too small: %zu < 256", workspace_bytes);
  auto st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  tvbf::K1Params kp;
  rc = fill_k1_params(f, &q, sp.pl, ws, &kp);
  if (rc != TVBF_OK) return rc;
  // nothing of the top-k sweep's lists is used
  kp.scratch = kp.cand = kp.g_list = nullptr;
  kp.cand_cnt = nullptr;
  kp.cand_theta = nullptr;
  kp.g_theta = kp.g_cnt = nullptr;
  kp.progress = reinterpret_cast<unsigned int*>(ws);
  kp.pairs = reinterpret_cast<int2*>(pairs);
  kp.pair_count = reinterpret_cast<unsigned long long*>(n_candidates);
  kp.pair_cap = capacity;
  TVBF_CUDA_OK(cudaMemsetAsync(kp.progress, 0, 256, st));
  TVBF_CUDA_OK(cudaMemsetAsync(n_candidates, 0, sizeof(int64_t), st));
  return tvbf::k1_launch_pairs(f, kp, sp.pl.grid, st);
}

int tvbf_neighbours_finish(const tvbf_features* f, const tvbf_params* p, const int32_t* pairs, int64_t n_candidates,
                           int32_t max_per_row, int64_t* row_ptr, int32_t* indices, double* hybrid, double* genre,
                           double* text, double* metadata, void* workspace, size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(row_ptr && indices && hybrid && genre && text && metadata && workspace && (pairs || n_candidates == 0),
               "tvbf_neighbours_finish: NULL buffer");
  TVBF_REQUIRE(max_per_row >= 0, "max_per_row must be >= 0 (0: no cap)");
  rc = neighbours_sizes_ok(f, n_candidates);
  if (rc != TVBF_OK) return rc;
  SymPlan sp;
  tvbf_params q;
  rc = neighbours_plan(f, p, &sp, &q);
  if (rc != TVBF_OK) return rc;
  tvbf::ScoreParams scp = score_params(f, p);
  scp.exclude_self = p->exclude_self ? 1 : 0;
  const tvbf::NeighboursOut out{reinterpret_cast<long long*>(row_ptr), indices, hybrid, genre, text, metadata};
  return tvbf::neighbours_finish_launch(scp, reinterpret_cast<const int2*>(pairs), n_candidates, max_per_row, out,
                                        workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t tvbf_exact_workspace_bytes(const tvbf_features* f, int32_t n_rows_listed) {
  if (f == nullptr || n_rows_listed <= 0) return 0;
  int sms = 0;
  if (sm_count_cached(&sms) != TVBF_OK) return 0;
  return align_up(tvbf::k6_scratch_bytes(*f, sms), 256);
}

int tvbf_exact_rows(const tvbf_features* f, const tvbf_params* p, const int32_t* rows,
                    int32_t n_rows_listed, const tvbf_topk_out* out, void* workspace,
                    size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p && p->k >= 1 && rows && n_rows_listed > 0, "tvbf_exact_rows: bad arguments");
  TVBF_REQUIRE(out && out->indices && out->counts && out->hybrid && out->genre && out->text &&
                   out->metadata,
               "output table has NULL members");
  const size_t need = tvbf_exact_workspace_bytes(f, n_rows_listed);
  if (need == 0) return TVBF_ERR_UNSUPPORTED;
  if (workspace == nullptr || workspace_bytes < need) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, need);
    return TVBF_ERR_WORKSPACE;
  }
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  const tvbf::ScoreParams sp = score_params(f, p);
  return tvbf::k6_launch(sp, rows, n_rows_listed, nullptr, nullptr, 0, 0,
                         static_cast<unsigned long long*>(workspace), sms, *out,
                         static_cast<cudaStream_t>(stream));
}

int tvbf_matrix_rows_topk(const double* hybrid, const double* genre, const double* text,
                          const double* metadata, int32_t n, const tvbf_params* p,
                          const int32_t* rows, int32_t n_rows_listed, const tvbf_topk_out* out,
                          void* workspace, size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(hybrid && genre && text && metadata && n > 0, "tvbf_matrix_rows_topk: bad matrices");
  TVBF_REQUIRE(p && p->k >= 1 && rows && n_rows_listed > 0, "tvbf_matrix_rows_topk: bad arguments");
  TVBF_REQUIRE(out && out->indices && out->counts && out->hybrid && out->genre && out->text &&
                   out->metadata,
               "output table has NULL members");
  int sms = 0;
  int rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  int grid = 2 * sms;
  if (grid > n_rows_listed) grid = n_rows_listed;
  const size_t need = align_up(static_cast<size_t>(grid) * n * 8, 256);
  if (workspace == nullptr || workspace_bytes < need) {
    tvbf_set_error("workspace too small: %zu < %zu", workspace_bytes, need);
    return TVBF_ERR_WORKSPACE;
  }
  return tvbf::k6_launch_matrix(hybrid, genre, text, metadata, n, p->k, p->exclude_self,
                                p->min_similarity, rows, n_rows_listed,
                                static_cast<unsigned long long*>(workspace), grid, *out,
                                static_cast<cudaStream_t>(stream));
}

static int debug_tile(const tvbf_features* f, int32_t row0, int32_t col0, float* out, int cg,
                      void* stream) {
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(out != nullptr, "out is NULL");
  TVBF_REQUIRE(row0 >= 0 && row0 + 128 * cg <= f->n_pad && col0 >= 0 && col0 + 256 <= f->n_pad,
               "tile origin outside the padded operand");
  int sms = 0;
  rc = sm_count_cached(&sms);
  if (rc != TVBF_OK) return rc;
  tvbf::K1Params kp;
  memset(&kp, 0, sizeof(kp));
  kp.col_side = static_cast<const TvbfColSide*>(f->col_side);
  kp.meta_scale = f->meta_scale;
  kp.dump = out;
  kp.n_shows = f->n_shows;
  kp.row_begin = row0;
  kp.row_end = row0 + 128 * cg;
  kp.k_blocks = f->k_pad / 64;
  kp.col_tiles = 1;
  kp.splits = 1;
  kp.rb_count = 1;
  kp.rb_per_group = 1;
  kp.tiles_per_split = 1;
  kp.tile_stride = 1;
  kp.deal_r = 1;
  kp.stages = cg == 2 ? 6 : 4;
  kp.dump_col0 = col0;
  kp.kp = 32;
  return tvbf::k1_launch_dump(f, kp, cg, static_cast<cudaStream_t>(stream));
}

// host-only: how many tensor-core tiles the candidate pass of this job executes
int tvbf_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                    int32_t tile_sharded, int64_t* out4) {
  int rc = validate_features(f);
  if (rc != TVBF_OK) return rc;
  TVBF_REQUIRE(p && out4, "tvbf_plan_tiles: NULL argument");
  uint8_t* fake_ws = reinterpret_cast<uint8_t*>(static_cast<uintptr_t>(4096));   // offsets only, never dereferenced
  tvbf::K1Params kp;
  long long t[2] = {0, 0};
  if (tile_sharded) {
    SymPlan sp;
    rc = make_sym_plan(f, p, rank, world, &sp);
    if (rc != TVBF_OK) return rc;
    rc = fill_sym_params(f, p, sp, rank, world, fake_ws, nullptr, &kp);
    if (rc != TVBF_OK) return rc;
    kp.sym_phase = 0;
    if (sp.local_sb > 0) tvbf::k1_executed_tiles(kp, sp.pl.grid, t);
    out4[2] = 256;
    out4[3] = 1;
  } else {
    rc = validate_params(f, p);
    if (rc != TVBF_OK) return rc;
    Plan pl;
    rc = make_plan(f, p, &pl);
    if (rc != TVBF_OK) return rc;
    const bool use_k1 = !p->force_exact && pl.entries != 0;
    if (use_k1) {
      rc = fill_k1_params(f, p, pl, fake_ws, &kp);
      if (rc != TVBF_OK) return rc;
      tvbf::k1_executed_tiles(kp, pl.grid, t);
    }
    out4[2] = 128 * pl.cg;
    out4[3] = pl.sym;
  }
  out4[0] = t[0];
  out4[1] = t[1];
  return TVBF_OK;
}

// host-only: the slack constants of the candidate pass' upper bound for this job
int tvbf_debug_slack(const tvbf_features* f, const tvbf_params* p, float* out5) {
  TVBF_REQUIRE(f && p && out5, "tvbf_debug_slack: NULL argument");
  const Slack sl = make_slack(f, p->genre_weight, p->text_weight, p->metadata_weight, p->text_rel_err);
  out5[0] = sl.w_text;
  out5[1] = sl.w_text_err;
  out5[2] = sl.w_text_acc;
  out5[3] = sl.eps;
  out5[4] = sl.eps_term;
  return TVBF_OK;
}

// host-only: the work items of one K1 launch (no device needed)
int32_t tvbf_debug_schedule(int32_t col_tiles, int32_t super_blocks, int32_t sb_per_group, int32_t splits,
                            int32_t world, int32_t rank, int32_t symmetric, int32_t* out, int32_t max_items) {
  if (col_tiles < 1 || super_blocks < 0 || sb_per_group < 1 || splits < 1 || world < 1 || rank < 0 ||
      rank >= world || out == nullptr || max_items < 0) {
    tvbf_set_error("tvbf_debug_schedule: bad arguments");
    return TVBF_ERR_INVALID;
  }
  tvbf::K1Params kp;
  memset(&kp, 0, sizeof(kp));
  kp.col_tiles = col_tiles;
  kp.splits = splits;
  kp.rb_count = super_blocks;
  kp.rb_per_group = sb_per_group;
  kp.tiles_per_split = (col_tiles + splits - 1) / splits;
  kp.deal_r = 1;
  if (world > 1) {
    kp.deal_r = sb_per_group;
    kp.deal_groups = tvbf::k1_deal_groups(super_blocks, sb_per_group, world, rank, kp.deal_gid, &kp.rb_count);
    if (kp.deal_groups < 0) {
      tvbf_set_error("tvbf_debug_schedule: too many groups per GPU");
      return TVBF_ERR_INVALID;
    }
    if (kp.deal_groups == 0) return 0;   // nothing dealt to this GPU
  }
  kp.sym = symmetric ? 1 : 0;
  return tvbf::k1_debug_schedule(kp, out, max_items);
}

int tvbf_debug_gemm_tile(const tvbf_features* f, int32_t row0, int32_t col0, float* out,
                         void* stream) {
  TVBF_ENTER_CALL(stream);
  return debug_tile(f, row0, col0, out, 1, stream);
}

int tvbf_debug_gemm_tile_pair(const tvbf_features* f, int32_t row0, int32_t col0, float* out,
                              void* stream) {
  TVBF_ENTER_CALL(stream);
  return debug_tile(f, row0, col0, out, 2, stream);
}

}  // extern "C"
