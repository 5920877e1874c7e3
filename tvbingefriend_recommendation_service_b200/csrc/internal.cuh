// Types and launchers shared between the translation units of libtvbf (not part of the ABI).
#pragma once

#include "common.cuh"

namespace tvbf {

// Raw accumulators of the streaming upper-triangle statistics (ml/similarity_computer.py:171-190
// for catalogues whose N x N matrices cannot exist).  Matrix order: genre, text, metadata, hybrid.
constexpr int kStatsBins = 1024;
constexpr int kStatsCand = 2048;
struct StatsAccum {
  double sum[4];
  double sumsq[4];
  unsigned long long zeros[4];            // elements that are exactly 0 (kept out of the histogram)
  unsigned long long hist[4][kStatsBins]; // bin b covers [b, b+1) * hi / kStatsBins
  unsigned int min_bits[4];               // float bits of the smallest / largest element seen
  unsigned int max_bits[4];
  float hi[4];                            // histogram range per matrix
  int n_cand;                             // reserved
  int cand_ij[2][kStatsCand][2];          // argmax candidates of {text, hybrid}: one slot per epilogue warp
  float cand_val[2][kStatsCand];
  double sum_gm;                          // sum of genre * metadata (cross moment of the hybrid's variance)
};

// parameters of the tcgen05 candidate kernel (hybrid_topk.cu)
constexpr int kMaxDealGroups = 192;
constexpr int kMaxPeers = 16;
constexpr int kMaxSweep = 5;   // weight triples that can share one symmetric tensor-core sweep

struct K1Params {
  const TvbfColSide* col_side;
  const float* meta_scale;
  const unsigned long long* genre_hi;   // genre bits 64..127 per show, or NULL (G <= 64)
  uint2* scratch;      // [gridDim.x][128][32*E] working candidate lists (score bits, column)
  uint2* cand;         // [rows][splits][kp] sorted candidates
  int* cand_cnt;       // [rows][splits]
  float* cand_theta;   // [rows][splits] bound on every dropped U, -inf if nothing was dropped
  float* dump;         // dump kernel only: [128*CG][256] raw accumulators of one tile
  unsigned int* progress;  // grid-wide pacing counter (zeroed before launch), see sync_kb
  int n_shows;
  int row_begin;       // multiple of 128
  int row_end;
  int k_blocks;        // k_pad / 64
  int col_tiles;       // ceil(n_shows / 256)
  int splits;
  int rb_count;        // super blocks (128 * cta_group rows) of this shard
  int rb_per_group;    // super blocks processed concurrently (clusters = rb_per_group * splits)
  int dump_col0;       // dump kernel only
  int tiles_per_split; // every item walks exactly this many column tiles (phantom past the end)
  int sync_kb;         // producers pace themselves every sync_kb k-blocks (0 = no pacing)
  int sync_slack;      // ... staying at most this many chunks ahead of the slowest CTA
  int stages;          // smem ring depth actually used (<= compiled maximum)
  // symmetric mode (hybrid(i,j) == hybrid(j,i)): only tiles on or above the diagonal are computed
  // and every score is offered to BOTH shows' candidate lists, which therefore live in global
  // memory and are shared by all CTAs
  int sym;
  StatsAccum* stats;       // statistics sweep only
  float inv_scale2;        // 2^-2s: accumulator -> text cosine
  float w_text_plain;      // text weight without the error inflation (statistics sweep)
  // Several GPUs (symmetric sweep): the super blocks are dealt in GROUPS of deal_r consecutive
  // blocks (what one launch wave sweeps together, so a wave's blocks differ by < deal_r diagonal
  // tiles), longest group to the least-loaded GPU.  deal_groups == 0: single GPU, local == global.
  int deal_groups;         // groups owned by this launch
  int deal_r;              // super blocks per dealt group
  unsigned short deal_gid[kMaxDealGroups];   // global group number of each local group, cost descending
  // The threshold seed pass of a multi-GPU job is dealt by super-block COUNT (block b to GPU b mod
  // seed_world), not by the sweep's tile-balanced groups: its cost is per block, and the seeded
  // thresholds are MAX-reduced over the GPUs anyway.
  int seed_world, seed_rank, seed_clusters;
  int wide_epilogue;       // symmetric sweep with 16 epilogue warps (small vocabularies: epilogue-bound)
  int cand_packed;         // K4s writes {count, bound bits} as entry kp of each row, row stride kp + 1;
                           // 2: ... straight into the OWNER GPU's receive buffer over NVLink (peer stores):
                           // show r belongs to GPU r / peer_shard_rows, whose buffer peer_cand[owner] is laid
                           // out [world][peer_shard_rows][kp + 1] -- slice peer_rank is this GPU's
  uint2* peer_cand[kMaxPeers];
  int peer_shard_rows, peer_rank;
  int tile_stride;         // one-sided sweep visits every tile_stride-th column tile (1 = all)
  int seed_theta;          // one-sided sweep only seeds g_theta with the kp-th best sampled score
  int sym_phase;           // 0: init + seed + sweep in one call; 1: init + seed only; 2: sweep only
  int sym_cap;             // entries per shared list
  unsigned int* g_theta;   // [n_pad] raw bits of the (positive) float threshold of each show
  unsigned int* g_cnt;     // [n_pad] appends so far (> sym_cap = overflow)
  uint2* g_list;           // [n_pad][sym_cap] (score bits, column)
  // threshold seed pass (kMode 3): bin = floor(u * hist_inv_w + hist_off), bin b >= 1 = [lo + (b-1) w, lo + b w)
  float hist_lo, hist_w, hist_inv_w, hist_off;
  float score_hi;      // no upper bound U exceeds this (sum of the weights, inflated)
  int fold;            // the operand carries the packed genre / metadata groups (tvbf_features.bits_folded):
                       // the accumulator is the whole hybrid and the epilogue skips the popcounts
  int refresh_period;  // a list's threshold is refreshed at 2*kp entries and every refresh_period further ones
                       // (a power of two; 0: at 2*kp, 4*kp, 8*kp, ...)
  int wait_ns;         // first sleep of the backed-off mbarrier waits
  int* dbg_entries;    // diagnostics (TVBF_DEBUG_COUNTS=1): K4s adds every list's length to stats[4]
  int cooperative;     // launch with the cooperative attribute (co-residency guaranteed)
  int kp;              // candidates kept per (row, split)
  int exclude_self;
  float w_text;        // text_weight * 2^-2s
  float w_text_err;    // |text_weight| * 2^-2s * rel_err  (multiplies |acc|)
  // The tensor-core accumulation error grows with the number of non-zero products of a pair, which
  // is at most the number of non-zero operand entries of the row ("terms" = its text nnz + the
  // folded columns): per row, w_text_err += terms * w_text_acc and eps += terms * eps_term.
  const int64_t* text_indptr;
  int folded_cols;
  float w_text_acc;    // relative accumulation allowance per term (0 in absolute mode)
  float eps_term;      // absolute allowance per term: fp16 subnormal operands (+ accumulation in absolute mode)
  float w_genre;
  float w_meta;        // metadata_weight
  int meta_hstack;     // 1: per-column 1/sqrt(#categories) scale is read from meta_scale
  float eps;           // absolute slack: fp32 rounding of the epilogue (+ folded-group bounds)
  float theta_init;    // just below min_similarity
  // weight sweep (symmetric mode, n_weights > 1): triple w keeps its own shared lists under the
  // virtual show id  w * n_pad + show  (g_theta / g_cnt / g_list / cand have n_weights * n_pad rows)
  int n_weights;
  int n_pad;
  float mw_text[kMaxSweep], mw_text_err[kMaxSweep], mw_genre[kMaxSweep], mw_meta[kMaxSweep], mw_eps[kMaxSweep];
  float mw_text_acc[kMaxSweep], mw_eps_term[kMaxSweep];
  float mw_score_hi[kMaxSweep];   // score_hi of each triple (histogram range of its seed pass)
  // append sweep (kMode 6, tvbf_append_topk): shows [0, append_n_old) had a table already; only tiles
  // with a column tile >= append_b0 = append_n_old / 256 are computed, and pairs of two old shows are
  // offered to neither list
  int append_n_old;
  int append_b0;
  // update sweep (kMode 7), its threshold seed pass (kMode 8) and the repair sweep of a removal
  // (kMode 9, tvbf_remove_topk, which indexes the lists by gathered row), tvbf_update_topk: the A operand is
  // the gather of the updated shows' operand rows, and gathered row r < upd_q is show upd_rows[r],
  // whose records, slack terms, threshold and list are read through that map.  A column whose bit is
  // set in upd_bits (bit j % 32 of word j / 32) was updated itself: it is offered nothing from the
  // column side, its own gathered row feeds its list.
  const int* upd_rows;
  int upd_q;
  const unsigned int* upd_bits;
  // refresh sweep (kMode 10, tvbf_refresh_topk): upd_bits marks G (every gathered show), upd_sbits the
  // shows of S (updated or appended); only a gathered row whose show is in S feeds the column side
  const unsigned int* upd_sbits;
};

// The previous table of an update and where its rows go (list 1 of the two-list candidate table, as
// AppendPrev), plus the rank cut K5 checks for every show whose previous row was full.
struct UpdatePrev {
  const int* indices;   // [n_shows, k]
  const int* counts;    // [n_shows]
  const double* hybrid; // [n_shows, k]
  int k;
  const unsigned int* upd_bits;
  uint2* list;          // [n_shows][kp]
  int* cnt;             // [n_shows]
  float* bound;         // [n_shows]
  double* cut_score;    // [n_shows] previous k-th entry (score, index); index -1: no cut
  int* cut_index;
};

// The previous table of a refresh (old numbering) read as the renumbered table T': new row r is old row
// old_row[r] (-1: appended) with every index j renumbered to map[j].  Lists and cut as UpdatePrev.
struct RefreshPrev {
  const int* indices;   // [n_old, k]
  const int* counts;    // [n_old]
  const double* hybrid; // [n_old, k]
  int k;
  const int* old_row;   // [n_shows]
  const int* map;       // [n_old] (-1: removed)
  const unsigned int* s_bits;   // S: updated or appended shows
  const unsigned int* g_bits;   // G: S and the remaining shows whose previous row names a removed show
  uint2* list;          // [n_shows][kp]
  int* cnt;             // [n_shows]
  float* bound;         // [n_shows]
  double* cut_score;    // [n_shows]
  int* cut_index;
};

// The previous table of an append and where its rows go: list 1 of the two-list candidate table K5
// merges (list 0 is K4s' compaction of the append sweep's shared lists).
struct AppendPrev {
  const int* indices;   // [n_old, k]
  const int* counts;    // [n_old]
  const double* hybrid; // [n_old, k]
  int n_old, k;
  uint2* list;          // [n_shows][kp]
  int* cnt;             // [n_shows]
  float* bound;         // [n_shows]
};

// parameters of the exact fp64 scorers (rescore.cu)
struct ScoreParams {
  tvbf_features f;
  double wg, wt, wm;
  double min_similarity;
  int k;
  int exclude_self;
};

int k1_entries_per_lane(int k);
int k1_default_candidates(int k);
int k1_choose_splits(int rb_count, int col_tiles, int sm_count);
int k1_launch(const tvbf_features* f, const K1Params& kp, int entries_per_lane, int cta_group,
              int grid, cudaStream_t st);
void k1_executed_tiles(const K1Params& kp, int grid, long long* out2);
int k1_launch_dump(const tvbf_features* f, const K1Params& kp, int cta_group, cudaStream_t st);
// candidate list s of shard row r lives in slot  slot_base + r * row_stride + s * list_stride;
// packed: a slot is kp + 1 entries, the last one holding {count, bound bits}, and cand_cnt /
// cand_theta are not used
struct CandLayout {
  long long slot_base, row_stride, list_stride;
  int packed;
  int gathered;   // k5_launch_listed only: the lists of rows[e] are at row position e instead of rows[e]
};
int k5_launch(const ScoreParams& sp, const uint2* cand, const int* cand_cnt,
              const float* cand_theta, int splits, CandLayout lay, int kp, int row_begin, int n_rows,
              const tvbf_topk_out& out, int* flagged_rows, double* flagged_floor, cudaStream_t st);
// K5 over the table rows rows[0 .. *n_listed) (a device count; at most n_rows).  With cut_index
// (update): a row r with cut_index[r] >= 0 is final only if its k-th entry also ranks at or above
// (cut_score[r], cut_index[r]).
int k5_launch_listed(const ScoreParams& sp, const uint2* cand, const int* cand_cnt, const float* cand_theta,
                     int splits, CandLayout lay, int kp, int row_begin, int n_rows, const int* rows,
                     const int* n_listed, const tvbf_topk_out& out, int* flagged_rows, double* flagged_floor,
                     cudaStream_t st, const double* cut_score = nullptr, const int* cut_index = nullptr);
// deal the ceil(total / r) groups of r consecutive super blocks to `world` GPUs; fills gid[] with the
// groups of `rank` (cost descending) and returns {groups, super blocks} of that rank, or -1 when a
// rank would own more than kMaxDealGroups groups
int k1_deal_groups(int total_super_blocks, int r, int world, int rank, unsigned short* gid, int* local_sb);
int k1_debug_schedule(const K1Params& p, int* out, int max_items);
// geometry of the append sweep over n_shows shows of which the first n_old are old, on `clusters` CTA
// pairs: fills col_tiles, rb_count (= super blocks), splits and rb_per_group of p
void k1_append_geometry(int n_old, int n_shows, int clusters, K1Params* p);
// items of the append sweep, as k1_debug_schedule
int k1_debug_append_schedule(const K1Params& p, int* out, int max_items);
// seed pass over the new shows, thresholds of the old shows from the previous table, the previous
// table as candidate list 1, then the append sweep (kp.sym == 1, kp.append_* set)
int k1_launch_append(const tvbf_features* f, const K1Params& kp, int grid, const AppendPrev& prev,
                     cudaStream_t st);
// tiles of the append: out[0] its seed pass over the new super blocks, out[1] the append sweep
void k1_append_executed_tiles(const tvbf_features* f, const K1Params& kp, int grid, long long* out);
// geometry of the update sweep of q gathered rows against n_shows columns on `clusters` CTA pairs:
// a rectangle of ceil(q / 256) super blocks x ceil(n_shows / 256) column tiles (p->sym = 0 schedule)
void k1_update_geometry(int q, int n_shows, int clusters, K1Params* p);
// thresholds and list 1 from the previous table, seed pass over the gathered rows, then the update
// sweep; g: f with the gathered operand ([kp.upd_q rounded up to 256, k_pad]) as its operand
int k1_launch_update(const tvbf_features* f, const tvbf_features* g, const K1Params& kp, int grid,
                     const UpdatePrev& prev, cudaStream_t st);
// tiles of the update: out[0] its seed pass over the gathered rows, out[1] the update sweep
void k1_update_executed_tiles(const K1Params& kp, int grid, long long* out);
// seed pass over the gathered rows of a removal (kp.upd_rows, thresholds in kp.g_theta by show), then
// the repair sweep (kMode 9) on the update geometry: the lists kp.g_cnt / kp.g_list and the thresholds
// gtheta ([rb_count * 256]) are indexed by the gathered row; only those lists are cleared
int k1_launch_remove(const tvbf_features* f, const tvbf_features* g, const K1Params& kp, int grid,
                     unsigned int* gtheta, cudaStream_t st);
// thresholds and list 1 from the renumbered previous table, seed pass over the gathered rows of G, then
// the refresh sweep (kMode 10); kp.upd_bits holds G, kp.upd_sbits S
int k1_launch_refresh(const tvbf_features* f, const tvbf_features* g, const K1Params& kp, int grid,
                      const RefreshPrev& prev, cudaStream_t st);
int k4s_launch(const K1Params& kp, int n_rows, cudaStream_t st);
int k1_launch_stats(const tvbf_features* f, const K1Params& kp, int grid, cudaStream_t st);
int score_pairs_launch(const ScoreParams& sp, const int* pairs, int n_pairs, double* out, cudaStream_t st);
size_t k6_scratch_bytes(int n_shows, int sm_count);
int k6_launch(const ScoreParams& sp, const int* rows, int n_listed, const int* count_ptr,
              const double* floors, int row_begin, int rows_are_local, unsigned long long* key_scratch,
              int grid, const tvbf_topk_out& out, cudaStream_t st, int no_text = 0, int list_cap = 0);
// the two lists K5 leaves behind: flagged shows with text (front) and without (back of the arrays)
int k6_launch_flagged(const ScoreParams& sp, const int* flagged, const double* floors, int n_rows,
                      int row_begin, unsigned long long* key_scratch, int grid, const tvbf_topk_out& out,
                      cudaStream_t st);

int k6_launch_matrix(const double* h, const double* g, const double* t, const double* m, int n,
                     int k, int exclude_self, double min_similarity, const int* rows, int n_listed,
                     unsigned long long* key_scratch, int grid, const tvbf_topk_out& out,
                     cudaStream_t st);

}  // namespace tvbf
