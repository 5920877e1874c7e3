/*
 * libtvbf -- C ABI of the B200 (sm_100a) hybrid-similarity -> top-K path.
 *
 * The reference (tomboone/tvbingefriend-recommendation-service) is pure Python and has no FFI
 * layer; its boundary for this path is the Python API of
 *   ml/similarity_computer.py:12-190            (SimilarityComputer)
 *   scripts/populate_database.py:85-259         (compute_and_store_similarities, loop :170-218)
 *   services/content_based_service.py:161-338   (get_recommendations_from_matrix, bulk variant)
 * and all arithmetic below it is sklearn.metrics.pairwise.cosine_similarity + numpy.argsort.
 * This header declares the entry points a ctypes binding of that path uses (INTEGRATION.md
 * shows the stub).  Every function cites the reference call it replaces.
 *
 * Conventions
 *   - plain C types only; all array pointers are DEVICE pointers owned by the caller (torch
 *     tensors on the host side), `stream` is a cudaStream_t passed as void*;
 *   - every function returns TVBF_OK (0) or a negative TVBF_ERR_* code; tvbf_last_error()
 *     returns a thread-local message for the last failure; no exception crosses the boundary;
 *   - functions enqueue work on `stream` and return without synchronising unless stated;
 *   - thread-compatible: no global mutable state besides the thread-local last error and a
 *     launch counter (tvbf_kernel_launches).
 */
#ifndef TVBF_H_
#define TVBF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TVBF_VERSION 100 /* 0.1.0 */

enum {
  TVBF_OK = 0,
  TVBF_ERR_INVALID = -1,     /* bad argument / unsupported shape */
  TVBF_ERR_CUDA = -2,        /* CUDA runtime / driver error      */
  TVBF_ERR_UNSUPPORTED = -3, /* device is not sm_100             */
  TVBF_ERR_WORKSPACE = -4    /* workspace too small              */
};

/* text operand precision of the tensor-core pass (candidates are always rescored in fp64) */
enum { TVBF_TEXT_FP16 = 0, TVBF_TEXT_BF16 = 1 };

/* how a feature group reaches the scorer */
enum {
  TVBF_GROUP_ABSENT = 0, /* contributes 0                                                       */
  TVBF_GROUP_PACKED = 1, /* genre: 64-bit multi-hot mask; metadata: one-hot category ids         */
  TVBF_GROUP_FOLDED = 2  /* arbitrary float features: normalised, scaled by sqrt(w) and appended */
                         /* as extra K columns of the tensor-core operand                        */
};

enum { TVBF_META_MEAN3 = 0, TVBF_META_HSTACK = 1 };

/* Device-resident, prepared features of one catalogue (built by the tvbf_prep_* calls).
 * Replaces the five matrices populate_database.py:125-131 loads and the per-iteration
 * normalisations inside cosine_similarity (populate_database.py:180-186). */
typedef struct tvbf_features {
  int32_t n_shows;           /* N                                                             */
  int32_t n_pad;             /* rows of operand / col_side / meta_scale; multiple of 256      */
  int32_t k_pad;             /* operand columns: text vocab + folded columns, padded to 64    */
  int32_t text_dtype;        /* TVBF_TEXT_*                                                   */
  int32_t text_scale_log2;   /* operand text columns hold x * 2^s                             */
  int32_t vocab;             /* V                                                             */
  const void* operand;       /* [n_pad, k_pad] fp16/bf16 row-major (K-major), zero padded     */
  const int64_t* text_indptr;  /* [N+1] CSR of the L2-normalised fp64 text matrix             */
  const int32_t* text_indices; /* sorted within each row                                      */
  const double* text_values;
  int32_t genre_mode;        /* TVBF_GROUP_*                                                  */
  int32_t genre_dim;         /* G                                                             */
  const double* genre_dense; /* FOLDED: [N, G] L2-normalised fp64 rows (exact rescoring)      */
  int32_t meta_mode;         /* TVBF_GROUP_*                                                  */
  int32_t meta_kind;         /* TVBF_META_*: mean of 3 cosines (populate_database.py:184-187) */
                             /* or cosine of the hstack (similarity_computer.py:84-86)        */
  int32_t meta_groups;       /* FOLDED: number of dense groups (3 for MEAN3, 1 for HSTACK)    */
  int32_t meta_dims[3];
  const double* meta_dense[3]; /* FOLDED: [N, dims[g]] L2-normalised fp64 rows                */
  const void* col_side;      /* [n_pad] 16-byte records {u64 genre bits, f32 1/sqrt(popc),    */
                             /*  u32 one-hot bits platform | type<<P | language<<(P+T)}       */
  const float* meta_scale;   /* [n_pad] MEAN3: 1/sqrt(3) ; HSTACK: 1/sqrt(#categories) or 0   */
  const uint64_t* genre_hi;  /* [n_pad] genre bits 64..127 (multi-hot genres with 64 < G <= 128; zero    */
                             /* padded), NULL for G <= 64: the popcount then runs over two words        */
  int32_t text_signed;       /* 1: text values may be negative (embeddings, SVD): the candidate   */
                             /* pass then bounds the fp16 error absolutely instead of relative to */
                             /* the accumulator (cancellation); 0 for TF-IDF                      */
  int32_t bits_folded;       /* 1: besides the packed records, the operand carries the PACKED genre */
                             /* and metadata groups as columns fold_col0 .. fold_col0 + genre_dim +  */
                             /* 32 (tvbf_prep_fold_bits), scaled so that the tensor-core accumulator */
                             /* is the whole hybrid for fold_weights: the candidate pass then skips  */
                             /* its popcounts (small vocabularies, where the epilogue is the bound); */
                             /* rescoring still uses the packed records                              */
  int32_t fold_col0;
  double fold_weights[3];    /* genre / text / metadata weights baked by tvbf_prep_fold_bits         */
  int32_t text_cols;         /* 0: text column c of the operand is vocabulary column c.  > 0: the  */
                             /* operand carries MERGED text (tvbf_prep_csr_to_operand_mapped) in   */
                             /* columns [0, text_cols): for non-negative text the tensor-core dot  */
                             /* is an upper bound of the text cosine, not the cosine; only the      */
                             /* candidate pass takes such an operand (needs text_signed == 0)       */
  int64_t text_nnz;          /* entries of the text CSR (text_indptr[N]): sizes the column-major    */
                             /* copy the exact row kernel builds in its workspace                   */
} tvbf_features;

/* Parameters of one top-K job: populate_database.py:85-91 (weights, top_n_per_show,
 * min_similarity) / content_based_service.py:262-264. */
typedef struct tvbf_params {
  double genre_weight, text_weight, metadata_weight; /* used as given (already normalised by  */
                                                     /* the caller for variants A/C)          */
  double min_similarity;  /* keep score >= min_similarity (populate_database.py:204-205)      */
  int32_t k;              /* top_n_per_show                                                   */
  int32_t exclude_self;   /* populate_database.py:199-200                                     */
  int32_t row_begin;      /* first source row of this shard (multiple of 128)                 */
  int32_t row_end;        /* one past the last source row                                     */
  int32_t splits;         /* column splits per row block (0 = choose)                         */
  int32_t candidates;     /* K' candidates kept per (row, split) before rescoring (0=choose)  */
  int32_t force_exact;    /* 1: send every row through the exact fp64 row kernel              */
  int32_t skip_fallback;  /* 1: do not repair flagged rows (diagnostics only)                 */
  double text_rel_err;    /* 0 = default bound for text_dtype                                 */
  int32_t phases;         /* 0 = all; else bitmask 1: K1 candidate pass, 2: K5 rescore+certify, */
                          /* 4: K6 exact repair -- lets a caller time the kernels separately     */
                          /* (same workspace must be passed to every phase call)                 */
  int32_t tuning;         /* 0 = defaults. bits 0-3: tcgen05 cta_group (1 or 2; default 2);     */
                          /* bits 4-11: producer pacing chunk in 64-wide k-blocks (default 16,   */
                          /* 255 = off); bits 12-15: pacing slack in chunks (default 2);        */
                          /* bits 16-19: smem ring stages; bits 20-21: symmetric mode (0 auto,  */
                          /* 1 off, 2 on: compute only tiles on/above the diagonal and feed     */
                          /* both shows of every score); bits 22-27: column-tile stride of the  */
                          /* symmetric sweep's threshold seed pass (0 auto, 1..48 as given,     */
                          /* 49..62 -> 48 + 8 per step, 63 none); bits 28-29: 16 epilogue warps in the  */
                          /* symmetric sweep (0 auto: k_pad <= 6144, 1 off, 2 on); bit 30:           */
                          /* non-cooperative launch                                                 */
} tvbf_params;

/* Result table of the shard rows [row_begin, row_end): the a9 record stream of
 * populate_database.py:211-217 in columnar form. */
typedef struct tvbf_topk_out {
  int32_t* indices;  /* [rows, k] column index of the similar show, -1 padded                 */
  int32_t* counts;   /* [rows]   number of valid entries (0 -> show omitted, :220-221)        */
  double* hybrid;    /* [rows, k] similarity_score                                            */
  double* genre;     /* [rows, k] genre_score                                                 */
  double* text;      /* [rows, k] text_score                                                  */
  double* metadata;  /* [rows, k] metadata_score                                              */
  int32_t* stats;    /* [8] device ints: 0 flagged rows repaired by the exact kernel,         */
                     /*     1 candidate pairs rescored, 2 / 3 flagged rows with / without text,*/
                     /*     5 rows repaired by the second sweep of tvbf_refresh_topk,         */
                     /*     rest reserved                                                     */
} tvbf_topk_out;

int tvbf_version(void);
const char* tvbf_last_error(void);
/* cumulative number of CUDA kernels this library has launched in this process */
uint64_t tvbf_kernel_launches(void);
/* K1 launches that the runtime refused as cooperative (a profiler patched the kernel) and that
 * were retried as plain launches; 0 in normal operation */
uint64_t tvbf_noncooperative_fallbacks(void);
/* sm count and compute capability of the current device; TVBF_ERR_UNSUPPORTED unless 10.x */
int tvbf_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);

/* ---- K0: feature preparation (replaces sklearn normalize() inside every cosine_similarity
 *      call, populate_database.py:180-186, and the dtype promotion of check_pairwise_arrays) -- */
/* values_out[e] = values[e] / ||row||_2 in fp64; zero rows untouched. */
int tvbf_prep_csr_normalize(const int64_t* indptr, const double* values, int32_t n_rows,
                            double* values_out, void* stream);
/* scatter the normalised CSR rows into operand[:, col_offset + c] = x * scale (fp16/bf16).
 * operand must be zero-initialised. */
int tvbf_prep_csr_to_operand(const int64_t* indptr, const int32_t* indices, const double* values,
                             int32_t n_rows, void* operand, int32_t k_pad, int32_t col_offset,
                             double scale, int32_t dtype, void* stream);
/* ---- merged text operand (large vocabularies, non-negative text) ----------------------------------
 * A merge plan maps the V vocabulary columns onto text_cols < V operand columns: the text_cols / 2
 * columns with the most non-zeros (document frequency; ties by ascending column) keep a column of
 * their own, the others are dealt round-robin by that rank over the remaining columns.
 * col_map[V]: operand column of every vocabulary column; slot_ptr[text_cols + 1] / slot_cols[V]:
 * the vocabulary columns of every operand column (CSR, in rank order).  Deterministic: the same CSR
 * gives the same plan on every GPU.  Fails unless every operand column takes at most 4096 vocabulary
 * columns (a merged entry of a unit row stays <= 64 before the 2^s scale, far below fp16's range). */
size_t tvbf_merge_plan_workspace_bytes(int32_t vocab);
int tvbf_merge_plan(const int64_t* indptr, const int32_t* indices, int32_t n_rows, int32_t vocab,
                    int32_t text_cols, int32_t* col_map, int32_t* slot_ptr, int32_t* slot_cols,
                    void* workspace, size_t workspace_bytes, void* stream);
/* tvbf_prep_csr_to_operand through a merge plan: operand[r, col_offset + col_map[c]] = sum of x * scale
 * over the row's entries that share that column, summed in fp64 in slot_cols order and rounded once
 * (fp16 / bf16).  operand must be zero-initialised. */
int tvbf_prep_csr_to_operand_mapped(const int64_t* indptr, const int32_t* indices, const double* values,
                                    int32_t n_rows, const int32_t* col_map, const int32_t* slot_ptr,
                                    const int32_t* slot_cols, void* operand, int32_t k_pad, int32_t col_offset,
                                    double scale, int32_t dtype, void* stream);
/* Recycling an operand buffer: store 0 at every position the CSR of the catalogue it held had set
 * (one 2-byte store per old non-zero instead of a memset of the whole n_pad x k_pad array). */
int tvbf_prep_clear_csr_positions(const int64_t* indptr, const int32_t* indices, int32_t n_rows,
                                  void* operand, int32_t k_pad, int32_t col_offset, int32_t dtype,
                                  void* stream);
/* Several GPUs: replicate this GPU's slices of a set of identically laid out buffers into every
 * peer's copy with plain stores over NVLink (peer mappings, e.g. torch symmetric memory):
 * for every field f and every peer p != rank,
 *   peer_base[p] + offsets[f] .. + bytes[f]  <-  peer_base[rank] + offsets[f] .. + bytes[f].
 * Replaces the all-gather of the [N, k] result tables (each rank has just written its row shard of
 * every field); the caller follows it with a device-side barrier.  n_fields <= 8, world <= 16,
 * offsets and sizes multiples of 4 bytes. */
int tvbf_peer_push(const uint64_t* peer_base, int32_t world, int32_t rank, const uint64_t* offsets,
                   const uint64_t* bytes, int32_t n_fields, void* stream);
/* cudaMemsetAsync(ptr, 0, bytes) on `stream` (fresh operand / column-side buffers). */
int tvbf_device_zero(void* ptr, size_t bytes, void* stream);
/* out[r, :] = in[r, :] / ||in[r, :]||_2 (fp64, zero rows stay zero). */
int tvbf_prep_dense_normalize(const double* in, int32_t n_rows, int32_t dim, double* out,
                              void* stream);
/* operand[r, col_offset + c] = dense[r, c] * scale. */
int tvbf_prep_dense_to_operand(const double* dense, int32_t n_rows, int32_t dim, void* operand,
                               int32_t k_pad, int32_t col_offset, double scale, int32_t dtype,
                               void* stream);
/* Packed genre / metadata records -> operand columns [col0, col0 + genre_dim + 32): genre column g of
 * show i holds scale_genre / sqrt(popcount_i) where bit g is set, metadata column b holds
 * scale_meta * meta_scale[i] where one-hot bit b is set, 0 elsewhere (every one of the columns is
 * written).  With scale_group = 2^s * sqrt(w_group / w_text) the accumulator of the text GEMM becomes
 * 2^2s / w_text times the hybrid of populate_database.py:190-192. */
int tvbf_prep_fold_bits(const void* col_side, const uint64_t* genre_hi, const float* meta_scale,
                        int32_t n_rows, int32_t genre_dim, void* operand, int32_t k_pad, int32_t col0,
                        double scale_genre, double scale_meta, int32_t dtype, void* stream);
/* genre multi-hot bytes [n_rows, dim <= 128] -> col_side[].genre_bits / genre_rnorm (+ genre_hi[] for
 * the columns 64.., required when dim > 64, [n_pad] entries zeroed by the caller). */
int tvbf_prep_genre_bits(const uint8_t* genre, int32_t n_rows, int32_t dim, void* col_side,
                         uint64_t* genre_hi, void* stream);
/* one-hot bytes of platform/type/language (P+T+L <= 32) -> col_side[].meta_bits and meta_scale[]. Rows
 * [n_rows, n_pad) are filled with "none". */
int tvbf_prep_meta_ids(const uint8_t* platform, int32_t p_dim, const uint8_t* type, int32_t t_dim,
                       const uint8_t* language, int32_t l_dim, int32_t n_rows, int32_t n_pad,
                       int32_t meta_kind, void* col_side, float* meta_scale, void* stream);

/* ---- device-side ingest of the raw arrays of compute_features.py:115-129 (what np.load / load_npz
 *      hand over: int64 multi-hot genres, float64 / bool one-hots, a scipy CSR with int32 or int64
 *      index arrays): classification and narrowing happen on the GPU, the host only copies bytes.
 *      dtype codes: 0 uint8 / bool, 1 int32, 2 int64, 3 float32, 4 float64.  `flags` is one device
 *      int32 the kernels OR into: 1 genre not {0,1}-valued, 2 metadata not one-hot, 4 CSR rows not
 *      strictly ascending (unsorted / duplicates), 8 negative text values.  With 1 or 2 set the
 *      packed words are meaningless and the caller takes the general (folded float) path. */
int tvbf_ingest_genre(const void* raw, int32_t dtype, int32_t n_rows, int32_t n_pad, int32_t dim, void* col_side,
                      uint64_t* genre_hi /* [n_pad], required for dim > 64 */, int32_t* flags, void* stream);
int tvbf_ingest_meta(const void* platform, int32_t p_dtype, int32_t p_dim, const void* type, int32_t t_dtype,
                     int32_t t_dim, const void* language, int32_t l_dtype, int32_t l_dim, int32_t n_rows,
                     int32_t n_pad, int32_t meta_kind, void* col_side, float* meta_scale, int32_t* flags,
                     void* stream);
/* raw CSR -> int64 indptr[n_rows + 1], int32 indices, float64 values (not yet normalised) */
int tvbf_ingest_csr(const void* indptr_raw, int32_t indptr64, const void* indices_raw, int32_t indices64,
                    const void* values_raw, int32_t values64, int32_t n_rows, int64_t* indptr, int32_t* indices,
                    double* values, int32_t* flags, void* stream);

/* ---- K1+K4+K5(+K6): hybrid all-pairs score -> per-row top-K
 *      (replaces the loop populate_database.py:170-218 and content_based_service.py:293-308) - */
size_t tvbf_topk_workspace_bytes(const tvbf_features* f, const tvbf_params* p);
int tvbf_hybrid_topk(const tvbf_features* f, const tvbf_params* p, const tvbf_topk_out* out,
                     void* workspace, size_t workspace_bytes, void* stream);
/* ---- weight sweep (BASELINE config C5; notebooks/03 cell 6 of the reference compares weighting
 *      schemes by re-running everything): the same whole-catalogue job for n_weights <= 5 triples
 *      p[0..n) that differ ONLY in their weights, sharing ONE symmetric tensor-core sweep.  The
 *      epilogue scores every pair under every triple and keeps one shared candidate list per
 *      (triple, show); rescoring, certificate and exact repair run per triple into out[w].  Every
 *      triple must be eligible for the symmetric sweep (tvbf_sym_eligible).  The tables are
 *      identical to those of n_weights separate tvbf_hybrid_topk calls. */
size_t tvbf_topk_sweep_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_weights);
int tvbf_hybrid_topk_sweep(const tvbf_features* f, const tvbf_params* p, int32_t n_weights,
                           const tvbf_topk_out* out, void* workspace, size_t workspace_bytes,
                           void* stream);
/* ---- the same job tile-sharded over several GPUs (symmetric sweep).  hybrid(i,j) == hybrid(j,i),
 *      so GPU `rank` of `world` computes only the tiles on/above the diagonal of the 256-row super
 *      blocks dealt to it and feeds BOTH shows of every score; it ends with partial candidate lists
 *      for ALL shows.  The super blocks are dealt in groups of consecutive blocks (one launch wave
 *      each), longest group first to the least-loaded GPU.  Call sequence per GPU, with one small
 *      collective (done by the caller) between the calls:
 *        tvbf_sym_seed       theta[n_pad]                   -> all_reduce(MAX, uint32) of theta
 *        tvbf_sym_sweep      cand[n_shows][L], cnt, bound   -> all_to_all: GPU r receives every GPU's
 *                                                              lists of ITS rows (or all_gather)
 *        tvbf_rescore_lists  rows [row_begin,row_end) of p  -> gather of the result tables
 *      L = tvbf_sym_list_len(); eligibility (packed groups, non-negative weights, positive
 *      min_similarity, k <= 100): tvbf_sym_eligible().  row_begin/row_end of p are ignored by the
 *      first two calls.
 *      Packed rows: with cand_cnt == cand_bound == NULL (tvbf_sym_sweep) / cnt_all == bound_all ==
 *      NULL (tvbf_rescore_lists) a candidate row is L + 1 entries of 8 bytes, the last one holding
 *      {int32 count, float bound}, so that ONE all-to-all moves everything. */
int tvbf_sym_eligible(const tvbf_features* f, const tvbf_params* p);
int32_t tvbf_sym_list_len(const tvbf_features* f, const tvbf_params* p);
size_t tvbf_sym_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t world);
int tvbf_sym_seed(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                  uint32_t* theta, void* workspace, size_t workspace_bytes, void* stream);
int tvbf_sym_sweep(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                   uint32_t* theta, void* cand, int32_t* cand_cnt, float* cand_bound,
                   void* workspace, size_t workspace_bytes, void* stream);
/* tvbf_sym_sweep with the exchange FUSED into the compaction: every finished candidate row (packed,
 * L + 1 entries) is stored straight into the receive buffer of the GPU that rescores that show, over
 * NVLink peer mappings -- no all-to-all.  peer_ptrs: HOST array of `world` device addresses, entry r =
 * GPU r's receive buffer laid out [world][shard_rows][L + 1] x 8 bytes as mapped into THIS process
 * (e.g. torch symmetric memory's buffer_ptrs); show s is owned by GPU s / shard_rows and lands in
 * slice `rank` of its buffer.  The caller runs a cross-GPU barrier before tvbf_rescore_lists reads
 * its own buffer (cnt_all = bound_all = NULL, table_rows = shard_rows). */
int tvbf_sym_sweep_peer(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                        uint32_t* theta, const uint64_t* peer_ptrs, int32_t shard_rows, void* workspace,
                        size_t workspace_bytes, void* stream);
/* fp64 rescoring + certificate + exact repair of rows [p->row_begin, p->row_end) from `lists`
 * candidate tables laid out [lists][table_rows][L] that cover the shows
 * [table_row0, table_row0 + table_rows): (0, n_shows) after an all_gather, (row_begin, rows) after
 * an all_to_all.  Of the merged lists only the 2L largest upper bounds are rescored; the rest
 * joins the row's bound. */
int tvbf_rescore_lists(const tvbf_features* f, const tvbf_params* p, const void* cand_all,
                       const int32_t* cnt_all, const float* bound_all, int32_t lists,
                       int32_t table_row0, int32_t table_rows, const tvbf_topk_out* out,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---- append shows to a catalogue whose table exists (instead of the whole job again).
 *      f: the grown catalogue of n_shows = N + Q shows, rows [0, n_old = N) unchanged since `prev` was
 *      computed, rows [N, N + Q) the new shows in the same vocabulary and widths; prev: the [N, k]
 *      table of the old catalogue from a job with the same p (weights, k, min_similarity,
 *      exclude_self = 1).  Writes the [N + Q, k] table of the grown catalogue to `out` -- bit-identical
 *      to tvbf_hybrid_topk on f (indices, counts and the four scores; stats differ) -- and
 *      changed[r] = 1 for every old row r whose indices or counts differ from prev (0 otherwise:
 *      the row is byte-identical).  An old row that receives no new candidate above its threshold is
 *      copied from prev without rescoring.  Only the 256 x 256 tiles that hold a new show are computed; the
 *      old rows' thresholds start just below their previous k-th score.  Jobs tvbf_sym_eligible
 *      rejects, and signed text, are rejected (the caller runs the whole job).  `out` must not alias `prev`. */
size_t tvbf_append_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_old);
int tvbf_append_topk(const tvbf_features* f, const tvbf_params* p, int32_t n_old, const tvbf_topk_out* prev,
                     const tvbf_topk_out* out, int32_t* changed, void* workspace, size_t workspace_bytes,
                     void* stream);

/* ---- update the features of shows in a catalogue whose table exists (instead of the whole job again).
 *      f: the catalogue of n_shows shows AFTER the update, the rows rows[0 .. n_rows) (device array,
 *      sorted, distinct, in [0, n_shows)) with their new features, every other row unchanged since
 *      `prev` was computed, all in the same vocabulary and widths; prev: the [n_shows, k] table of the
 *      catalogue before the update from a job with the same p (weights, k, min_similarity,
 *      exclude_self = 1).  Writes the [n_shows, k] table of the updated catalogue to `out` --
 *      bit-identical to tvbf_hybrid_topk on f (indices, counts and the four scores; stats differ) --
 *      and changed[r] = 1 for every row r, updated or not, that differs from prev in any of the six
 *      fields (0 otherwise: the row is byte-identical).  Only the updated shows' rows are swept against
 *      all columns; a row that names no updated show and receives no candidate from one above its
 *      threshold is copied from prev without rescoring.  Jobs tvbf_sym_eligible rejects, and signed
 *      text, are rejected (the caller runs the whole job).  `out` must not alias `prev`. */
size_t tvbf_update_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_rows);
int tvbf_update_topk(const tvbf_features* f, const tvbf_params* p, const int32_t* rows, int32_t n_rows,
                     const tvbf_topk_out* prev, const tvbf_topk_out* out, int32_t* changed, void* workspace,
                     size_t workspace_bytes, void* stream);

/* ---- remove shows from a catalogue whose table exists (instead of the whole job again).
 *      f: the catalogue of n_shows shows AFTER the removal (the remaining shows in their old order, the
 *      same features as before); removed: the n_removed removed rows in the OLD numbering (device array,
 *      sorted, distinct, in [0, n_shows + n_removed)); prev: the [n_shows + n_removed, k] table of the
 *      catalogue before the removal from a job with the same p (weights, k, min_similarity,
 *      exclude_self = 1).  Writes the [n_shows, k] table of the remaining catalogue to `out` (new
 *      numbering) -- bit-identical to tvbf_hybrid_topk on f (indices, counts and the four scores; stats
 *      differ) -- and changed[r] = 1 for every new row r whose previous row names a removed show (0
 *      otherwise: the row is byte-identical to its previous row with the indices renumbered).  Only
 *      those rows are swept against all columns; every other row is copied without rescoring.  The call
 *      waits for the stream once, to size the sweep by their number.  Jobs tvbf_sym_eligible rejects,
 *      and signed text, are rejected (the caller runs the whole job).  `out` must not alias `prev`. */
size_t tvbf_remove_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_removed);
int tvbf_remove_topk(const tvbf_features* f, const tvbf_params* p, const int32_t* removed, int32_t n_removed,
                     const tvbf_topk_out* prev, const tvbf_topk_out* out, int32_t* changed, void* workspace,
                     size_t workspace_bytes, void* stream);

/* ---- refresh a catalogue whose table exists: remove, update and append shows in one call (instead of
 *      the whole job again).  f: the catalogue of n_shows = N - n_removed + n_appended shows AFTER the
 *      refresh -- the N - n_removed remaining shows in their old order, the updated ones with their new
 *      features, then the n_appended new shows, all in the same vocabulary and widths; removed: the
 *      removed rows, updated: the updated rows, both in the OLD numbering (device arrays, sorted,
 *      distinct, in [0, N), disjoint; NULL when empty); prev: the [N, k] table of the catalogue before the
 *      refresh from a job with the same p (weights, k, min_similarity, exclude_self = 1).  Writes the
 *      [n_shows, k] table of f to `out` (new numbering) -- bit-identical to tvbf_hybrid_topk on f
 *      (indices, counts and the four scores; stats differ) -- and changed[r] = 1 for every appended row
 *      and for every remaining row that differs in any of the six fields from its previous row with the
 *      indices renumbered (0 otherwise: the row is byte-identical to it).  Unlike tvbf_append_topk,
 *      whose changed flags cover the old rows only, the appended rows are flagged too.
 *      The updated and appended shows (S), and the remaining shows whose previous row names a removed show
 *      (A), are swept against all columns; a row outside those that names no show of S and receives no
 *      candidate from one above its threshold is copied without rescoring.  Rows outside S and A that fail
 *      the certificate are swept against all columns a second time (stats[5] counts them) instead of
 *      going to the exact kernel.  The call waits for the stream twice, to size the two sweeps.  Jobs
 *      tvbf_sym_eligible rejects, signed text, and an `out` aliasing `prev` are rejected (the caller runs
 *      the whole job); at least one show must remain. */
size_t tvbf_refresh_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int32_t n_removed,
                                    int32_t n_updated, int32_t n_appended);
int tvbf_refresh_topk(const tvbf_features* f, const tvbf_params* p, const int32_t* removed, int32_t n_removed,
                      const int32_t* updated, int32_t n_updated, int32_t n_appended, const tvbf_topk_out* prev,
                      const tvbf_topk_out* out, int32_t* changed, void* workspace, size_t workspace_bytes,
                      void* stream);

/* exact fp64 scoring of explicit source rows against all columns + exact top-K
 * (replaces get_recommendations_from_matrix, content_based_service.py:161-236, for any n). */
size_t tvbf_exact_workspace_bytes(const tvbf_features* f, int32_t n_rows_listed);
int tvbf_exact_rows(const tvbf_features* f, const tvbf_params* p, const int32_t* rows,
                    int32_t n_rows_listed, const tvbf_topk_out* out, void* workspace,
                    size_t workspace_bytes, void* stream);

/* same selection over rows of precomputed N x N float64 matrices: the service's matrix path
 * (_load_similarity_matrices + get_recommendations_from_matrix,
 * content_based_service.py:113-140,161-236).  Workspace: tvbf_exact_workspace_bytes-sized
 * (min(2*SMs, n_rows_listed) * n * 8 bytes). `rows` are absolute row numbers. */
int tvbf_matrix_rows_topk(const double* hybrid, const double* genre, const double* text,
                          const double* metadata, int32_t n, const tvbf_params* p,
                          const int32_t* rows, int32_t n_rows_listed, const tvbf_topk_out* out,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- full-matrix variant (SimilarityComputer, ml/similarity_computer.py:30-190) ------------- */
/* csr (normalised) -> dense fp64 [n_rows, dim]; dense must be zero-initialised. */
int tvbf_csr_to_dense_f64(const int64_t* indptr, const int32_t* indices, const double* values,
                          int32_t n_rows, int32_t dim, double* dense, void* stream);
/* out[i, j] = sum_c x[i, c] * x[j, c]  (x already L2-normalised): cosine_similarity(X),
 * similarity_computer.py:41,58,86. */
int tvbf_cosine_matrix_f64(const double* x, int32_t n_rows, int32_t dim, double* out,
                           void* stream);
/* out = wg*g + wt*t + wm*m elementwise, similarity_computer.py:122-124. */
int tvbf_hybrid_combine_f64(const double* g, const double* t, const double* m, double wg,
                            double wt, double wm, int64_t count, double* out, void* stream);
/* mean / std / min / max / median of the strict upper triangle (similarity_computer.py:171-190).
 * Synchronises `stream`; out5 is a HOST pointer. */
size_t tvbf_matrix_stats_workspace_bytes(void);
int tvbf_matrix_stats_f64(const double* mat, int32_t n, double* out5_host, void* workspace,
                          size_t workspace_bytes, void* stream);

/* ---- streaming statistics for catalogues whose N x N matrices cannot exist
 *      (get_similarity_statistics, ml/similarity_computer.py:171-190, as used by
 *      scripts/compute_similarities.py:119-131).  One symmetric tensor-core sweep accumulates, for
 *      genre / text / metadata / hybrid over the strict upper triangle: sum and sum of squares
 *      (fp64), min / max (fp32), the count of exact zeros and a 1024-bin histogram; `accum` is a
 *      device buffer of tvbf_stats_accum_bytes() holding, in this order:
 *        double sum[4], sumsq[4]; uint64 zeros[4]; uint64 hist[4][1024]; uint32 min_bits[4],
 *        max_bits[4]; float hi[4]; int32 n_cand; int32 cand_ij[2][2048][2]; float cand_val[2][2048]
 *      (cand_*: argmax candidates of text and hybrid, to be rescored exactly with
 *      tvbf_score_pairs).  Text values come from the fp16 operand (relative error <= 1e-3 per
 *      element, correlated per vocabulary column): mean / std agree with float64 to ~1e-5
 *      relative, the median to one bin. */
/*        ...; double sum_gm (sum of genre * metadata)
 *      The fp16 text operand limits mean / std of text and hybrid to ~1e-5; tvbf_text_moments below
 *      delivers the text-dependent sums exactly (float64), from which the caller assembles mean and
 *      std of text and hybrid to ~1e-9 (engine.similarity_stats). */
size_t tvbf_stats_accum_bytes(void);
#define TVBF_MOMENTS 24
/* exact float64 moments over ALL (i, j) pairs, no N x N; out8 has TVBF_MOMENTS entries:
 *   [0..7]   sum t, sum t^2 (0 unless with_gram), sum g*t, sum m*t,
 *            diagonal: sum_i t_ii, sum_i t_ii^2, sum_i g_ii t_ii, sum_i m_ii t_ii
 *   [8..12]  sum g, sum g^2, sum m, sum m^2, sum g*m
 *   [13..17] diagonal: sum_i g_ii, g_ii^2, m_ii, m_ii^2, g_ii m_ii
 * (t / g / m = text / genre / metadata cosine; strict upper triangle = (all - diagonal) / 2).
 * with_gram needs a [vocab, vocab] float64 Gram matrix in the workspace (800 MB at V = 10 000).
 * Packed genre / metadata only.  out8 is a DEVICE pointer. */
size_t tvbf_text_moments_workspace_bytes(const tvbf_features* f, int32_t with_gram);
int tvbf_text_moments(const tvbf_features* f, int32_t with_gram, double* out8, void* workspace,
                      size_t workspace_bytes, void* stream);
int tvbf_similarity_stats(const tvbf_features* f, const tvbf_params* p, void* accum, void* workspace,
                          size_t workspace_bytes, void* stream);
/* exact float64 scores of explicit pairs: out4[p] = {hybrid, genre, text, metadata} of
 * (pairs[2p], pairs[2p+1]). */
int tvbf_score_pairs(const tvbf_features* f, const tvbf_params* p, const int32_t* pairs,
                     int32_t n_pairs, double* out4, void* stream);

/* ---- every neighbour at or above a threshold (the loop populate_database.py:170-218 cut by
 *      min_similarity alone): one variable-length row per show instead of a [N, k] table.  Two calls,
 *      because the size of the result is known only after the sweep:
 *        tvbf_neighbours_sweep   the tiles on/above the diagonal of the symmetric sweep; writes every
 *                                pair {int32 i, int32 j}, i < j, whose tensor-core upper bound U
 *                                (>= the exact hybrid) exceeds theta (the top-k sweep's initial
 *                                threshold: min_similarity rounded to the nearest fp32, one fp32 step
 *                                down; always below min_similarity) to pairs[0 .. capacity), in no
 *                                particular order, and the number of such pairs to *n_candidates
 *                                (DEVICE int64).  The count goes on past capacity (nothing is stored
 *                                there): when it exceeds capacity, run the sweep again with at least
 *                                that capacity.  pairs may be NULL when capacity is 0 (count only).  Every pair whose exact
 *                                score is >= min_similarity is a candidate.
 *        tvbf_neighbours_finish  n_candidates (HOST value, <= the sweep's capacity) pairs of the sweep
 *                                scored in float64 exactly as tvbf_score_pairs and K5 score them
 *                                (bit-identical), kept when hybrid >= min_similarity, emitted as (i, j)
 *                                and (j, i), plus (i, i) when p->exclude_self == 0 and its score
 *                                qualifies.  Row r is entries row_ptr[r] .. row_ptr[r + 1] of indices /
 *                                hybrid / genre / text / metadata, ordered by (hybrid descending, column
 *                                ascending) and cut to max_per_row entries (0: no cap); row_ptr has
 *                                n_shows + 1 int64 entries and row_ptr[n_shows] is the number of entries
 *                                written.  The outputs need room for 2 * n_candidates + n_shows entries.
 *                                With max_per_row = k, row r equals row r of tvbf_hybrid_topk's table
 *                                for the same p and k (indices, count and the four scores).
 *      Workspace: tvbf_neighbours_workspace_bytes for the sweep's capacity, shared by both calls.
 *      p supplies the weights, min_similarity and exclude_self; k, candidates, splits and the row range
 *      are ignored.  Jobs are taken when tvbf_sym_eligible takes them for the whole catalogue with
 *      exclude_self = 1 and without its k <= 100 condition, and min_similarity > 0; everything else
 *      (min_similarity <= 0, float (folded) groups, negative weights, ...) is refused with
 *      TVBF_ERR_INVALID and a message.  Neither call synchronises; the caller reads *n_candidates
 *      back before it sizes the finish.  Single GPU. */
size_t tvbf_neighbours_workspace_bytes(const tvbf_features* f, const tvbf_params* p, int64_t capacity);
int tvbf_neighbours_sweep(const tvbf_features* f, const tvbf_params* p, int32_t* pairs, int64_t capacity,
                          int64_t* n_candidates, void* workspace, size_t workspace_bytes, void* stream);
int tvbf_neighbours_finish(const tvbf_features* f, const tvbf_params* p, const int32_t* pairs, int64_t n_candidates,
                           int32_t max_per_row, int64_t* row_ptr, int32_t* indices, double* hybrid, double* genre,
                           double* text, double* metadata, void* workspace, size_t workspace_bytes, void* stream);

/* ---- diagnostics ---------------------------------------------------------------------------- */
/* host-only (no device): the work items of one K1 launch for a catalogue of col_tiles 256-column
 * tiles and super_blocks 256-row super blocks dealt to `world` GPUs; out[6 * item + {0..5}] =
 * {super block or -1, column split, tile0, tile1, real0, real1}: the item walks [tile0, tile1) for
 * the producer pacing and computes [real0, real1).  Returns the number of items.  Used by the CPU
 * tests to prove that every tile on/above the diagonal is computed exactly once. */
int32_t tvbf_debug_schedule(int32_t col_tiles, int32_t super_blocks, int32_t sb_per_group, int32_t splits,
                            int32_t world, int32_t rank, int32_t symmetric, int32_t* out,
                            int32_t max_items);
/* host-only: tensor-core tiles tvbf_append_topk executes for this job, out2 = {tiles of its threshold
 * seed pass over the super blocks that hold new shows, tiles of the append sweep} (256 x 256 x k_pad
 * each).  Fails like tvbf_append_workspace_bytes for a job the append does not take. */
int tvbf_append_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t n_old, int64_t* out2);
/* host-only: the work items of the append sweep of tvbf_append_topk for n_shows shows of which the
 * first n_old are old, on a device with sm_count SMs; out as tvbf_debug_schedule.  Returns the number
 * of items.  Used by the CPU tests to prove that every pair with a new show is computed exactly once. */
int32_t tvbf_debug_append_schedule(int32_t n_old, int32_t n_shows, int32_t sm_count, int32_t* out,
                                   int32_t max_items);
/* host-only: tensor-core tiles tvbf_update_topk executes for this job with n_rows updated shows,
 * out2 = {tiles of its threshold seed pass over the gathered rows, tiles of the update sweep}
 * (256 x 256 x k_pad each).  Fails like tvbf_update_workspace_bytes for a job the update does not take. */
int tvbf_update_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t n_rows, int64_t* out2);
/* host-only: tensor-core tiles tvbf_remove_topk executes for this job (f after the removal) when
 * n_rows remaining shows named a removed one, out2 = {tiles of its threshold seed pass over their
 * gathered rows, tiles of the repair sweep} (256 x 256 x k_pad each); the schedule is the update
 * sweep's for n_rows rows.  Fails like tvbf_remove_workspace_bytes for a job the removal does not take. */
int tvbf_remove_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t n_rows, int64_t* out2);
/* host-only: tensor-core tiles tvbf_refresh_topk executes for this job (f after the refresh) when
 * n_gathered rows are in S or A and n_repaired rows go to the second sweep, out4 = {seed pass tiles,
 * sweep tiles} of the refresh sweep, then of the second sweep (256 x 256 x k_pad each; 0 for a stage
 * without rows).  Both are the update sweep's schedule for their row counts.  Fails like
 * tvbf_refresh_workspace_bytes for a job the refresh does not take. */
int tvbf_refresh_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t n_gathered, int32_t n_repaired,
                            int64_t* out4);
/* host-only: the work items of the update sweep of tvbf_update_topk for q updated shows in a catalogue
 * of n_shows on a device with sm_count SMs; out as tvbf_debug_schedule (super block = block of 256
 * gathered rows).  Returns the number of items.  Used by the CPU tests to prove that every (gathered
 * row block, column tile) is computed exactly once. */
int32_t tvbf_debug_update_schedule(int32_t q, int32_t n_shows, int32_t sm_count, int32_t* out, int32_t max_items);
/* host-only: tensor-core tiles the candidate pass of this job executes -- out4 = {tiles of the
 * threshold seed pass, tiles of the main sweep, rows per tile (128 or 256; columns are 256 and the
 * depth is k_pad), 1 if the symmetric sweep is used}.  tile_sharded = 0: the job as tvbf_hybrid_topk
 * runs it for rows [row_begin, row_end) of p; 1: as tvbf_sym_seed + tvbf_sym_sweep run it on GPU
 * `rank` of `world`.  bench.py derives the executed FLOPs of its roofline line from this. */
int tvbf_plan_tiles(const tvbf_features* f, const tvbf_params* p, int32_t rank, int32_t world,
                    int32_t tile_sharded, int64_t* out4);
/* host-only: the constants of the candidate pass' upper bound for this job.  For a pair whose
 * source row has T non-zero operand entries and whose raw accumulator is a,
 *   U = wg*g + wm*m + out5[0]*a + (out5[1] + T*out5[2])*|a| + out5[3] + T*out5[4]  >=  exact hybrid
 * (api.cu: make_slack).  The tests check this inequality against float64. */
int tvbf_debug_slack(const tvbf_features* f, const tvbf_params* p, float* out5);
/* raw tensor-core tile dump: out[i, j] = sum_k operand[row0+i, k] * operand[col0+j, k] for a
 * 128 x 256 tile (fp32), used by the tests to validate descriptors and the error bound. */
int tvbf_debug_gemm_tile(const tvbf_features* f, int32_t row0, int32_t col0, float* out,
                         void* stream);
/* same through the cta_group::2 path: a 256 x 256 tile computed by a CTA pair. */
int tvbf_debug_gemm_tile_pair(const tvbf_features* f, int32_t row0, int32_t col0, float* out,
                              void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TVBF_H_ */
