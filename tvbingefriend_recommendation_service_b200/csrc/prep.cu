// K0 -- feature preparation kernels (HBM-bound, one pass over the inputs).
//
// They replace what sklearn does inside every cosine_similarity call of the reference
// (scripts/populate_database.py:180-186; ml/similarity_computer.py:41,58,86): dtype promotion to
// float64 and row-wise L2 normalisation with zero rows left untouched, done ONCE per catalogue
// instead of five times per source show, plus the packing of the binary groups.
#include "common.cuh"

#include <cub/device/device_radix_sort.cuh>

namespace {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(tvbf::kFullMask, v, o);
  return v;
}

// one warp per CSR row: values_out = values / sqrt(sum(values^2)); zero rows untouched
__global__ void csr_normalize_kernel(const int64_t* __restrict__ indptr,
                                     const double* __restrict__ values, int n_rows,
                                     double* __restrict__ out) {
  int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int64_t b = indptr[row], e = indptr[row + 1];
  double s = 0.0;
  for (int64_t i = b + lane; i < e; i += 32) s += values[i] * values[i];
  s = warp_sum(s);
  double norm = sqrt(s);
  if (norm == 0.0) norm = 1.0;
  for (int64_t i = b + lane; i < e; i += 32) out[i] = values[i] / norm;
}

template <typename T>
__device__ __forceinline__ T cvt_operand(double v);
template <>
__device__ __forceinline__ __half cvt_operand<__half>(double v) {
  return __double2half(v);  // round-to-nearest-even from fp64: a single rounding
}
template <>
__device__ __forceinline__ __nv_bfloat16 cvt_operand<__nv_bfloat16>(double v) {
  return __double2bfloat16(v);
}

template <typename T>
__global__ void csr_to_operand_kernel(const int64_t* __restrict__ indptr,
                                      const int32_t* __restrict__ indices,
                                      const double* __restrict__ values, int n_rows,
                                      T* __restrict__ operand, int k_pad, int col_offset,
                                      double scale) {
  int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int64_t b = indptr[row], e = indptr[row + 1];
  T* dst = operand + static_cast<size_t>(row) * k_pad + col_offset;
  for (int64_t i = b + lane; i < e; i += 32) dst[indices[i]] = cvt_operand<T>(values[i] * scale);
}

// Merged text (tvbf_prep_csr_to_operand_mapped): one warp per row, one lane per entry.  An entry
// finds the row's other entries of its operand column by binary search for every vocabulary column of
// that slot (a handful, in slot_cols order); the lane of the first one present stores the fp64 sum,
// rounded once, and the others store nothing -- no atomics, the same bits on every run.
template <typename T>
__global__ void csr_to_operand_mapped_kernel(const int64_t* __restrict__ indptr,
                                             const int32_t* __restrict__ indices,
                                             const double* __restrict__ values, int n_rows,
                                             const int32_t* __restrict__ col_map,
                                             const int32_t* __restrict__ slot_ptr,
                                             const int32_t* __restrict__ slot_cols,
                                             T* __restrict__ operand, int k_pad, int col_offset, double scale) {
  int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t b = indptr[row], e = indptr[row + 1];
  T* dst = operand + static_cast<size_t>(row) * k_pad + col_offset;
  for (int64_t i = b + lane; i < e; i += 32) {
    const int c = indices[i];
    const int s = col_map[c];
    const int p0 = slot_ptr[s], p1 = slot_ptr[s + 1];
    if (p1 - p0 == 1) {
      dst[s] = cvt_operand<T>(values[i] * scale);
      continue;
    }
    double sum = 0.0;
    int owner = -1;
    for (int p = p0; p < p1; ++p) {
      const int c2 = slot_cols[p];
      int64_t lo = b, hi = e;          // first position in [b, e) whose column is >= c2
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (indices[mid] < c2) lo = mid + 1; else hi = mid;
      }
      if (lo < e && indices[lo] == c2) {
        if (owner < 0) owner = c2;
        sum += values[lo];
      }
    }
    if (owner == c) dst[s] = cvt_operand<T>(sum * scale);
  }
}

// document frequency of every vocabulary column: an integer histogram of the CSR's column indices
__global__ void column_df_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                 int n_rows, int vocab, int32_t* __restrict__ df) {
  const int64_t nnz = indptr[n_rows];
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < nnz;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = indices[i];
    if (c >= 0 && c < vocab) atomicAdd(df + c, 1);
  }
}

__global__ void iota_kernel(int32_t* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = i;
}

// order[r] = vocabulary column of rank r (descending frequency).  Ranks below head keep their own
// operand column r; rank r >= head goes to head + (r - head) % tail, so slot head + t holds the ranks
// head + t + j * tail, j = 0, 1, ...: q + 1 of them for t < rem, q for the others.
__global__ void merge_plan_fill_kernel(const int32_t* __restrict__ order, int vocab, int text_cols,
                                       int32_t* __restrict__ col_map, int32_t* __restrict__ slot_ptr,
                                       int32_t* __restrict__ slot_cols) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int head = text_cols / 2, tail = text_cols - head;
  const int q = (vocab - head) / tail, rem = (vocab - head) % tail;
  if (i < vocab) {
    const int c = order[i];
    if (i < head) {
      col_map[c] = i;
      slot_cols[i] = c;
    } else {
      const int t = (i - head) % tail, j = (i - head) / tail;
      col_map[c] = head + t;
      slot_cols[head + t * q + min(t, rem) + j] = c;
    }
  }
  if (i <= text_cols) {
    const int t = i - head;
    slot_ptr[i] = i <= head ? i : (i == text_cols ? vocab : head + t * q + min(t, rem));
  }
}

// un-scatter: zero the operand entries a previous catalogue's CSR had set (recycling an operand
// buffer costs one 2-byte store per old non-zero instead of a memset of the whole N x V array)
template <typename T>
__global__ void csr_clear_operand_kernel(const int64_t* __restrict__ indptr,
                                         const int32_t* __restrict__ indices, int n_rows,
                                         T* __restrict__ operand, int k_pad, int col_offset) {
  int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int64_t b = indptr[row], e = indptr[row + 1];
  T* dst = operand + static_cast<size_t>(row) * k_pad + col_offset;
  for (int64_t i = b + lane; i < e; i += 32) dst[indices[i]] = T(0.0f);
}

__global__ void dense_normalize_kernel(const double* __restrict__ in, int n_rows, int dim,
                                       double* __restrict__ out) {
  int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const double* x = in + static_cast<size_t>(row) * dim;
  double s = 0.0;
  for (int c = 0; c < dim; ++c) s += x[c] * x[c];
  double norm = sqrt(s);
  if (norm == 0.0) norm = 1.0;
  double* y = out + static_cast<size_t>(row) * dim;
  for (int c = 0; c < dim; ++c) y[c] = x[c] / norm;
}

template <typename T>
__global__ void dense_to_operand_kernel(const double* __restrict__ dense, int n_rows, int dim,
                                        T* __restrict__ operand, int k_pad, int col_offset,
                                        double scale) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t total = static_cast<size_t>(n_rows) * dim;
  if (i >= total) return;
  size_t row = i / dim;
  int c = static_cast<int>(i - row * dim);
  operand[row * k_pad + col_offset + c] = cvt_operand<T>(dense[i] * scale);
}

__global__ void genre_bits_kernel(const uint8_t* __restrict__ genre, int n_rows, int dim,
                                  TvbfColSide* __restrict__ col_side, unsigned long long* __restrict__ genre_hi) {
  int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_rows) return;
  const uint8_t* g = genre + static_cast<size_t>(row) * dim;
  unsigned long long bits = 0ull, hi = 0ull;
  for (int c = 0; c < dim; ++c)
    if (g[c]) {
      if (c < 64) bits |= 1ull << c; else hi |= 1ull << (c - 64);
    }
  int pc = __popcll(bits) + __popcll(hi);
  if (genre_hi != nullptr) genre_hi[row] = hi;
  col_side[row].genre_bits = bits;
  col_side[row].genre_rnorm = pc ? 1.0f / sqrtf(static_cast<float>(pc)) : 0.0f;
}

__device__ __forceinline__ uint32_t one_hot_bits(const uint8_t* m, int dim, int row, int offset) {
  if (m == nullptr || dim <= 0) return 0u;
  const uint8_t* x = m + static_cast<size_t>(row) * dim;
  uint32_t bits = 0u;
  for (int c = 0; c < dim; ++c)
    if (x[c]) bits |= 1u << (offset + c);
  return bits;
}

// one-hot platform / type / language rows -> one 32-bit mask per show; the number of matching
// groups of two shows is then popc(a & b)
__global__ void meta_bits_kernel(const uint8_t* __restrict__ platform, int p_dim,
                                 const uint8_t* __restrict__ type, int t_dim,
                                 const uint8_t* __restrict__ language, int l_dim, int n_rows,
                                 int n_pad, int meta_kind, TvbfColSide* __restrict__ col_side,
                                 float* __restrict__ meta_scale) {
  int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_pad) return;
  uint32_t bits = 0u;
  if (row < n_rows)
    bits = one_hot_bits(platform, p_dim, row, 0) | one_hot_bits(type, t_dim, row, p_dim) |
           one_hot_bits(language, l_dim, row, p_dim + t_dim);
  col_side[row].meta_bits = bits;
  const int valid = __popc(bits);
  float s;
  if (row >= n_rows) s = 0.0f;
  else if (meta_kind == TVBF_META_MEAN3) s = 0.57735026918962576f;  // 1/sqrt(3)
  else s = valid ? 1.0f / sqrtf(static_cast<float>(valid)) : 0.0f;
  meta_scale[row] = s;
}

// Packed records -> operand columns (tvbf_prep_fold_bits): one thread per (show, column), consecutive
// threads write consecutive 2-byte entries of a row.
template <typename T>
__global__ void fold_bits_kernel(const TvbfColSide* __restrict__ col_side,
                                 const unsigned long long* __restrict__ genre_hi,
                                 const float* __restrict__ meta_scale, int n_rows, int g_dim,
                                 T* __restrict__ operand, int k_pad, int col0, double scale_genre, double scale_meta) {
  const int width = g_dim + 32;
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<size_t>(n_rows) * width) return;
  const int row = static_cast<int>(i / width), c = static_cast<int>(i - static_cast<size_t>(row) * width);
  const TvbfColSide cs = col_side[row];
  double v = 0.0;   // one rounding, from fp64, like the text columns
  if (c < g_dim) {
    const unsigned long long word = c < 64 ? cs.genre_bits : genre_hi[row];
    if ((word >> (c & 63)) & 1ull) v = static_cast<double>(cs.genre_rnorm) * scale_genre;
  } else if ((cs.meta_bits >> (c - g_dim)) & 1u) {
    v = static_cast<double>(meta_scale[row]) * scale_meta;
  }
  operand[static_cast<size_t>(row) * k_pad + col0 + c] = cvt_operand<T>(v);
}

// tvbf_peer_push: blockIdx.y picks the peer, the blocks of a peer stride over 16-byte words (4-byte
// words for a field whose slice is not 16-byte aligned) of every field in turn.
struct PeerPush {
  unsigned long long base[16];
  unsigned long long off[8], bytes[8];
  int world, rank, n_fields;
};
__global__ void peer_push_kernel(const PeerPush a) {
  int p = static_cast<int>(blockIdx.y);
  if (p >= a.rank) ++p;   // every peer but this GPU itself
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x, stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (int f = 0; f < a.n_fields; ++f) {
    const unsigned long long src = a.base[a.rank] + a.off[f], dst = a.base[p] + a.off[f];
    if (((src | dst | a.bytes[f]) & 15ull) == 0ull) {
      const uint4* s = reinterpret_cast<const uint4*>(src);
      uint4* d = reinterpret_cast<uint4*>(dst);
      for (size_t i = tid; i < a.bytes[f] / 16; i += stride) d[i] = s[i];
    } else {
      const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
      uint32_t* d = reinterpret_cast<uint32_t*>(dst);
      for (size_t i = tid; i < a.bytes[f] / 4; i += stride) d[i] = s[i];
    }
  }
}

// ---- device-side ingest of the raw feature arrays (any of the dtypes numpy hands over) --------------
// dtype codes of the raw arrays: 0 uint8 / bool, 1 int32, 2 int64, 3 float32, 4 float64
__device__ __forceinline__ double load_raw(const void* p, int dtype, size_t i) {
  switch (dtype) {
    case 0: return static_cast<double>(static_cast<const uint8_t*>(p)[i]);
    case 1: return static_cast<double>(static_cast<const int32_t*>(p)[i]);
    case 2: return static_cast<double>(static_cast<const int64_t*>(p)[i]);
    case 3: return static_cast<double>(static_cast<const float*>(p)[i]);
    default: return static_cast<const double*>(p)[i];
  }
}

enum { INGEST_NOT_BINARY = 1, INGEST_NOT_ONE_HOT = 2, INGEST_NOT_CANONICAL = 4, INGEST_NEGATIVE_TEXT = 8 };

// genre multi-hot of any dtype -> col_side[].genre_bits / genre_rnorm; flags |= NOT_BINARY when a
// value is neither 0 nor 1 (the caller then takes the general float path)
__global__ void ingest_genre_kernel(const void* __restrict__ raw, int dtype, int n_rows, int n_pad, int dim,
                                    TvbfColSide* __restrict__ col_side, unsigned long long* __restrict__ genre_hi,
                                    int* __restrict__ flags) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_pad) return;
  unsigned long long bits = 0ull, hi = 0ull;
  bool bad = false;
  if (row < n_rows)
    for (int c = 0; c < dim; ++c) {
      const double v = load_raw(raw, dtype, static_cast<size_t>(row) * dim + c);
      bad |= !(v == 0.0 || v == 1.0);
      if (v != 0.0) {
        if (c < 64) bits |= 1ull << c; else hi |= 1ull << (c - 64);
      }
    }
  const int pc = __popcll(bits) + __popcll(hi);
  if (genre_hi != nullptr) genre_hi[row] = hi;
  col_side[row].genre_bits = bits;
  col_side[row].genre_rnorm = pc ? 1.0f / sqrtf(static_cast<float>(pc)) : 0.0f;
  if (bad) atomicOr(flags, INGEST_NOT_BINARY);
}

__device__ __forceinline__ uint32_t ingest_group(const void* raw, int dtype, int dim, int row, int offset, bool* bad) {
  uint32_t bits = 0u;
  int ones = 0;
  for (int c = 0; c < dim; ++c) {
    const double v = load_raw(raw, dtype, static_cast<size_t>(row) * dim + c);
    *bad |= !(v == 0.0 || v == 1.0);
    if (v != 0.0) { bits |= 1u << (offset + c); ++ones; }
  }
  *bad |= ones > 1;
  return bits;
}

// platform / type / language one-hot rows of any dtype -> col_side[].meta_bits and meta_scale[];
// flags |= NOT_ONE_HOT when a row is not {0,1}-valued with at most one 1 per group
__global__ void ingest_meta_kernel(const void* __restrict__ platform, int p_dtype, int p_dim,
                                   const void* __restrict__ type, int t_dtype, int t_dim,
                                   const void* __restrict__ language, int l_dtype, int l_dim, int n_rows,
                                   int n_pad, int meta_kind, TvbfColSide* __restrict__ col_side,
                                   float* __restrict__ meta_scale, int* __restrict__ flags) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n_pad) return;
  uint32_t bits = 0u;
  bool bad = false;
  if (row < n_rows)
    bits = ingest_group(platform, p_dtype, p_dim, row, 0, &bad) |
           ingest_group(type, t_dtype, t_dim, row, p_dim, &bad) |
           ingest_group(language, l_dtype, l_dim, row, p_dim + t_dim, &bad);
  col_side[row].meta_bits = bits;
  const int valid = __popc(bits);
  float s;
  if (row >= n_rows) s = 0.0f;
  else if (meta_kind == TVBF_META_MEAN3) s = 0.57735026918962576f;
  else s = valid ? 1.0f / sqrtf(static_cast<float>(valid)) : 0.0f;
  meta_scale[row] = s;
  if (bad) atomicOr(flags, INGEST_NOT_ONE_HOT);
}

// text CSR as scipy hands it over (int32 or int64 indptr / indices, float32 or float64 data) ->
// int64 indptr, int32 indices, float64 values; flags |= NOT_CANONICAL when a row's column indices
// are not strictly ascending (unsorted or duplicated), NEGATIVE_TEXT when a value is negative
__global__ void ingest_csr_kernel(const void* __restrict__ indptr_raw, int indptr64,
                                  const void* __restrict__ indices_raw, int indices64,
                                  const void* __restrict__ values_raw, int values64, int n_rows,
                                  int64_t* __restrict__ indptr, int32_t* __restrict__ indices,
                                  double* __restrict__ values, int* __restrict__ flags) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row > n_rows) return;
  auto ptr_at = [&](int r) -> int64_t {
    return indptr64 ? static_cast<const int64_t*>(indptr_raw)[r]
                    : static_cast<int64_t>(static_cast<const int32_t*>(indptr_raw)[r]);
  };
  if (row == n_rows) {
    if (lane == 0) indptr[n_rows] = ptr_at(n_rows);
    return;
  }
  const int64_t b = ptr_at(row), e = ptr_at(row + 1);
  if (lane == 0) indptr[row] = b;
  int bad = 0;
  for (int64_t i = b + lane; i < e; i += 32) {
    const int64_t c = indices64 ? static_cast<const int64_t*>(indices_raw)[i]
                                : static_cast<int64_t>(static_cast<const int32_t*>(indices_raw)[i]);
    const double v = values64 ? static_cast<const double*>(values_raw)[i]
                              : static_cast<double>(static_cast<const float*>(values_raw)[i]);
    if (i > b) {
      const int64_t prev = indices64 ? static_cast<const int64_t*>(indices_raw)[i - 1]
                                     : static_cast<int64_t>(static_cast<const int32_t*>(indices_raw)[i - 1]);
      if (prev >= c) bad |= INGEST_NOT_CANONICAL;
    }
    if (v < 0.0) bad |= INGEST_NEGATIVE_TEXT;
    indices[i] = static_cast<int32_t>(c);
    values[i] = v;
  }
  if (bad) atomicOr(flags, bad);
}

__global__ void csr_to_dense_kernel(const int64_t* __restrict__ indptr,
                                    const int32_t* __restrict__ indices,
                                    const double* __restrict__ values, int n_rows, int dim,
                                    double* __restrict__ dense) {
  int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int64_t b = indptr[row], e = indptr[row + 1];
  double* dst = dense + static_cast<size_t>(row) * dim;
  for (int64_t i = b + lane; i < e; i += 32) dst[indices[i]] = values[i];
}

inline unsigned blocks_for(size_t work, unsigned per_block) {
  return static_cast<unsigned>((work + per_block - 1) / per_block);
}

}  // namespace

extern "C" {

int tvbf_prep_csr_normalize(const int64_t* indptr, const double* values, int32_t n_rows,
                            double* values_out, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(indptr && values_out && n_rows >= 0, "tvbf_prep_csr_normalize: bad arguments");
  if (n_rows == 0) return TVBF_OK;
  auto st = static_cast<cudaStream_t>(stream);
  csr_normalize_kernel<<<blocks_for(static_cast<size_t>(n_rows) * 32, 256), 256, 0, st>>>(
      indptr, values, n_rows, values_out);
  TVBF_LAUNCH_OK("csr_normalize_kernel");
  return TVBF_OK;
}

int tvbf_prep_csr_to_operand(const int64_t* indptr, const int32_t* indices, const double* values,
                             int32_t n_rows, void* operand, int32_t k_pad, int32_t col_offset,
                             double scale, int32_t dtype, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(indptr && operand && n_rows >= 0 && k_pad > 0 && col_offset >= 0,
               "tvbf_prep_csr_to_operand: bad arguments");
  TVBF_REQUIRE(dtype == TVBF_TEXT_FP16 || dtype == TVBF_TEXT_BF16,
               "tvbf_prep_csr_to_operand: dtype must be TVBF_TEXT_FP16 or TVBF_TEXT_BF16");
  if (n_rows == 0) return TVBF_OK;
  auto st = static_cast<cudaStream_t>(stream);
  unsigned grid = blocks_for(static_cast<size_t>(n_rows) * 32, 256);
  if (dtype == TVBF_TEXT_FP16)
    csr_to_operand_kernel<__half><<<grid, 256, 0, st>>>(indptr, indices, values, n_rows,
                                                        static_cast<__half*>(operand), k_pad,
                                                        col_offset, scale);
  else
    csr_to_operand_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(
        indptr, indices, values, n_rows, static_cast<__nv_bfloat16*>(operand), k_pad, col_offset,
        scale);
  TVBF_LAUNCH_OK("csr_to_operand_kernel");
  return TVBF_OK;
}

namespace {
struct MergeWs {
  size_t df, keys, iota, order, cub, cub_bytes, total;
};
MergeWs merge_ws(int vocab) {
  MergeWs w;
  const size_t v = static_cast<size_t>(vocab) * 4, a = (v + 255) / 256 * 256;
  w.df = 0;
  w.keys = a;
  w.iota = 2 * a;
  w.order = 3 * a;
  w.cub = 4 * a;
  w.cub_bytes = 0;
  cub::DeviceRadixSort::SortPairsDescending(nullptr, w.cub_bytes, static_cast<const int32_t*>(nullptr),
                                            static_cast<int32_t*>(nullptr), static_cast<const int32_t*>(nullptr),
                                            static_cast<int32_t*>(nullptr), vocab);
  w.total = w.cub + w.cub_bytes;
  return w;
}
}  // namespace

size_t tvbf_merge_plan_workspace_bytes(int32_t vocab) { return vocab > 0 ? merge_ws(vocab).total : 0; }

int tvbf_merge_plan(const int64_t* indptr, const int32_t* indices, int32_t n_rows, int32_t vocab,
                    int32_t text_cols, int32_t* col_map, int32_t* slot_ptr, int32_t* slot_cols,
                    void* workspace, size_t workspace_bytes, void* stream) {
  TVBF_REQUIRE(indptr && indices && col_map && slot_ptr && slot_cols && workspace && n_rows >= 0 && vocab > 0,
               "tvbf_merge_plan: bad arguments");
  TVBF_REQUIRE(text_cols >= 2 && text_cols <= vocab, "tvbf_merge_plan: text_cols %d outside [2, %d]", text_cols, vocab);
  {
    const int head = text_cols / 2, tail = text_cols - head;
    const int most = (vocab - head + tail - 1) / tail;
    TVBF_REQUIRE(most <= 4096, "tvbf_merge_plan: %d vocabulary columns per operand column (at most 4096)", most);
  }
  TVBF_ENTER_CALL(stream);   // after the argument checks, which touch no device
  const MergeWs w = merge_ws(vocab);
  TVBF_REQUIRE(workspace_bytes >= w.total, "tvbf_merge_plan: workspace of %zu bytes, needs %zu", workspace_bytes,
               w.total);
  auto st = static_cast<cudaStream_t>(stream);
  auto* ws = static_cast<uint8_t*>(workspace);
  auto* df = reinterpret_cast<int32_t*>(ws + w.df);
  auto* keys = reinterpret_cast<int32_t*>(ws + w.keys);
  auto* iota = reinterpret_cast<int32_t*>(ws + w.iota);
  auto* order = reinterpret_cast<int32_t*>(ws + w.order);
  TVBF_CUDA_OK(cudaMemsetAsync(df, 0, static_cast<size_t>(vocab) * 4, st));
  column_df_kernel<<<296, 512, 0, st>>>(indptr, indices, n_rows, vocab, df);
  TVBF_LAUNCH_OK("column_df_kernel");
  iota_kernel<<<blocks_for(vocab, 256), 256, 0, st>>>(iota, vocab);
  TVBF_LAUNCH_OK("iota_kernel");
  // stable: equal frequencies keep the ascending column order of iota
  size_t cub_bytes = w.cub_bytes;
  TVBF_CUDA_OK(cub::DeviceRadixSort::SortPairsDescending(ws + w.cub, cub_bytes, df, keys, iota, order, vocab, 0, 32,
                                                         st));
  tvbf_count_launch();   // the sort's kernels count as one launch
  merge_plan_fill_kernel<<<blocks_for(static_cast<size_t>(vocab) + 1, 256), 256, 0, st>>>(
      order, vocab, text_cols, col_map, slot_ptr, slot_cols);
  TVBF_LAUNCH_OK("merge_plan_fill_kernel");
  return TVBF_OK;
}

int tvbf_prep_csr_to_operand_mapped(const int64_t* indptr, const int32_t* indices, const double* values,
                                    int32_t n_rows, const int32_t* col_map, const int32_t* slot_ptr,
                                    const int32_t* slot_cols, void* operand, int32_t k_pad, int32_t col_offset,
                                    double scale, int32_t dtype, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(indptr && operand && col_map && slot_ptr && slot_cols && n_rows >= 0 && k_pad > 0 && col_offset >= 0,
               "tvbf_prep_csr_to_operand_mapped: bad arguments");
  TVBF_REQUIRE(dtype == TVBF_TEXT_FP16 || dtype == TVBF_TEXT_BF16,
               "tvbf_prep_csr_to_operand_mapped: dtype must be TVBF_TEXT_FP16 or TVBF_TEXT_BF16");
  if (n_rows == 0) return TVBF_OK;
  auto st = static_cast<cudaStream_t>(stream);
  unsigned grid = blocks_for(static_cast<size_t>(n_rows) * 32, 256);
  if (dtype == TVBF_TEXT_FP16)
    csr_to_operand_mapped_kernel<__half><<<grid, 256, 0, st>>>(indptr, indices, values, n_rows, col_map, slot_ptr,
                                                               slot_cols, static_cast<__half*>(operand), k_pad,
                                                               col_offset, scale);
  else
    csr_to_operand_mapped_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(
        indptr, indices, values, n_rows, col_map, slot_ptr, slot_cols, static_cast<__nv_bfloat16*>(operand), k_pad,
        col_offset, scale);
  TVBF_LAUNCH_OK("csr_to_operand_mapped_kernel");
  return TVBF_OK;
}

int tvbf_prep_clear_csr_positions(const int64_t* indptr, const int32_t* indices, int32_t n_rows,
                                  void* operand, int32_t k_pad, int32_t col_offset, int32_t dtype,
                                  void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(indptr && operand && n_rows >= 0 && k_pad > 0 && col_offset >= 0,
               "tvbf_prep_clear_csr_positions: bad arguments");
  TVBF_REQUIRE(dtype == TVBF_TEXT_FP16 || dtype == TVBF_TEXT_BF16,
               "tvbf_prep_clear_csr_positions: dtype must be TVBF_TEXT_FP16 or TVBF_TEXT_BF16");
  if (n_rows == 0) return TVBF_OK;
  auto st = static_cast<cudaStream_t>(stream);
  unsigned grid = blocks_for(static_cast<size_t>(n_rows) * 32, 256);
  if (dtype == TVBF_TEXT_FP16)
    csr_clear_operand_kernel<__half><<<grid, 256, 0, st>>>(indptr, indices, n_rows, static_cast<__half*>(operand),
                                                           k_pad, col_offset);
  else
    csr_clear_operand_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(
        indptr, indices, n_rows, static_cast<__nv_bfloat16*>(operand), k_pad, col_offset);
  TVBF_LAUNCH_OK("csr_clear_operand_kernel");
  return TVBF_OK;
}

int tvbf_peer_push(const uint64_t* peer_base, int32_t world, int32_t rank, const uint64_t* offsets,
                   const uint64_t* bytes, int32_t n_fields, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(peer_base && offsets && bytes && world >= 1 && world <= 16 && rank >= 0 && rank < world &&
                   n_fields >= 1 && n_fields <= 8,
               "tvbf_peer_push: bad arguments");
  if (world == 1) return TVBF_OK;
  PeerPush a;
  size_t most = 0;
  for (int p = 0; p < world; ++p) {
    TVBF_REQUIRE(peer_base[p] != 0 && (peer_base[p] & 15) == 0, "tvbf_peer_push: peer %d has no 16-byte aligned mapping", p);
    a.base[p] = peer_base[p];
  }
  for (int f = 0; f < n_fields; ++f) {
    TVBF_REQUIRE((offsets[f] & 3) == 0 && (bytes[f] & 3) == 0, "tvbf_peer_push: field %d is not 4-byte aligned", f);
    a.off[f] = offsets[f];
    a.bytes[f] = bytes[f];
    most = bytes[f] > most ? bytes[f] : most;
  }
  a.world = world;
  a.rank = rank;
  a.n_fields = n_fields;
  if (most == 0) return TVBF_OK;
  // enough blocks per peer to keep the NVLink stores of all peers in flight (16 B per thread and step)
  unsigned bx = static_cast<unsigned>((most / 16 + 255) / 256);
  bx = bx < 1 ? 1 : (bx > 64 ? 64 : bx);
  peer_push_kernel<<<dim3(bx, static_cast<unsigned>(world - 1)), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  TVBF_LAUNCH_OK("peer_push_kernel");
  return TVBF_OK;
}

int tvbf_device_zero(void* ptr, size_t bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(ptr != nullptr || bytes == 0, "tvbf_device_zero: NULL pointer");
  if (bytes == 0) return TVBF_OK;
  TVBF_CUDA_OK(cudaMemsetAsync(ptr, 0, bytes, static_cast<cudaStream_t>(stream)));
  return TVBF_OK;
}

int tvbf_prep_dense_normalize(const double* in, int32_t n_rows, int32_t dim, double* out,
                              void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(in && out && n_rows >= 0 && dim > 0, "tvbf_prep_dense_normalize: bad arguments");
  if (n_rows == 0) return TVBF_OK;
  dense_normalize_kernel<<<blocks_for(n_rows, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      in, n_rows, dim, out);
  TVBF_LAUNCH_OK("dense_normalize_kernel");
  return TVBF_OK;
}

int tvbf_prep_dense_to_operand(const double* dense, int32_t n_rows, int32_t dim, void* operand,
                               int32_t k_pad, int32_t col_offset, double scale, int32_t dtype,
                               void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(dense && operand && n_rows >= 0 && dim > 0 && col_offset >= 0 &&
                   col_offset + dim <= k_pad,
               "tvbf_prep_dense_to_operand: bad arguments");
  TVBF_REQUIRE(dtype == TVBF_TEXT_FP16 || dtype == TVBF_TEXT_BF16,
               "tvbf_prep_dense_to_operand: dtype must be TVBF_TEXT_FP16 or TVBF_TEXT_BF16");
  if (n_rows == 0) return TVBF_OK;
  auto st = static_cast<cudaStream_t>(stream);
  unsigned grid = blocks_for(static_cast<size_t>(n_rows) * dim, 256);
  if (dtype == TVBF_TEXT_FP16)
    dense_to_operand_kernel<__half><<<grid, 256, 0, st>>>(
        dense, n_rows, dim, static_cast<__half*>(operand), k_pad, col_offset, scale);
  else
    dense_to_operand_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(
        dense, n_rows, dim, static_cast<__nv_bfloat16*>(operand), k_pad, col_offset, scale);
  TVBF_LAUNCH_OK("dense_to_operand_kernel");
  return TVBF_OK;
}

int tvbf_prep_fold_bits(const void* col_side, const uint64_t* genre_hi, const float* meta_scale,
                        int32_t n_rows, int32_t genre_dim, void* operand, int32_t k_pad, int32_t col0,
                        double scale_genre, double scale_meta, int32_t dtype, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(col_side && meta_scale && operand && n_rows >= 0 && genre_dim >= 1 && genre_dim <= 128 &&
                   col0 >= 0 && col0 + genre_dim + 32 <= k_pad,
               "tvbf_prep_fold_bits: bad arguments");
  TVBF_REQUIRE(genre_dim <= 64 || genre_hi != nullptr, "tvbf_prep_fold_bits: %d genre columns need genre_hi", genre_dim);
  TVBF_REQUIRE(dtype == TVBF_TEXT_FP16 || dtype == TVBF_TEXT_BF16,
               "tvbf_prep_fold_bits: dtype must be TVBF_TEXT_FP16 or TVBF_TEXT_BF16");
  if (n_rows == 0) return TVBF_OK;
  auto st = static_cast<cudaStream_t>(stream);
  const unsigned grid = blocks_for(static_cast<size_t>(n_rows) * (genre_dim + 32), 256);
  const auto* cs = static_cast<const TvbfColSide*>(col_side);
  const auto* gh = reinterpret_cast<const unsigned long long*>(genre_hi);
  if (dtype == TVBF_TEXT_FP16)
    fold_bits_kernel<__half><<<grid, 256, 0, st>>>(cs, gh, meta_scale, n_rows, genre_dim, static_cast<__half*>(operand),
                                                    k_pad, col0, scale_genre, scale_meta);
  else
    fold_bits_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(cs, gh, meta_scale, n_rows, genre_dim,
                                                           static_cast<__nv_bfloat16*>(operand), k_pad, col0,
                                                           scale_genre, scale_meta);
  TVBF_LAUNCH_OK("fold_bits_kernel");
  return TVBF_OK;
}

int tvbf_prep_genre_bits(const uint8_t* genre, int32_t n_rows, int32_t dim, void* col_side,
                         uint64_t* genre_hi, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(genre && col_side && n_rows >= 0, "tvbf_prep_genre_bits: bad arguments");
  TVBF_REQUIRE(dim >= 1 && dim <= 128, "tvbf_prep_genre_bits: dim %d outside 1..128", dim);
  TVBF_REQUIRE(dim <= 64 || genre_hi != nullptr, "tvbf_prep_genre_bits: dim %d needs genre_hi", dim);
  if (n_rows == 0) return TVBF_OK;
  genre_bits_kernel<<<blocks_for(n_rows, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      genre, n_rows, dim, static_cast<TvbfColSide*>(col_side), reinterpret_cast<unsigned long long*>(genre_hi));
  TVBF_LAUNCH_OK("genre_bits_kernel");
  return TVBF_OK;
}

int tvbf_prep_meta_ids(const uint8_t* platform, int32_t p_dim, const uint8_t* type, int32_t t_dim,
                       const uint8_t* language, int32_t l_dim, int32_t n_rows, int32_t n_pad,
                       int32_t meta_kind, void* col_side, float* meta_scale, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(col_side && meta_scale && n_rows >= 0 && n_pad >= n_rows,
               "tvbf_prep_meta_ids: bad arguments");
  TVBF_REQUIRE(p_dim >= 0 && t_dim >= 0 && l_dim >= 0 && p_dim + t_dim + l_dim <= 32,
               "tvbf_prep_meta_ids: the three one-hot groups must fit 32 bits together");
  TVBF_REQUIRE(meta_kind == TVBF_META_MEAN3 || meta_kind == TVBF_META_HSTACK,
               "tvbf_prep_meta_ids: bad meta_kind");
  if (n_pad == 0) return TVBF_OK;
  meta_bits_kernel<<<blocks_for(n_pad, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      platform, p_dim, type, t_dim, language, l_dim, n_rows, n_pad, meta_kind,
      static_cast<TvbfColSide*>(col_side), meta_scale);
  TVBF_LAUNCH_OK("meta_bits_kernel");
  return TVBF_OK;
}

int tvbf_ingest_genre(const void* raw, int32_t dtype, int32_t n_rows, int32_t n_pad, int32_t dim, void* col_side,
                      uint64_t* genre_hi, int32_t* flags, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(raw && col_side && flags && n_rows >= 0 && n_pad >= n_rows, "tvbf_ingest_genre: bad arguments");
  TVBF_REQUIRE(dim >= 1 && dim <= 128, "tvbf_ingest_genre: dim %d outside 1..128", dim);
  TVBF_REQUIRE(dim <= 64 || genre_hi != nullptr, "tvbf_ingest_genre: dim %d needs genre_hi", dim);
  TVBF_REQUIRE(dtype >= 0 && dtype <= 4, "tvbf_ingest_genre: bad dtype code %d", dtype);
  if (n_pad == 0) return TVBF_OK;
  ingest_genre_kernel<<<blocks_for(n_pad, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      raw, dtype, n_rows, n_pad, dim, static_cast<TvbfColSide*>(col_side),
      reinterpret_cast<unsigned long long*>(genre_hi), flags);
  TVBF_LAUNCH_OK("ingest_genre_kernel");
  return TVBF_OK;
}

int tvbf_ingest_meta(const void* platform, int32_t p_dtype, int32_t p_dim, const void* type, int32_t t_dtype,
                     int32_t t_dim, const void* language, int32_t l_dtype, int32_t l_dim, int32_t n_rows,
                     int32_t n_pad, int32_t meta_kind, void* col_side, float* meta_scale, int32_t* flags,
                     void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(platform && type && language && col_side && meta_scale && flags && n_rows >= 0 && n_pad >= n_rows,
               "tvbf_ingest_meta: bad arguments");
  TVBF_REQUIRE(p_dim >= 0 && t_dim >= 0 && l_dim >= 0 && p_dim + t_dim + l_dim <= 32,
               "tvbf_ingest_meta: the three one-hot groups must fit 32 bits together");
  TVBF_REQUIRE(meta_kind == TVBF_META_MEAN3 || meta_kind == TVBF_META_HSTACK, "tvbf_ingest_meta: bad meta_kind");
  if (n_pad == 0) return TVBF_OK;
  ingest_meta_kernel<<<blocks_for(n_pad, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      platform, p_dtype, p_dim, type, t_dtype, t_dim, language, l_dtype, l_dim, n_rows, n_pad, meta_kind,
      static_cast<TvbfColSide*>(col_side), meta_scale, flags);
  TVBF_LAUNCH_OK("ingest_meta_kernel");
  return TVBF_OK;
}

int tvbf_ingest_csr(const void* indptr_raw, int32_t indptr64, const void* indices_raw, int32_t indices64,
                    const void* values_raw, int32_t values64, int32_t n_rows, int64_t* indptr, int32_t* indices,
                    double* values, int32_t* flags, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(indptr_raw && indptr && flags && n_rows >= 0, "tvbf_ingest_csr: bad arguments");
  ingest_csr_kernel<<<blocks_for((static_cast<size_t>(n_rows) + 1) * 32, 256), 256, 0,
                      static_cast<cudaStream_t>(stream)>>>(indptr_raw, indptr64, indices_raw, indices64, values_raw,
                                                           values64, n_rows, indptr, indices, values, flags);
  TVBF_LAUNCH_OK("ingest_csr_kernel");
  return TVBF_OK;
}

int tvbf_csr_to_dense_f64(const int64_t* indptr, const int32_t* indices, const double* values,
                          int32_t n_rows, int32_t dim, double* dense, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(indptr && dense && n_rows >= 0 && dim > 0, "tvbf_csr_to_dense_f64: bad arguments");
  if (n_rows == 0) return TVBF_OK;
  csr_to_dense_kernel<<<blocks_for(static_cast<size_t>(n_rows) * 32, 256), 256, 0,
                        static_cast<cudaStream_t>(stream)>>>(indptr, indices, values, n_rows, dim,
                                                             dense);
  TVBF_LAUNCH_OK("csr_to_dense_kernel");
  return TVBF_OK;
}

}  // extern "C"
