// Exact float64 moments of the text similarity matrix (and of its products with the genre and
// metadata matrices) WITHOUT forming N x N -- the part of get_similarity_statistics
// (ml/similarity_computer.py:171-190) that the fp16 tensor-core sweep cannot deliver to 1e-6:
//
//   sum_ij t_ij        = || X^T 1 ||^2            column sums            [V]
//   sum_ij t_ij^2      = || X^T X ||_F^2          vocabulary Gram matrix [V, V]  (upper triangle kept)
//   sum_ij g_ij t_ij   = || Ghat^T X ||_F^2       Ghat = genre bits / sqrt(popcount)     [64, V]
//   sum_ij m_ij t_ij   = || Mhat^T X ||_F^2       Mhat = one-hot bits * per-show scale   [32, V]
//
//   sum_ij g_ij        = || Ghat^T 1 ||^2,   sum_ij g_ij^2 = || Ghat^T Ghat ||_F^2   [64, 64]
//   sum_ij m_ij        = || Mhat^T 1 ||^2,   sum_ij m_ij^2 = || Mhat^T Mhat ||_F^2   [32, 32]
//   sum_ij g_ij m_ij   = || Ghat^T Mhat ||_F^2                                       [64, 32]
//
// (t = X X^T, g = Ghat Ghat^T, m = Mhat Mhat^T, all symmetric; sums run over ALL (i, j), the caller
// subtracts the diagonal terms, also returned here, and halves.)  X is the normalised text CSR.
// All accumulation is float64 atomics: exact up to rounding, order-independent to ~1e-15 relative.
#include "internal.cuh"

namespace {

__global__ void __launch_bounds__(256)
moments_scatter_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                       const double* __restrict__ values, const TvbfColSide* __restrict__ cs,
                       const float* __restrict__ meta_scale, int meta_hstack, int n_rows, int vocab,
                       double* __restrict__ colsum, double* __restrict__ mg, double* __restrict__ mm,
                       double* __restrict__ out8) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t b = indptr[row], e = indptr[row + 1];
  const TvbfColSide c = cs[row];
  const int gn = __popcll(c.genre_bits), mn = __popc(c.meta_bits);
  const double ghat = gn ? 1.0 / sqrt(static_cast<double>(gn)) : 0.0;
  // MEAN3: m_ij = matches / 3 = sum_bits (1/sqrt3)(1/sqrt3); HSTACK: matches / sqrt(n_i n_j)
  const double mhat = meta_hstack ? (mn ? 1.0 / sqrt(static_cast<double>(mn)) : 0.0) : 0.57735026918962576451;
  (void)meta_scale;
  double tii = 0.0;
  for (int64_t i = b + lane; i < e; i += 32) {
    const double x = values[i];
    const int col = indices[i];
    tii += x * x;
    atomicAdd(colsum + col, x);
    unsigned long long gb = c.genre_bits;
    while (gb) {
      const int bit = __ffsll(static_cast<long long>(gb)) - 1;
      gb &= gb - 1;
      atomicAdd(mg + static_cast<size_t>(bit) * vocab + col, x * ghat);
    }
    unsigned int mb = c.meta_bits;
    while (mb) {
      const int bit = __ffs(mb) - 1;
      mb &= mb - 1;
      atomicAdd(mm + static_cast<size_t>(bit) * vocab + col, x * mhat);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) tii += __shfl_xor_sync(0xffffffffu, tii, o);
  if (lane == 0) {
    const double gii = gn ? 1.0 : 0.0;   // cosine of a non-empty row with itself
    const double mii = meta_hstack ? (mn ? 1.0 : 0.0) : static_cast<double>(mn) / 3.0;
    atomicAdd(out8 + 4, tii);
    atomicAdd(out8 + 5, tii * tii);
    atomicAdd(out8 + 6, gii * tii);
    atomicAdd(out8 + 7, mii * tii);
  }
}

// genre / metadata Gram matrices: accumulated per CTA in shared memory (the same 4096 + 1024 + 2048
// addresses are hit by every show), flushed once.  small = [gg 64x64][mm 32x32][gm 64x32][sg 64][sm 32]
constexpr int kSmallDoubles = 64 * 64 + 32 * 32 + 64 * 32 + 64 + 32;

__global__ void __launch_bounds__(256)
moments_bits_kernel(const TvbfColSide* __restrict__ cs, int meta_hstack, int n_rows,
                    double* __restrict__ small, double* __restrict__ out) {
  extern __shared__ double sh[];
  double* gg = sh;
  double* mmx = gg + 64 * 64;
  double* gm = mmx + 32 * 32;
  double* sg = gm + 64 * 32;
  double* sm = sg + 64;
  for (int i = threadIdx.x; i < kSmallDoubles; i += blockDim.x) sh[i] = 0.0;
  __syncthreads();
  double d_g = 0.0, d_m = 0.0, d_m2 = 0.0, d_gm = 0.0;
  for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < n_rows; row += gridDim.x * blockDim.x) {
    const TvbfColSide c = cs[row];
    const int gn = __popcll(c.genre_bits), mn = __popc(c.meta_bits);
    const double ghat = gn ? 1.0 / sqrt(static_cast<double>(gn)) : 0.0;
    const double mhat = meta_hstack ? (mn ? 1.0 / sqrt(static_cast<double>(mn)) : 0.0) : 0.57735026918962576451;
    const double g2 = ghat * ghat, m2 = mhat * mhat, gmh = ghat * mhat;
    for (unsigned long long a = c.genre_bits; a; a &= a - 1) {
      const int ba = __ffsll(static_cast<long long>(a)) - 1;
      atomicAdd(sg + ba, ghat);
      for (unsigned long long b = c.genre_bits; b; b &= b - 1)
        atomicAdd(gg + ba * 64 + (__ffsll(static_cast<long long>(b)) - 1), g2);
      for (unsigned int b = c.meta_bits; b; b &= b - 1) atomicAdd(gm + ba * 32 + (__ffs(b) - 1), gmh);
    }
    for (unsigned int a = c.meta_bits; a; a &= a - 1) {
      const int ba = __ffs(a) - 1;
      atomicAdd(sm + ba, mhat);
      for (unsigned int b = c.meta_bits; b; b &= b - 1) atomicAdd(mmx + ba * 32 + (__ffs(b) - 1), m2);
    }
    const double gii = gn ? 1.0 : 0.0;
    const double mii = static_cast<double>(mn) * m2;   // MEAN3: matches / 3, HSTACK: 1 for a non-empty row
    d_g += gii;
    d_m += mii;
    d_m2 += mii * mii;
    d_gm += gii * mii;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kSmallDoubles; i += blockDim.x)
    if (sh[i] != 0.0) atomicAdd(small + i, sh[i]);
  // diagonal terms: out[13..17] = sum_i g_ii, g_ii^2 (= g_ii), m_ii, m_ii^2, g_ii m_ii
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    d_g += __shfl_xor_sync(0xffffffffu, d_g, o);
    d_m += __shfl_xor_sync(0xffffffffu, d_m, o);
    d_m2 += __shfl_xor_sync(0xffffffffu, d_m2, o);
    d_gm += __shfl_xor_sync(0xffffffffu, d_gm, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(out + 13, d_g);
    atomicAdd(out + 14, d_g);
    atomicAdd(out + 15, d_m);
    atomicAdd(out + 16, d_m2);
    atomicAdd(out + 17, d_gm);
  }
}

// upper triangle of the vocabulary Gram matrix: G[c, d] += x_ic x_id for c <= d (indices are sorted
// within a row, so entry pairs (a <= b) give c <= d); one warp per row, lanes stride the pairs
__global__ void __launch_bounds__(256)
gram_scatter_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                    const double* __restrict__ values, int n_rows, int vocab, double* __restrict__ gram) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t b = indptr[row];
  const int len = static_cast<int>(indptr[row + 1] - b);
  for (int a = 0; a < len; ++a) {
    const double xa = values[b + a];
    double* grow = gram + static_cast<size_t>(indices[b + a]) * vocab;
    for (int q = a + lane; q < len; q += 32) atomicAdd(grow + indices[b + q], xa * values[b + q]);
  }
}

// out += sum of squares of `count` doubles; `gram` mode: the array is a [vocab, vocab] upper triangle,
// off-diagonal entries count twice
__global__ void __launch_bounds__(256)
sum_squares_kernel(const double* __restrict__ x, size_t count, int vocab, int gram, double* __restrict__ out) {
  double s = 0.0;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride) {
    const double v = x[i];
    double w = 1.0;
    if (gram) {
      const size_t r = i / vocab, c = i - r * vocab;
      w = c > r ? 2.0 : (c == r ? 1.0 : 0.0);
    }
    s += w * v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __shared__ double sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sh[w];
    atomicAdd(out, t);
  }
}

inline size_t align256(size_t v) { return (v + 255) / 256 * 256; }

}  // namespace

extern "C" {

size_t tvbf_text_moments_workspace_bytes(const tvbf_features* f, int32_t with_gram) {
  if (f == nullptr || f->vocab <= 0) return 0;
  const size_t v = static_cast<size_t>(f->vocab);
  size_t bytes = align256(v * 8) + align256(64 * v * 8) + align256(32 * v * 8) + align256(kSmallDoubles * 8);
  if (with_gram) bytes += align256(v * v * 8);
  return bytes;
}

int tvbf_text_moments(const tvbf_features* f, int32_t with_gram, double* out8, void* workspace,
                      size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  // out8 has TVBF_MOMENTS (24) entries: [0..7] the text moments, [8..12] sum g, g^2, m, m^2, g*m,
  // [13..17] their diagonal terms
  TVBF_REQUIRE(f && out8 && workspace, "tvbf_text_moments: NULL argument");
  TVBF_REQUIRE(f->genre_mode != TVBF_GROUP_FOLDED && f->meta_mode != TVBF_GROUP_FOLDED && f->genre_hi == nullptr,
               "tvbf_text_moments needs binary genre (at most 64 columns) / one-hot metadata features");
  const size_t need = tvbf_text_moments_workspace_bytes(f, with_gram);
  if (workspace_bytes < need) {
    tvbf_set_error("tvbf_text_moments: workspace too small: %zu < %zu", workspace_bytes, need);
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  const int n = f->n_shows, v = f->vocab;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  double* colsum = reinterpret_cast<double*>(ws);
  double* mg = reinterpret_cast<double*>(ws + align256(static_cast<size_t>(v) * 8));
  double* mm = reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(mg) + align256(static_cast<size_t>(64) * v * 8));
  double* small = reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(mm) + align256(static_cast<size_t>(32) * v * 8));
  double* gram = reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(small) + align256(kSmallDoubles * 8));
  TVBF_CUDA_OK(cudaMemsetAsync(workspace, 0, need, st));
  TVBF_CUDA_OK(cudaMemsetAsync(out8, 0, TVBF_MOMENTS * sizeof(double), st));
  {
    const size_t smem = kSmallDoubles * sizeof(double);
    TVBF_CUDA_OK(cudaFuncSetAttribute(moments_bits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(smem)));
    moments_bits_kernel<<<148, 256, smem, st>>>(static_cast<const TvbfColSide*>(f->col_side),
                                                f->meta_kind == TVBF_META_HSTACK ? 1 : 0, n, small, out8);
    TVBF_LAUNCH_OK("moments_bits_kernel");
    const double* gg = small;
    const double* mmx = gg + 64 * 64;
    const double* gm = mmx + 32 * 32;
    const double* sg = gm + 64 * 32;
    const double* smv = sg + 64;
    sum_squares_kernel<<<1, 256, 0, st>>>(sg, 64, 1, 0, out8 + 8);
    sum_squares_kernel<<<8, 256, 0, st>>>(gg, 64 * 64, 1, 0, out8 + 9);
    sum_squares_kernel<<<1, 256, 0, st>>>(smv, 32, 1, 0, out8 + 10);
    sum_squares_kernel<<<4, 256, 0, st>>>(mmx, 32 * 32, 1, 0, out8 + 11);
    sum_squares_kernel<<<8, 256, 0, st>>>(gm, 64 * 32, 1, 0, out8 + 12);
    TVBF_LAUNCH_OK("sum_squares_kernel");
  }
  const unsigned row_blocks = static_cast<unsigned>((static_cast<size_t>(n) * 32 + 255) / 256);
  moments_scatter_kernel<<<row_blocks, 256, 0, st>>>(f->text_indptr, f->text_indices, f->text_values,
                                                     static_cast<const TvbfColSide*>(f->col_side), f->meta_scale,
                                                     f->meta_kind == TVBF_META_HSTACK ? 1 : 0, n, v, colsum, mg, mm,
                                                     out8);
  TVBF_LAUNCH_OK("moments_scatter_kernel");
  sum_squares_kernel<<<148, 256, 0, st>>>(colsum, static_cast<size_t>(v), v, 0, out8 + 0);
  TVBF_LAUNCH_OK("sum_squares_kernel");
  sum_squares_kernel<<<148, 256, 0, st>>>(mg, static_cast<size_t>(64) * v, v, 0, out8 + 2);
  TVBF_LAUNCH_OK("sum_squares_kernel");
  sum_squares_kernel<<<148, 256, 0, st>>>(mm, static_cast<size_t>(32) * v, v, 0, out8 + 3);
  TVBF_LAUNCH_OK("sum_squares_kernel");
  if (with_gram) {
    gram_scatter_kernel<<<row_blocks, 256, 0, st>>>(f->text_indptr, f->text_indices, f->text_values, n, v, gram);
    TVBF_LAUNCH_OK("gram_scatter_kernel");
    sum_squares_kernel<<<148 * 8, 256, 0, st>>>(gram, static_cast<size_t>(v) * v, v, 1, out8 + 1);
    TVBF_LAUNCH_OK("sum_squares_kernel");
  }
  return TVBF_OK;
}

}  // extern "C"
