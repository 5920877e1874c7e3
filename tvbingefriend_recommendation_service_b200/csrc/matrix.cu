// Full-matrix variant of the path: what ml/similarity_computer.py materialises (four N x N
// float64 matrices and their upper-triangle statistics).  Only sensible for small catalogues
// (32 * N^2 bytes); the production path is hybrid_topk.cu.  All fp64, deterministic order.
#include "common.cuh"

namespace {

// C[i, j] = sum_c X[i, c] * X[j, c]   (cosine_similarity(X) once rows are normalised;
// similarity_computer.py:41,58,86).  64 x 64 tile per CTA, 4 x 4 outputs per thread.
constexpr int TS = 64, TK = 16;

__global__ void __launch_bounds__(256)
cosine_matrix_kernel(const double* __restrict__ x, int n, int dim, double* __restrict__ out) {
  __shared__ double As[TK][TS + 1];
  __shared__ double Bs[TK][TS + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int row0 = blockIdx.y * TS, col0 = blockIdx.x * TS;
  double acc[4][4] = {};
  for (int k0 = 0; k0 < dim; k0 += TK) {
    for (int e = threadIdx.x; e < TS * TK; e += 256) {
      const int r = e / TK, c = e % TK;
      const int gr = row0 + r, gc = col0 + r, gk = k0 + c;
      As[c][r] = (gr < n && gk < dim) ? x[static_cast<size_t>(gr) * dim + gk] : 0.0;
      Bs[c][r] = (gc < n && gk < dim) ? x[static_cast<size_t>(gc) * dim + gk] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < TK; ++c) {
      double a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        a[u] = As[c][ty * 4 + u];
        b[u] = Bs[c][tx * 4 + u];
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] += a[u] * b[v];
    }
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int r = row0 + ty * 4 + u, c = col0 + tx * 4 + v;
      if (r < n && c < n) out[static_cast<size_t>(r) * n + c] = acc[u][v];
    }
}

__global__ void hybrid_combine_kernel(const double* __restrict__ g, const double* __restrict__ t,
                                      const double* __restrict__ m, double wg, double wt,
                                      double wm, long long count, double* __restrict__ out) {
  long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (; i < count; i += stride) out[i] = tvbf::hybrid_rn(wg, g[i], wt, t[i], wm, m[i]);
}

// ---- upper-triangle statistics (similarity_computer.py:171-190) --------------------------------
struct StatsState {
  double sum, min, max, mean, m2;
  unsigned long long prefix;  // radix-select state
  long long rank;
  double median_lo, median_hi;
  unsigned long long hist[256];
};

__device__ __forceinline__ unsigned long long ord64(double d) {
  unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(d));
  return b ^ ((b >> 63) ? 0xFFFFFFFFFFFFFFFFull : 0x8000000000000000ull);
}
__device__ __forceinline__ double unord64(unsigned long long u) {
  unsigned long long b = u ^ ((u >> 63) ? 0x8000000000000000ull : 0xFFFFFFFFFFFFFFFFull);
  return __longlong_as_double(static_cast<long long>(b));
}

constexpr int ST_BLOCKS = 592, ST_THREADS = 256;

__device__ __forceinline__ double block_sum(double v, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < ST_THREADS / 32; ++w) t += sh[w];
  __syncthreads();
  return t;  // valid in thread 0
}

// pass 0: per-block sum/min/max; pass 1: per-block sum of squared deviations
__global__ void __launch_bounds__(ST_THREADS)
stats_reduce_kernel(const double* __restrict__ mat, int n, int pass, const StatsState* state,
                    double* __restrict__ partial) {
  __shared__ double sh[ST_THREADS / 32];
  const double mean = pass ? state->mean : 0.0;
  double s = 0.0, mn = INFINITY, mx = -INFINITY;
  for (int r = blockIdx.x; r < n; r += gridDim.x) {
    const double* row = mat + static_cast<size_t>(r) * n;
    for (int c = r + 1 + threadIdx.x; c < n; c += ST_THREADS) {
      const double v = row[c];
      if (pass) {
        const double d = v - mean;
        s += d * d;
      } else {
        s += v;
        mn = fmin(mn, v);
        mx = fmax(mx, v);
      }
    }
  }
  const double tot = block_sum(s, sh);
  if (threadIdx.x == 0) partial[blockIdx.x * 3 + 0] = tot;
  if (!pass) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __shared__ double shmn[ST_THREADS / 32], shmx[ST_THREADS / 32];
    if ((threadIdx.x & 31) == 0) { shmn[threadIdx.x >> 5] = mn; shmx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < ST_THREADS / 32; ++w) { mn = fmin(mn, shmn[w]); mx = fmax(mx, shmx[w]); }
      partial[blockIdx.x * 3 + 1] = fmin(mn, shmn[0]);
      partial[blockIdx.x * 3 + 2] = fmax(mx, shmx[0]);
    }
  }
}

__global__ void stats_finish_kernel(const double* partial, int blocks, int pass, long long count,
                                    StatsState* state) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double s = 0.0, mn = INFINITY, mx = -INFINITY;
  for (int b = 0; b < blocks; ++b) {
    s += partial[b * 3];
    if (!pass) { mn = fmin(mn, partial[b * 3 + 1]); mx = fmax(mx, partial[b * 3 + 2]); }
  }
  if (!pass) {
    state->sum = s; state->min = mn; state->max = mx;
    state->mean = s / static_cast<double>(count);
  } else {
    state->m2 = s;
  }
}

__global__ void __launch_bounds__(ST_THREADS)
stats_hist_kernel(const double* __restrict__ mat, int n, int shift, StatsState* state) {
  __shared__ unsigned int h[256];
  for (int b = threadIdx.x; b < 256; b += ST_THREADS) h[b] = 0u;
  __syncthreads();
  const unsigned long long prefix = state->prefix;
  const unsigned long long hi_mask = shift == 56 ? 0ull : (~0ull << (shift + 8));
  for (int r = blockIdx.x; r < n; r += gridDim.x) {
    const double* row = mat + static_cast<size_t>(r) * n;
    for (int c = r + 1 + threadIdx.x; c < n; c += ST_THREADS) {
      const unsigned long long key = ord64(row[c]);
      if ((key & hi_mask) == prefix) atomicAdd(&h[(key >> shift) & 0xFFu], 1u);
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < 256; b += ST_THREADS)
    if (h[b]) atomicAdd(&state->hist[b], static_cast<unsigned long long>(h[b]));
}

// rank = 0-based ascending rank still to find among keys matching the prefix
__global__ void stats_pick_kernel(int shift, int which, StatsState* state) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  long long rank = state->rank;
  int d = 0;
  for (; d < 255; ++d) {
    const long long c = static_cast<long long>(state->hist[d]);
    if (rank < c) break;
    rank -= c;
  }
  state->prefix |= static_cast<unsigned long long>(d) << shift;
  state->rank = rank;
  for (int b = 0; b < 256; ++b) state->hist[b] = 0ull;
  if (shift == 0) {
    const double v = unord64(state->prefix);
    if (which == 0) state->median_lo = v; else state->median_hi = v;
  }
}

__global__ void stats_begin_select_kernel(long long rank, StatsState* state) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  state->prefix = 0ull;
  state->rank = rank;
  for (int b = 0; b < 256; ++b) state->hist[b] = 0ull;
}

}  // namespace

extern "C" {

int tvbf_cosine_matrix_f64(const double* x, int32_t n_rows, int32_t dim, double* out,
                           void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(x && out && n_rows >= 0 && dim > 0, "tvbf_cosine_matrix_f64: bad arguments");
  if (n_rows == 0) return TVBF_OK;
  dim3 grid((n_rows + TS - 1) / TS, (n_rows + TS - 1) / TS);
  cosine_matrix_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, n_rows, dim, out);
  TVBF_LAUNCH_OK("cosine_matrix_kernel");
  return TVBF_OK;
}

int tvbf_hybrid_combine_f64(const double* g, const double* t, const double* m, double wg,
                            double wt, double wm, int64_t count, double* out, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(g && t && m && out && count >= 0, "tvbf_hybrid_combine_f64: bad arguments");
  if (count == 0) return TVBF_OK;
  long long blocks = (count + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  hybrid_combine_kernel<<<static_cast<unsigned>(blocks), 256, 0,
                          static_cast<cudaStream_t>(stream)>>>(g, t, m, wg, wt, wm, count, out);
  TVBF_LAUNCH_OK("hybrid_combine_kernel");
  return TVBF_OK;
}

size_t tvbf_matrix_stats_workspace_bytes(void) {
  return sizeof(StatsState) + ST_BLOCKS * 3 * sizeof(double) + 256;
}

int tvbf_matrix_stats_f64(const double* mat, int32_t n, double* out5_host, void* workspace,
                          size_t workspace_bytes, void* stream) {
  TVBF_ENTER_CALL(stream);
  TVBF_REQUIRE(mat && out5_host && workspace, "tvbf_matrix_stats_f64: bad arguments");
  TVBF_REQUIRE(n >= 2, "tvbf_matrix_stats_f64: need at least 2 rows (empty upper triangle)");
  if (workspace_bytes < tvbf_matrix_stats_workspace_bytes()) {
    tvbf_set_error("tvbf_matrix_stats_f64: workspace too small");
    return TVBF_ERR_WORKSPACE;
  }
  auto st = static_cast<cudaStream_t>(stream);
  StatsState* state = static_cast<StatsState*>(workspace);
  double* partial = reinterpret_cast<double*>(static_cast<uint8_t*>(workspace) +
                                              ((sizeof(StatsState) + 255) / 256) * 256);
  const long long count = static_cast<long long>(n) * (n - 1) / 2;
  const int blocks = n < ST_BLOCKS ? n : ST_BLOCKS;
  TVBF_CUDA_OK(cudaMemsetAsync(state, 0, sizeof(StatsState), st));
  for (int pass = 0; pass < 2; ++pass) {
    stats_reduce_kernel<<<blocks, ST_THREADS, 0, st>>>(mat, n, pass, state, partial);
    TVBF_LAUNCH_OK("stats_reduce_kernel");
    stats_finish_kernel<<<1, 32, 0, st>>>(partial, blocks, pass, count, state);
    TVBF_LAUNCH_OK("stats_finish_kernel");
  }
  // numpy.median: middle element, or the mean of the two middle elements for an even count
  const long long ranks[2] = {(count - 1) / 2, count / 2};
  for (int which = 0; which < 2; ++which) {
    stats_begin_select_kernel<<<1, 32, 0, st>>>(ranks[which], state);
    for (int shift = 56; shift >= 0; shift -= 8) {
      stats_hist_kernel<<<blocks, ST_THREADS, 0, st>>>(mat, n, shift, state);
      stats_pick_kernel<<<1, 32, 0, st>>>(shift, which, state);
    }
    TVBF_LAUNCH_OK("stats select");
  }
  StatsState host;
  TVBF_CUDA_OK(cudaMemcpyAsync(&host, state, sizeof(StatsState), cudaMemcpyDeviceToHost, st));
  TVBF_CUDA_OK(cudaStreamSynchronize(st));
  out5_host[0] = host.mean;
  out5_host[1] = sqrt(host.m2 / static_cast<double>(count));
  out5_host[2] = host.min;
  out5_host[3] = host.max;
  out5_host[4] = (host.median_lo + host.median_hi) / 2.0;
  return TVBF_OK;
}

}  // extern "C"
