// Relaxation-time distribution and total chargeability over a decomposition chain: bisip_rtd_stats.
//
// Replaces the host path of PolynomialDecomposition.get_rtd(p=...) (products.relaxation_time_distribution of every
// flat-chain sample, then np.percentile; reference docs/tutorials/decomposition.ipynb cells 25-29) and gives batch fits
// the same products.  Column l < n_tau of a spectrum is m_l = sum_i a_i log_taus[i][l] of every sample, column n_tau its
// total chargeability.  As in model_percentile_kernel, one CTA owns one (column, spectrum) pair, evaluates its column for
// all samples straight into shared memory and selects there (stats.cuh), so the (n, n_tau) RTD matrix is never written.
//   * m_l is accumulated in ascending i from 0.0 with unfused multiply and add, the arithmetic of
//     relaxation_time_distribution: every value, and so every percentile, equals NumPy's bit for bit.
//   * The total column is sum_i a_i S_i with S_i = sum_l log_taus[i][l] (ascending l, once per CTA): n_coef operations
//     per sample instead of n_coef * n_tau.  It differs from the sum of the m_l by rounding only.
//   * A column longer than one CTA's shared memory runs the same statistics from global memory (global_column_stats),
//     recomputing the value of sample i wherever the radix select asks for it: no workspace, no length limit.
#pragma once
#include "common.cuh"
#include "model_pct.cuh"
#include "stats.cuh"

namespace bisip {

struct RtdParams {
  const double* theta;              // [B][n][ndim], ndim = 1 + n_coef (r0, a_0 .. a_{n_coef-1})
  const double* log_taus;           // [n_coef][n_tau], or per spectrum at b * tau_stride * n_coef
  long long tau_stride;
  int ndim, n_coef, n_tau;
  StatsParams st;                   // n, npct, lo, gamma; pct_out [B][npct][n_tau+1], mean_out / std_out [B][n_tau+1]
};

// Weights that turn a sample's a_0 .. a_{n_coef-1} into the value of column `col`: log_taus[:, col], or the row sums of
// log_taus for the total chargeability (col == n_tau).  Threads < n_coef write s_w; the caller synchronises.
__device__ __forceinline__ void rtd_stage_weights(const RtdParams& P, int col, int b, double* s_w) {
  const int i = threadIdx.x;
  if (i >= P.n_coef) return;
  const double* row = P.log_taus + (size_t)b * P.tau_stride * P.n_coef + (size_t)i * P.n_tau;
  double v;
  if (col < P.n_tau) {
    v = row[col];
  } else {
    v = 0.0;
    for (int l = 0; l < P.n_tau; ++l) v = __dadd_rn(v, row[l]);
  }
  s_w[i] = v;
}

__device__ __forceinline__ double rtd_value(const double* __restrict__ a, const double* s_w, int n_coef) {
  double m = 0.0;
  for (int i = 0; i < n_coef; ++i) m = __dadd_rn(m, __dmul_rn(__ldg(a + i), s_w[i]));
  return m;
}

// grid (n_tau+1, B), kStatThreads threads, dynamic shared memory stats_smem_bytes(n, 2 npct)
__global__ void __launch_bounds__(kStatThreads, 1) rtd_stats_smem_kernel(const RtdParams P) {
  extern __shared__ __align__(16) unsigned char stats_dyn[];
  __shared__ double red[32];
  __shared__ double s_w[kMaxCoefPct];
  constexpr int NT = kStatThreads;
  const int col = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int n = (int)P.st.n, D = P.n_coef, ndim = P.ndim;
  double* vals = reinterpret_cast<double*>(stats_dyn);
  double* pool = vals + n;
  unsigned int* hist = reinterpret_cast<unsigned int*>(pool + kStatPool);
  rtd_stage_weights(P, col, b, s_w);
  __syncthreads();
  const double* a = P.theta + (size_t)b * P.st.n * ndim + 1;
  double s = 0.0, mn = __longlong_as_double(0x7ff0000000000000LL), mx = -mn;
  int nan = 0;
  for (int i = tid; i < n; i += NT) {
    const double v = rtd_value(a + (size_t)i * ndim, s_w, D);
    vals[i] = v;
    s += v;
    mn = fmin(mn, v);
    mx = fmax(mx, v);
    nan |= (v != v) ? 1 : 0;
  }
  const double sum = block_sum_nt<NT>(s, red);
  mn = block_minmax_nt<NT, false>(mn, red);
  mx = block_minmax_nt<NT, true>(mx, red);
  const bool has_nan = __syncthreads_or(nan) != 0;
  const int C = P.n_tau + 1;
  const size_t o = (size_t)b * C + col;
  // the two-pass mean / std of smem_column_stats, with the warp sums added by one warp's shuffle tree: block_sum_nt's
  // 32 loads per thread would spill at the 64 registers of a 1024-thread CTA here
  if (P.st.mean_out != nullptr || P.st.std_out != nullptr) {
    const double mean = sum / (double)n;
    double v = 0.0;
    for (int i = tid; i < n; i += NT) {
      const double d = vals[i] - mean;
      v = fma(d, d, v);
    }
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) v += __shfl_xor_sync(0xffffffffu, v, k);
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    if (tid < 32) {
      v = red[tid];
#pragma unroll
      for (int k = 16; k > 0; k >>= 1) v += __shfl_xor_sync(0xffffffffu, v, k);
      if (tid == 0) {
        if (P.st.mean_out) P.st.mean_out[o] = mean;
        if (P.st.std_out) P.st.std_out[o] = sqrt(v / (double)n);
      }
    }
  }
  smem_column_stats<NT>(vals, n, sum, mn, mx, has_nan, P.st,
                        P.st.pct_out ? P.st.pct_out + (size_t)b * P.st.npct * C + col : nullptr, C, nullptr, nullptr,
                        hist, pool, red);
}

// Columns past shared memory.  grid (n_tau+1, B), kThreads threads, no dynamic shared memory.
__global__ void __launch_bounds__(kThreads) rtd_stats_global_kernel(const RtdParams P) {
  __shared__ unsigned int hist[kMaxRanks * 256];
  __shared__ double red[32];
  __shared__ double s_w[kMaxCoefPct];
  const int col = blockIdx.x, b = blockIdx.y;
  const int D = P.n_coef;
  const size_t ndim = P.ndim;
  rtd_stage_weights(P, col, b, s_w);
  __syncthreads();
  const double* a = P.theta + (size_t)b * P.st.n * ndim + 1;
  auto load = [&](long long i) { return rtd_value(a + (size_t)i * ndim, s_w, D); };
  const int C = P.n_tau + 1;
  const size_t o = (size_t)b * C + col;
  global_column_stats<kThreads>(load, P.st.n, P.st, P.st.pct_out ? P.st.pct_out + (size_t)b * P.st.npct * C + col : nullptr,
                                C, P.st.mean_out ? P.st.mean_out + o : nullptr, P.st.std_out ? P.st.std_out + o : nullptr,
                                hist, red);
}

}  // namespace bisip
