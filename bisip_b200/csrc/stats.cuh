// Column statistics of data[B][n][ncol]: exact order statistics (NumPy 'linear' percentile),
// mean and population std.  Replaces np.percentile / np.mean / np.std over the flat chain
// (reference utils.py:35, :53, :69, :85), and — through model_percentile_kernel — the per-sample forward loop +
// np.percentile of get_model_percentile (utils.py:17-35).
//
// The chain is read IN PLACE, once: one CTA per (column, spectrum) pulls its column (stride ncol doubles; the ncol
// CTAs of a spectrum run together, so DRAM sees every sector once and the rest are L2 hits) into shared memory —
// a kept chain of 100 steps x 256 walkers is 25,600 doubles = 200 KB, one CTA per SM — and everything else happens
// there: sum / min / max while loading, the two-pass variance, and the selection:
//   * the values are binned MONOTONICALLY into 2,048 equal-width bins of [min, max] (x -> (x - min) * scale is
//     non-decreasing in IEEE arithmetic, so every value of a lower bin is <= every value of a higher bin);
//   * an inclusive scan of the bin counts locates the bin of every requested rank and its rank inside that bin;
//   * the (few dozen) members of those bins are gathered into a small pool and the wanted member is found by
//     counting: x is the k-th smallest iff #(y < x) <= k < #(y <= x).
// That is three passes over shared memory instead of eight radix passes over a transposed copy in HBM, no workspace
// and no transpose kernel.  Exactness does not depend on the binning (only speed does): if the selected bins hold
// more than the pool (pathological spread, or most values equal), or the column does not fit in shared memory
// (n > ~27,000), the generic 8-pass MSB radix select below runs on the same accessor, from shared or global memory.
// The order statistics are exact, and NumPy's _lerp is applied with unfused operations: bit-identical to np.percentile.
#pragma once
#include "common.cuh"

namespace bisip {

constexpr int kMaxPct = 16;              // percentiles per call
constexpr int kMaxRanks = 2 * kMaxPct;   // each needs the order statistics lo and lo+1
constexpr int kStatThreads = 1024;       // CTA of the shared-memory kernels (one per SM: the column fills it)
constexpr int kStatBins = 2048;
constexpr int kStatPool = 1536;          // doubles

struct StatsParams {
  const double* data;
  long long n;
  int ncol, B, npct;
  long long lo[kMaxPct];
  double gamma[kMaxPct];
  double* pct_out;
  double* mean_out;
  double* std_out;
};

// dynamic shared memory of the shared-memory kernels for a column of n values and R = 2 * npct ranks: the column, then
// the scratch area [pool | bin table], which the radix fallback re-uses for its R x 256 histograms
__host__ __device__ inline size_t stats_scratch_bytes(int R) {
  const size_t binned = (size_t)kStatPool * 8 + (size_t)(kStatBins + 32) * 4;
  const size_t radix = (size_t)(R > 0 ? R : 1) * 256 * 4;
  return binned > radix ? binned : radix;
}
__host__ __device__ inline size_t stats_smem_bytes(long long n, int R) { return (size_t)n * 8 + stats_scratch_bytes(R); }
constexpr size_t kStatStaticSmem = 4096;   // upper bound of the kernels' static shared memory (checked by the dispatcher)

__device__ __forceinline__ unsigned long long f64_key(double v) {
  unsigned long long u = (unsigned long long)__double_as_longlong(v);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_f64(unsigned long long k) {
  unsigned long long u = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)u);
}

// fixed-order block reductions (deterministic): lanes by xor-shuffle, then the warps in index order
template <int NT>
__device__ __forceinline__ double block_sum_nt(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < NT / 32; ++i) t += red[i];
  return t;
}
template <int NT, bool MAX>
__device__ __forceinline__ double block_minmax_nt(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double u = __shfl_xor_sync(0xffffffffu, v, o);
    v = MAX ? fmax(v, u) : fmin(v, u);
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = red[0];
  for (int i = 1; i < NT / 32; ++i) t = MAX ? fmax(t, red[i]) : fmin(t, red[i]);
  return t;
}

// ---- generic fallback: multi-rank MSB radix select, 8 passes of 8-bit digits over load(i), i in [0,n) --------------
// Every requested rank carries its own (prefix, remaining-rank) pair; ranks that still share a prefix share a
// histogram.  answers[r] = the krank[r]-th smallest value.  All threads of the CTA; ends synchronised.
template <int NT, class Load>
__device__ void radix_select_ranks(Load load, long long n, int R, const long long* krank, double* answers,
                                   unsigned int* hist /* [kMaxRanks*256] */) {
  __shared__ unsigned long long prefix[kMaxRanks], dprefix[kMaxRanks];
  __shared__ long long krem[kMaxRanks];
  __shared__ int owner[kMaxRanks];
  __shared__ int ndist_s;
  const int tid = threadIdx.x;
  if (tid < R) { krem[tid] = krank[tid]; prefix[tid] = 0ull; owner[tid] = 0; }
  if (tid == 0) { ndist_s = 1; dprefix[0] = 0ull; }
  __syncthreads();
  for (int pass = 0; pass < 8; ++pass) {
    const int ndist = ndist_s;
    for (int i = tid; i < ndist * 256; i += NT) hist[i] = 0u;
    __syncthreads();
    const int shift = 56 - 8 * pass;
    for (long long i0 = 0; i0 < n; i0 += NT) {
      const long long i = i0 + tid;
      const bool valid = i < n;
      const unsigned long long key = valid ? f64_key(load(i)) : 0ull;
      const unsigned int digit = (unsigned int)(key >> shift) & 255u;
      const unsigned long long hi = pass == 0 ? 0ull : (key >> (shift + 8));
      for (int u = 0; u < ndist; ++u) {
        const bool m = valid && (hi == dprefix[u]);
        const unsigned int mask = __ballot_sync(0xffffffffu, m);
        if (m) {
          const unsigned int peers = __match_any_sync(mask, digit);
          if ((int)(__ffs(peers) - 1) == (tid & 31)) atomicAdd(&hist[u * 256 + digit], __popc(peers));
        }
      }
    }
    __syncthreads();
    if (tid < R) {
      const int src = owner[tid];
      long long k = krem[tid];
      unsigned int d = 0;
      for (; d < 255u; ++d) {
        const unsigned int c = hist[src * 256 + d];
        if (k < (long long)c) break;
        k -= c;
      }
      krem[tid] = k;
      prefix[tid] = (prefix[tid] << 8) | d;
    }
    __syncthreads();
    if (tid == 0) {
      int nd = 0;
      for (int r = 0; r < R; ++r) {
        int o = -1;
        for (int u = 0; u < nd; ++u) if (dprefix[u] == prefix[r]) o = u;
        if (o < 0) { o = nd; dprefix[nd++] = prefix[r]; }
        owner[r] = o;
      }
      ndist_s = nd;
    }
    __syncthreads();
  }
  if (tid < R) answers[tid] = key_f64(prefix[tid]);
  __syncthreads();
}

// ---- binned select over a shared-memory column ----------------------------------------------------------------------
// vals[n] in shared memory, mn / mx = its extrema (no NaN).  hist: kStatBins + 32 words, pool: kStatPool doubles.
// Returns (uniformly) false when the selected bins overflow the pool: the caller then runs radix_select_ranks.
template <int NT>
__device__ bool binned_select_ranks(const double* vals, int n, double mn, double mx, int R, const long long* krank,
                                    double* answers, unsigned int* hist, double* pool) {
  __shared__ int s_bin[kMaxRanks], s_kin[kMaxRanks], s_cnt[kMaxRanks], s_off[kMaxRanks], s_slot[kMaxRanks];
  __shared__ int s_fill[kMaxRanks];
  __shared__ int s_total, s_nslots;
  __shared__ unsigned int s_wsum[NT / 32];
  const int tid = threadIdx.x;
  if (!(mx > mn)) {                       // constant column (or n == 1)
    if (tid < R) answers[tid] = mn;
    __syncthreads();
    return true;
  }
  const double scale = (double)kStatBins / (mx - mn);
  auto bin_of = [&](double x) {
    const int bq = (int)((x - mn) * scale);
    return bq < kStatBins - 1 ? bq : kStatBins - 1;
  };
  for (int i = tid; i < kStatBins; i += NT) hist[i] = 0u;
  __syncthreads();
  for (int i = tid; i < n; i += NT) atomicAdd(&hist[bin_of(vals[i])], 1u);
  __syncthreads();
  // inclusive scan of the bin counts, kStatBins / NT consecutive bins per thread
  {
    constexpr int PER = kStatBins / NT;
    static_assert(kStatBins % NT == 0, "bins per thread");
    unsigned int loc[PER], run = 0;
#pragma unroll
    for (int e = 0; e < PER; ++e) { run += hist[tid * PER + e]; loc[e] = run; }
    unsigned int inc = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int u = __shfl_up_sync(0xffffffffu, inc, o);
      if ((tid & 31) >= o) inc += u;
    }
    if ((tid & 31) == 31) s_wsum[tid >> 5] = inc;
    __syncthreads();
    unsigned int base = 0;
    for (int wv = 0; wv < (tid >> 5); ++wv) base += s_wsum[wv];
    base += inc - run;
#pragma unroll
    for (int e = 0; e < PER; ++e) hist[tid * PER + e] = base + loc[e];
  }
  __syncthreads();
  if (tid < R) {                          // smallest bin whose inclusive count exceeds the rank
    const unsigned int k = (unsigned int)krank[tid];
    int lo = 0, hi = kStatBins - 1;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (hist[mid] > k) hi = mid; else lo = mid + 1;
    }
    const unsigned int below = lo ? hist[lo - 1] : 0u;
    s_bin[tid] = lo;
    s_kin[tid] = (int)(k - below);
    s_cnt[tid] = (int)(hist[lo] - below);
  }
  __syncthreads();
  if (tid == 0) {                         // distinct selected bins -> pool segments
    int ns = 0, total = 0;
    for (int r = 0; r < R; ++r) {
      int sl = -1;
      for (int q = 0; q < r; ++q) if (s_bin[q] == s_bin[r]) { sl = s_slot[q]; break; }
      if (sl < 0) {
        sl = ns++;
        s_off[sl] = total;
        s_fill[sl] = 0;
        total += s_cnt[r];
      }
      s_slot[r] = sl;
    }
    s_total = total;
    s_nslots = ns;
  }
  __syncthreads();
  if (s_total > kStatPool) return false;
  // the prefix sums are no longer needed: hist[bin] becomes 1 + segment of the selected bins, 0 elsewhere
  for (int i = tid; i < kStatBins; i += NT) hist[i] = 0u;
  __syncthreads();
  if (tid < R) hist[s_bin[tid]] = (unsigned int)s_slot[tid] + 1u;
  __syncthreads();
  for (int i = tid; i < n; i += NT) {
    const double x = vals[i];
    const unsigned int sl = hist[bin_of(x)];
    if (sl) pool[s_off[sl - 1] + atomicAdd(&s_fill[sl - 1], 1)] = x;
  }
  __syncthreads();
  // member x of the segment is the k-th smallest iff #(y < x) <= k < #(y <= x); all (rank, member) pairs in parallel
  for (int r = 0; r < R; ++r) {
    const double* seg = pool + s_off[s_slot[r]];
    const int m = s_cnt[r], k = s_kin[r];
    for (int j = tid; j < m; j += NT) {
      const double x = seg[j];
      int less = 0, leq = 0;
      for (int i = 0; i < m; ++i) {
        const double y = seg[i];
        less += y < x ? 1 : 0;
        leq += y <= x ? 1 : 0;
      }
      if (less <= k && k < leq) answers[r] = x;      // ties write the same value
    }
  }
  __syncthreads();
  return true;
}

// NumPy _lerp: a + (b-a)*t, and b - (b-a)*(1-t) where t >= 0.5 (no FMA contraction)
__device__ __forceinline__ double numpy_lerp(double a, double bb, double t) {
  const double diff = __dsub_rn(bb, a);
  double v = __dadd_rn(a, __dmul_rn(diff, t));
  if (t >= 0.5) v = __dsub_rn(bb, __dmul_rn(diff, __dsub_rn(1.0, t)));
  return v;
}

// Statistics of a column already in shared memory.  pct_out[q * pct_stride]; all threads; needs `red` [32].
template <int NT>
__device__ void smem_column_stats(const double* vals, int n, double sum, double mn, double mx, bool has_nan,
                                  const StatsParams& P, double* pct_out, long long pct_stride, double* mean_out,
                                  double* std_out, unsigned int* hist, double* pool, double* red) {
  __shared__ long long s_krank[kMaxRanks];
  __shared__ double s_ans[kMaxRanks];
  const int tid = threadIdx.x;
  const double mean = sum / (double)n;
  if (mean_out != nullptr || std_out != nullptr) {
    double v = 0.0;
    for (int i = tid; i < n; i += NT) {
      const double d = vals[i] - mean;
      v = fma(d, d, v);
    }
    const double var = block_sum_nt<NT>(v, red) / (double)n;
    if (tid == 0) {
      if (mean_out) *mean_out = mean;
      if (std_out) *std_out = sqrt(var);
    }
  }
  const int R = 2 * P.npct;
  if (R == 0) return;
  if (tid < R) {
    long long k = P.lo[tid >> 1] + (tid & 1);
    if (k > n - 1) k = n - 1;
    if (k < 0) k = 0;
    s_krank[tid] = k;
  }
  __syncthreads();
  if (has_nan) {                          // np.percentile propagates NaN
    if (tid < P.npct) pct_out[tid * pct_stride] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  if (!binned_select_ranks<NT>(vals, n, mn, mx, R, s_krank, s_ans, hist, pool)) {
    // the radix histograms (R x 256 words) re-use the scratch area from its start (pool | bin table, contiguous;
    // stats_scratch_bytes() sizes it for both)
    auto load = [&](long long i) { return vals[i]; };
    radix_select_ranks<NT>(load, (long long)n, R, s_krank, s_ans, reinterpret_cast<unsigned int*>(pool));
  }
  if (tid < P.npct) pct_out[tid * pct_stride] = numpy_lerp(s_ans[2 * tid], s_ans[2 * tid + 1], P.gamma[tid]);
}

// grid (ncol, B), kStatThreads threads, dynamic shared memory stats_smem_bytes(n)
__global__ void __launch_bounds__(kStatThreads, 1) column_stats_smem_kernel(const StatsParams P) {
  extern __shared__ __align__(16) unsigned char stats_dyn[];
  __shared__ double red[32];
  constexpr int NT = kStatThreads;
  const int col = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int n = (int)P.n;
  double* vals = reinterpret_cast<double*>(stats_dyn);
  double* pool = vals + n;
  unsigned int* hist = reinterpret_cast<unsigned int*>(pool + kStatPool);
  const double* src = P.data + (size_t)b * P.n * P.ncol + col;
  double s = 0.0, mn = __longlong_as_double(0x7ff0000000000000LL), mx = -mn;
  int nan = 0;
  for (int i = tid; i < n; i += NT) {
    const double v = __ldg(src + (size_t)i * P.ncol);
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
  const size_t o = (size_t)b * P.ncol + col;
  smem_column_stats<NT>(vals, n, sum, mn, mx, has_nan, P, P.pct_out ? P.pct_out + (size_t)b * P.npct * P.ncol + col : nullptr,
                        P.ncol, P.mean_out ? P.mean_out + o : nullptr, P.std_out ? P.std_out + o : nullptr, hist, pool, red);
}

// Statistics of a column of any length read through load(i), i in [0, n): the two-pass mean / std and the generic
// radix select, without a copy of the column.  pct_out[q * pct_stride]; all threads; needs `red` [32] and `hist`
// [kMaxRanks * 256].
template <int NT, class Load>
__device__ void global_column_stats(Load load, long long n, const StatsParams& P, double* pct_out, long long pct_stride,
                                    double* mean_out, double* std_out, unsigned int* hist, double* red) {
  __shared__ long long s_krank[kMaxRanks];
  __shared__ double s_ans[kMaxRanks];
  const int tid = threadIdx.x;
  double s = 0.0;
  int nan = 0;
  for (long long i = tid; i < n; i += NT) {
    const double v = load(i);
    s += v;
    nan |= (v != v) ? 1 : 0;
  }
  const double mean = block_sum_nt<NT>(s, red) / (double)n;
  const bool has_nan = __syncthreads_or(nan) != 0;
  if (mean_out != nullptr || std_out != nullptr) {
    double v = 0.0;
    for (long long i = tid; i < n; i += NT) {
      const double d = load(i) - mean;
      v = fma(d, d, v);
    }
    const double var = block_sum_nt<NT>(v, red) / (double)n;
    if (tid == 0) {
      if (mean_out) *mean_out = mean;
      if (std_out) *std_out = sqrt(var);
    }
  }
  const int R = 2 * P.npct;
  if (R == 0) return;
  if (tid < R) {
    long long k = P.lo[tid >> 1] + (tid & 1);
    if (k > n - 1) k = n - 1;
    if (k < 0) k = 0;
    s_krank[tid] = k;
  }
  __syncthreads();
  if (has_nan) {
    if (tid < P.npct) pct_out[(size_t)tid * pct_stride] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  radix_select_ranks<NT>(load, n, R, s_krank, s_ans, hist);
  if (tid < P.npct) pct_out[(size_t)tid * pct_stride] = numpy_lerp(s_ans[2 * tid], s_ans[2 * tid + 1], P.gamma[tid]);
}

// Columns that do not fit in shared memory: the same statistics straight from global memory (strided reads, the
// generic radix select).  grid (ncol, B), kThreads threads.
__global__ void __launch_bounds__(kThreads) column_stats_global_kernel(const StatsParams P) {
  __shared__ unsigned int hist[kMaxRanks * 256];
  __shared__ double red[32];
  const int col = blockIdx.x, b = blockIdx.y;
  const double* src = P.data + (size_t)b * P.n * P.ncol + col;
  const size_t stride = P.ncol;
  auto load = [&](long long i) { return __ldg(src + (size_t)i * stride); };
  const size_t o = (size_t)b * P.ncol + col;
  global_column_stats<kThreads>(load, P.n, P, P.pct_out ? P.pct_out + (size_t)b * P.npct * P.ncol + col : nullptr, P.ncol,
                                P.mean_out ? P.mean_out + o : nullptr, P.std_out ? P.std_out + o : nullptr, hist, red);
}

}  // namespace bisip
