// PSIS-LOO and Pareto-k diagnostics of every spectrum from its chain, read in place: bisip_psis_loo.
//
// Leave-one-out cross-validation by Pareto-smoothed importance sampling (Vehtari, Gelman & Gabry 2017; Vehtari, Simpson,
// Gelman, Yao & Gabry 2024), with the generalized Pareto fit of Zhang & Stephens (2009), step by step as ArviZ's
// psislw / _gpdfit / _gpinv with r_eff = 1.  The pointwise log-likelihood ll[s, j] is WAIC's (waic_ll over model_points:
// real and imaginary part together, with the 2 ln sigma^2 term; Z in FP64 for every precision).  For frequency j:
//   lppd_j = logsumexp_s ll - ln S;   x_s = -ll[s, j] - max_s(-ll[s, j]) = min_s ll - ll[s, j]   (log importance ratios)
//   M = ceil(min(0.2 S, 3 sqrt S)); cutoff = max((M+1)-th largest x, ln DBL_MIN); the tail T = {s : x_s > cutoff}, L = |T|
//   L > 4: k, sigma = gpdfit(exp(x_T) - exp(cutoff), ascending); if k is finite the i-th smallest tail sample gets
//          xt = min(ln(gpinv((i + 0.5) / L, k, sigma) + exp(cutoff)), 0), every other sample keeps xt = x
//   L <= 4: k = +inf, xt = x
//   elpd_loo_j = logsumexp_s(xt + ll) - logsumexp_s(xt),   p_loo_j = lppd_j - elpd_loo_j.
//
// loo_kernel: one CTA owns one (frequency, spectrum); blocks run frequency-fastest, so the N CTAs of a spectrum read its
// chain from L2.  With SMEM the CTA evaluates ll for every sample into shared memory once (a C5 kept chain of 25,600
// samples is 200 KB, one CTA per SM) and runs everything else there; without it, ll of sample i is recomputed wherever
// a pass asks for it (the radix select's 8 passes and the gather): no workspace and no length limit past the tail
// buffer.  The steps after the fill:
//   * the cutoff: ascending rank M of ll (x is a non-increasing function of ll in IEEE arithmetic), binned select in
//     shared memory with the radix fallback (stats.cuh);
//   * one pass: sum exp(ll - max) for lppd, sum exp(x - cutoff) over the body x <= cutoff, and the ll of the <= M tail
//     samples gathered into the tail buffer;
//   * the tail sorted by ll descending (x ascending; ties are equal values) by rank counting, u = exp(x) - exp(cutoff),
//     gpdfit with one warp per grid point, the smoothed values;
//   * the two logsumexps: every body sample contributes xt + ll = x + ll = min ll exactly (the identity), so only the
//     tail needs per-sample terms.
// All reductions run in a fixed order (the gathered tail is sorted before it is used), so a (frequency, spectrum)
// result depends only on its own chain and data.  loo_totals_kernel then sums every spectrum's pointwise values in
// ascending j and applies the NaN rule: two launches per call.
#pragma once
#include <cfloat>

#include "common.cuh"
#include "decomp_collapsed.cuh"
#include "model_pct.cuh"
#include "models.cuh"
#include "stats.cuh"
#include "waic.cuh"

namespace bisip {

struct LooParams {
  bisip_model_desc d;
  long long n;                      // samples per spectrum (S)
  int B;
  const double* theta;              // [B][n][ndim]
  const double* w; long long w_stride;
  const double* taus; const double* log_taus; long long tau_stride;
  const double* y; const double* yerr;              // [B][2][N]
  double* elpd_i_out; double* p_i_out; double* k_out;   // [B][N]
  double* elpd_out; double* p_loo_out; double* se_out;  // [B]
  int* n_high_k_out;                                // [B]
};

// M = ceil(min(0.2 S, 3 sqrt(S))): the tail length of psislw with r_eff = 1 (at most S - 1 for S >= 2)
__host__ __device__ inline long long loo_tail_len(long long n) {
  return (long long)ceil(fmin(0.2 * (double)n, 3.0 * sqrt((double)n)));
}
// gpdfit's grid size m = 30 + floor(sqrt(L)) for a tail of L <= M samples
__host__ __device__ inline int loo_grid_len(long long L) { return 30 + (int)floor(sqrt((double)L)); }
// the tail area: gathered ll [M], sorted ll [M] (then u, then the smoothed values), gpdfit's b, l and w [m each]
__host__ __device__ inline size_t loo_tail_bytes(long long n) {
  const long long M = loo_tail_len(n);
  return (size_t)(2 * M + 3 * (long long)loo_grid_len(M)) * 8;
}
// dynamic shared memory of the shared-memory kernel: the ll column, then the scratch area that the selection uses first
// and the tail after it (stats_scratch_bytes(1) at every chain that fits, e.g. C5's S = 25,600)
__host__ __device__ inline size_t loo_smem_bytes(long long n) {
  const size_t sel = stats_scratch_bytes(1), tail = loo_tail_bytes(n);
  return (size_t)n * 8 + (sel > tail ? sel : tail);
}

// fixed-order block reduction (sum, or max with MAX), result in every thread: lanes by xor-shuffle, then the warp
// partials by one warp's shuffle tree.  block_sum_nt's 32 loads per thread spill at the 64 registers of a 1024-thread CTA.
template <int NT, bool MAX>
__device__ __forceinline__ double loo_reduce(double v, double* red) {
  const int tid = threadIdx.x;
  auto op = [](double a, double b) { return MAX ? fmax(a, b) : a + b; };
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((tid & 31) == 0) red[tid >> 5] = v;
  __syncthreads();
  if (tid < 32) {
    v = tid < NT / 32 ? red[tid] : red[0];           // MAX: a repeat changes nothing; the sum masks it below
    if (!MAX && tid >= NT / 32) v = 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (tid == 0) red[32] = v;
  }
  __syncthreads();
  return red[32];
}

// generalized Pareto fit of u[0..L) (ascending, shared memory), Zhang & Stephens 2009 as ArviZ's _gpdfit: one warp per
// grid point, lanes stride the samples, fixed-order shuffle sums.  Not inlined: inside loo_kernel it spills at 64 registers.  g: 3 m doubles of shared scratch.  All threads; on
// return (synchronised) res[0] = k with the weakly informative prior, res[1] = sigma.
template <int NT>
__device__ __noinline__ void loo_gpdfit(const double* u, int L, double* g, double* res) {
  const int tid = threadIdx.x, lane = tid & 31;
  const int m = loo_grid_len(L);
  double* gb = g;
  double* gl = g + m;
  double* gw = g + 2 * m;
  const double q3 = 3.0 * u[(int)((double)L / 4.0 + 0.5) - 1], inv_max = 1.0 / u[L - 1];
  for (int i = tid >> 5; i < m; i += NT / 32) {
    const double b = (1.0 - sqrt((double)m / ((double)(i + 1) - 0.5))) / q3 + inv_max;
    double s = 0.0;
    for (int t = lane; t < L; t += 32) s += log1p(-b * u[t]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double k = s / (double)L;
    if (lane == 0) {
      gb[i] = b;
      gl[i] = (double)L * (log(-(b / k)) - k - 1.0);
    }
  }
  __syncthreads();
  if (tid < m) {                                   // w_i = 1 / sum_h exp(l_h - l_i); an overflow gives w_i = 0
    double s = 0.0;
    for (int h = 0; h < m; ++h) s += exp(gl[h] - gl[tid]);
    gw[tid] = 1.0 / s;
  }
  __syncthreads();
  if (tid < 32) {                                  // drop negligible weights, renormalise, posterior mean of b, k
    double wsum = 0.0;
    for (int i = 0; i < m; ++i) wsum += gw[i] >= 10.0 * DBL_EPSILON ? gw[i] : 0.0;
    double bp = 0.0;
    for (int i = 0; i < m; ++i) bp += gw[i] >= 10.0 * DBL_EPSILON ? gb[i] * (gw[i] / wsum) : 0.0;
    double s = 0.0;
    for (int t = lane; t < L; t += 32) s += log1p(-bp * u[t]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double kh = s / (double)L;
    if (lane == 0) {
      res[0] = ((double)L * kh + 5.0) / (double)(L + 10);
      res[1] = -kh / bp;
    }
  }
  __syncthreads();
}

// inverse GPD distribution function, as ArviZ's _gpinv for 0 < p < 1
__device__ __forceinline__ double loo_gpinv(double p, double k, double sigma) {
  if (!(sigma > 0.0)) return __longlong_as_double(0x7ff8000000000000LL);
  if (fabs(k) < DBL_EPSILON) return -log1p(-p) * sigma;
  return expm1(-k * log1p(-p)) / k * sigma;
}

// grid (N, B).  SMEM: kStatThreads threads, dynamic shared memory loo_smem_bytes(n); else kThreads threads and
// loo_tail_bytes(n).  One instantiation per model (MODEL == P.d.model), as waic_kernel.
template <int MODEL, bool SMEM>
__global__ void __launch_bounds__(SMEM ? kStatThreads : kThreads, 1) loo_kernel(const LooParams P) {
  constexpr int NT = SMEM ? kStatThreads : kThreads;
  extern __shared__ __align__(16) unsigned char loo_dyn[];
  __shared__ double red[33];
  __shared__ double s_g[2 * kMaxCoefPct];
  __shared__ __align__(16) double s_fq[kFq];
  __shared__ double s_dat[5];                      // y_re, y_im, 1/s_re, 1/s_im, -(ln s_re + ln s_im)
  __shared__ long long s_rank;
  __shared__ double s_cut, s_gpd[2];
  __shared__ int s_L;
  __shared__ double s_lse[3];                      // max ll, sum exp(ll - max), the body's sum exp(x - cutoff)
  const int j = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  bisip_model_desc d = P.d;
  d.model = MODEL;
  const int N = d.n_freq, ndim = d.ndim;
  const long long n = P.n;
  const double* theta = P.theta + (size_t)b * n * ndim;
  const double wj = P.w[(size_t)b * P.w_stride + j];
  if (MODEL == BISIP_MODEL_DECOMP) {
    const int D = d.n_coef, S = d.n_tau;
    const double* taus = P.taus + (size_t)b * P.tau_stride;
    const double* lts = P.log_taus + (size_t)b * P.tau_stride * D;
    if (tid < 2 * D) {                             // s_g[2 q + part], the layout of model_points<1>
      double cs, sn;
      sincospi(0.5 * d.c_exp, &sn, &cs);
      s_g[tid] = dot2_lk(lts + (size_t)(tid >> 1) * S, taus, S, wj, d.c_exp, cs, sn, (tid & 1) != 0, 1.0);
    }
  } else if (tid == 0) {
    s_fq[0] = wj; s_fq[1] = sqrt(wj); s_fq[2] = log(wj);
    for (int i = 3; i < kFq; ++i) s_fq[i] = 0.0;
  }
  if (tid == 0) {
    const double* y = P.y + (size_t)b * 2 * N;
    const double* ye = P.yerr + (size_t)b * 2 * N;
    const double s0 = ye[j] * ye[j], s1 = ye[N + j] * ye[N + j];
    s_dat[0] = y[j]; s_dat[1] = y[N + j];
    s_dat[2] = 1.0 / s0; s_dat[3] = 1.0 / s1;
    s_dat[4] = -(log(s0) + log(s1));
    s_rank = loo_tail_len(n);                      // ascending rank of ll whose x is the (M+1)-th largest
    s_L = 0;
  }
  __syncthreads();
  auto ll_of = [&](long long i) {
    double zre[1], zim[1];
    model_points<1>(d, theta + (size_t)i * ndim, s_g, s_fq, zre, zim);
    return waic_ll(zre[0], zim[0], s_dat[0], s_dat[1], s_dat[2], s_dat[3], s_dat[4]);
  };
  double* vals = reinterpret_cast<double*>(loo_dyn);
  double* scratch = SMEM ? vals + n : vals;
  auto load = [&](long long i) { return SMEM ? vals[i] : ll_of(i); };

  // fill: min, max and NaN of ll (the column into shared memory)
  double mn = __longlong_as_double(0x7ff0000000000000LL), mx = -mn;
  int nan = 0;
  for (long long i = tid; i < n; i += NT) {
    const double v = ll_of(i);
    if (SMEM) vals[i] = v;
    mn = fmin(mn, v);
    mx = fmax(mx, v);
    nan |= (v != v) ? 1 : 0;
  }
  mn = -loo_reduce<NT, true>(-mn, red);            // min as an exact negated max
  mx = loo_reduce<NT, true>(mx, red);
  const size_t o = (size_t)b * N + j;
  if (__syncthreads_or(nan)) {                     // the totals kernel turns the whole spectrum into NaN
    if (tid == 0) P.elpd_i_out[o] = P.p_i_out[o] = P.k_out[o] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }

  // the cutoff
  {
    unsigned int* hist = reinterpret_cast<unsigned int*>(scratch + (SMEM ? kStatPool : 0));
    bool done = false;
    if (SMEM) done = binned_select_ranks<NT>(vals, (int)n, mn, mx, 1, &s_rank, &s_cut, hist, scratch);
    if (!done) radix_select_ranks<NT>(load, n, 1, &s_rank, &s_cut, reinterpret_cast<unsigned int*>(scratch));
  }
  const double cutoff = fmax(mn - s_cut, log(DBL_MIN));
  const long long M = loo_tail_len(n);
  double* tl = scratch;                            // gathered tail ll, then u, then the smoothed values
  double* ts = scratch + M;                        // the tail ll, sorted descending
  __syncthreads();                                 // the selection's scratch becomes the tail

  // lppd's sum, the body's sum exp(x - cutoff), and the tail gathered
  double se = 0.0, sa = 0.0;
  for (long long i = tid; i < n; i += NT) {
    const double v = load(i);
    se += exp(v - mx);
    const double x = mn - v;
    if (x > cutoff) tl[atomicAdd(&s_L, 1)] = v;
    else sa += exp(x - cutoff);
  }
  se = loo_reduce<NT, false>(se, red);
  sa = loo_reduce<NT, false>(sa, red);
  if (tid == 0) { s_lse[0] = mx; s_lse[1] = se; s_lse[2] = sa; }   // thread 0 reads them back at the end
  const int L = s_L;
  for (int t = tid; t < L; t += NT) {              // rank by ll descending; equal ll are equal values, in any order
    const double v = tl[t];
    int r = 0;
    for (int q = 0; q < L; ++q) {
      const double y = tl[q];
      r += (y > v || (y == v && q < t)) ? 1 : 0;
    }
    ts[r] = v;
  }
  __syncthreads();

  const double ec = exp(cutoff);
  double k = __longlong_as_double(0x7ff0000000000000LL);
  bool smooth = false;
  if (L > 4) {
    for (int t = tid; t < L; t += NT) tl[t] = exp(mn - ts[t]) - ec;
    __syncthreads();
    loo_gpdfit<NT>(tl, L, ts + M, s_gpd);
    k = s_gpd[0];
    smooth = isfinite(k);
    if (smooth) {
      const double sigma = s_gpd[1];
      for (int t = tid; t < L; t += NT) tl[t] = fmin(log(loo_gpinv(((double)t + 0.5) / (double)L, k, sigma) + ec), 0.0);
    }
  }
  if (!smooth)
    for (int t = tid; t < L; t += NT) tl[t] = mn - ts[t];
  __syncthreads();

  // logsumexp_s(xt) and logsumexp_s(xt + ll): the body as summed above and, smoothed, (S - L) terms of exactly min ll
  double ma = -__longlong_as_double(0x7ff0000000000000LL), mb = ma;
  for (int t = tid; t < L; t += NT) {
    ma = fmax(ma, tl[t]);
    mb = fmax(mb, tl[t] + ts[t]);
  }
  ma = fmax(loo_reduce<NT, true>(ma, red), cutoff);
  mb = smooth ? fmax(loo_reduce<NT, true>(mb, red), mn) : mn;
  double ta = 0.0, tb = 0.0;
  for (int t = tid; t < L; t += NT) {
    ta += exp(tl[t] - ma);
    tb += exp((tl[t] + ts[t]) - mb);
  }
  ta = loo_reduce<NT, false>(ta, red);
  tb = loo_reduce<NT, false>(tb, red);
  if (tid == 0) {
    const double A = fma(s_lse[2], exp(cutoff - ma), ta);
    const double Bs = smooth ? fma((double)(n - s_L), exp(mn - mb), tb) : (double)n;
    const double lppd = (s_lse[0] + log(s_lse[1])) - log((double)n);
    const double elpd = (mb + log(Bs)) - (ma + log(A));
    P.elpd_i_out[o] = elpd;
    P.p_i_out[o] = lppd - elpd;
    P.k_out[o] = k;
  }
}

// Per-spectrum totals in ascending j, the count of high k, and the NaN rule.  One thread per spectrum, 128 per CTA.
__global__ void __launch_bounds__(128) loo_totals_kernel(const LooParams P) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  const int N = P.d.n_freq;
  double* e = P.elpd_i_out + (size_t)b * N;
  double* p = P.p_i_out + (size_t)b * N;
  double* k = P.k_out + (size_t)b * N;
  const double thr = fmin(1.0 - 1.0 / log10((double)P.n), 0.7);
  double es = 0.0, ps = 0.0;
  int nh = 0;
  bool any_nan = false;
  for (int j = 0; j < N; ++j) {
    es += e[j];
    ps += p[j];
    nh += k[j] > thr ? 1 : 0;
    any_nan |= e[j] != e[j];
  }
  double ss = 0.0;
  const double em = es / (double)N;
  for (int j = 0; j < N; ++j) {
    const double dv = e[j] - em;
    ss = fma(dv, dv, ss);
  }
  if (any_nan) {
    const double nan_v = __longlong_as_double(0x7ff8000000000000LL);
    for (int j = 0; j < N; ++j) e[j] = p[j] = k[j] = nan_v;
    es = ps = ss = nan_v;
    nh = 0;
  }
  P.elpd_out[b] = es;
  P.p_loo_out[b] = ps;
  P.se_out[b] = sqrt((double)N * (ss / (double)(N - 1)));
  P.n_high_k_out[b] = nh;
}

}  // namespace bisip
