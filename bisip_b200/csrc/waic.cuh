// WAIC of every spectrum from its chain, read in place: bisip_waic.
//
// The widely applicable information criterion (Watanabe; computed as in Vehtari, Gelman & Gabry 2017) needs the
// pointwise log-likelihood ll[s, j] of every sample s at every frequency j (one data point per frequency: its real and
// imaginary part are one measurement), reduced over the samples to
//   lppd[j] = logsumexp_s ll[s, j] - log n,   p[j] = var_s(ll[s, j], ddof=1),   elpd[j] = lppd[j] - p[j].
// The (n, N) matrix ll is never stored.  One CTA owns one spectrum and walks its frequencies in tiles of waic_tile(model); for
// each tile it makes two passes over the samples, recomputing Z (model_points, model_pct.cuh: FP64 for every
// precision, each sample's Z at a frequency once for both parts):
//   pass 1: per-frequency max and sum of ll;   pass 2: sum exp(ll - max) and sum (ll - mean)^2.
// Each sample is owned by one thread (i = tid, tid + NT, ...) and the per-thread partials are reduced in a fixed
// order, and the per-spectrum totals are summed by one thread in ascending frequency order: a spectrum's result
// depends only on its own chain and data, not on the batch, the sub-batch size or the number of ranks.  No workspace,
// no length limit on the chain; one launch per call.
#pragma once
#include "common.cuh"
#include "decomp_collapsed.cuh"
#include "model_pct.cuh"
#include "models.cuh"
#include "stats.cuh"

namespace bisip {

constexpr int kWaicThreads = 256;
// Frequencies per tile: 2F accumulators per thread and pass, and one read of the chain per F frequencies and pass.
// The decomposition reads G from shared memory and keeps 8 without spilling; the per-mode exp / sincospi of the other
// models spill past 4.
__host__ __device__ constexpr int waic_tile(int model) { return model == BISIP_MODEL_DECOMP ? 8 : 4; }

struct WaicParams {
  bisip_model_desc d;
  long long n;                      // samples per spectrum
  const double* theta;              // [B][n][ndim]
  const double* w; long long w_stride;
  const double* taus; const double* log_taus; long long tau_stride;
  const double* y; const double* yerr;          // [B][2][N]
  double* lppd_out; double* p_out;              // [B][N]
  double* elpd_out; double* p_waic_out; double* se_out;   // [B]
  int* n_high_p_out;                            // [B]
};

// ll of one (sample, frequency): -0.5 (r_re^2 / s_re + r_im^2 / s_im) - (ln s_re + ln s_im), s = yerr^2.  The constant
// keeps the reference likelihood's 2 ln sigma^2 term, so sum_j ll[s, j] is the log-likelihood of the sample.
__device__ __forceinline__ double waic_ll(double zre, double zim, double yre, double yim, double ire, double iim,
                                          double cst) {
  const double rre = yre - zre, rim = yim - zim;
  return fma(-0.5, fma(rre * rre, ire, rim * rim * iim), cst);
}

// grid (B), kWaicThreads threads, no dynamic shared memory.  One instantiation per model (MODEL == P.d.model): the
// model switch of model_points folds away, and the registers are those of one model's evaluation.
template <int MODEL>
__global__ void __launch_bounds__(kWaicThreads) waic_kernel(const WaicParams P) {
  constexpr int NT = kWaicThreads, F = waic_tile(MODEL);
  __shared__ __align__(16) double s_g[kMaxCoefPct * 2 * F];   // decomposition: G of the tile, model_points<F> layout
  __shared__ __align__(16) double s_fq[F * kFq];              // other models: the tile's frequency records
  __shared__ double s_dat[5][F];                              // y_re, y_im, 1/s_re, 1/s_im, -(ln s_re + ln s_im)
  __shared__ double red[32];
  const int b = blockIdx.x, tid = threadIdx.x;
  bisip_model_desc d = P.d;
  d.model = MODEL;
  const int N = d.n_freq, ndim = d.ndim;
  const long long n = P.n;
  const double* theta = P.theta + (size_t)b * n * ndim;
  const double* w = P.w + (size_t)b * P.w_stride;
  const double* y = P.y + (size_t)b * 2 * N;
  const double* ye = P.yerr + (size_t)b * 2 * N;
  double* lppd_out = P.lppd_out + (size_t)b * N;
  double* p_out = P.p_out + (size_t)b * N;
  const double log_n = log((double)n), inv_n = 1.0 / (double)n, inv_n1 = 1.0 / (double)(n - 1);
  bool any_nan = false;
  double elpd_sum = 0.0, p_sum = 0.0;
  int n_high = 0;

  for (int j0 = 0; j0 < N; j0 += F) {
    const int nf = min(F, N - j0);
    // tile constants; slots past the last frequency repeat it (evaluated, never written out)
    if (MODEL == BISIP_MODEL_DECOMP) {
      const int D = d.n_coef, S = d.n_tau;
      const double* taus = P.taus + (size_t)b * P.tau_stride;
      const double* lts = P.log_taus + (size_t)b * P.tau_stride * D;
      double cs, sn;
      sincospi(0.5 * d.c_exp, &sn, &cs);
      for (int t = tid; t < D * 2 * F; t += NT) {
        const int q = t / (2 * F), r = t - q * 2 * F;
        const int f = r < F ? r : r - F;
        const double wj = w[j0 + min(f, nf - 1)];
        s_g[t] = dot2_lk(lts + (size_t)q * S, taus, S, wj, d.c_exp, cs, sn, r >= F, 1.0);
      }
    } else if (tid < F) {
      const double wj = w[j0 + min(tid, nf - 1)];
      double* f = s_fq + tid * kFq;
      f[0] = wj; f[1] = sqrt(wj); f[2] = log(wj);
      for (int i = 3; i < kFq; ++i) f[i] = 0.0;
    }
    if (tid < F) {
      const int j = j0 + min(tid, nf - 1);
      const double e0 = ye[j], e1 = ye[N + j];
      const double s0 = e0 * e0, s1 = e1 * e1;
      s_dat[0][tid] = y[j];
      s_dat[1][tid] = y[N + j];
      s_dat[2][tid] = 1.0 / s0;
      s_dat[3][tid] = 1.0 / s1;
      s_dat[4][tid] = -(log(s0) + log(s1));
    }
    __syncthreads();

    // pass 1: max and sum of ll per frequency
    double mx[F], mean[F];
    {
      double sm[F];
#pragma unroll
      for (int f = 0; f < F; ++f) { mx[f] = -__longlong_as_double(0x7ff0000000000000LL); sm[f] = 0.0; }
      int nan = 0;
#pragma unroll 1
  #pragma unroll 1
    for (long long i = tid; i < n; i += NT) {
        double zre[F], zim[F];
        model_points<F>(d, theta + (size_t)i * ndim, s_g, s_fq, zre, zim);
#pragma unroll
        for (int f = 0; f < F; ++f) {
          const double ll = waic_ll(zre[f], zim[f], s_dat[0][f], s_dat[1][f], s_dat[2][f], s_dat[3][f], s_dat[4][f]);
          mx[f] = fmax(mx[f], ll);
          sm[f] += ll;
          nan |= (ll != ll) ? 1 : 0;
        }
      }
      any_nan |= __syncthreads_or(nan) != 0;
#pragma unroll
      for (int f = 0; f < F; ++f) {
        mx[f] = block_minmax_nt<NT, true>(mx[f], red);
        mean[f] = block_sum_nt<NT>(sm[f], red) * inv_n;
      }
    }

    // pass 2: sum exp(ll - max) and sum (ll - mean)^2 per frequency
    double se[F], sq[F];
#pragma unroll
    for (int f = 0; f < F; ++f) se[f] = sq[f] = 0.0;
#pragma unroll 1
    for (long long i = tid; i < n; i += NT) {
      double zre[F], zim[F];
      model_points<F>(d, theta + (size_t)i * ndim, s_g, s_fq, zre, zim);
#pragma unroll
      for (int f = 0; f < F; ++f) {
        const double ll = waic_ll(zre[f], zim[f], s_dat[0][f], s_dat[1][f], s_dat[2][f], s_dat[3][f], s_dat[4][f]);
        se[f] += exp(ll - mx[f]);
        const double dv = ll - mean[f];
        sq[f] = fma(dv, dv, sq[f]);
      }
    }
#pragma unroll
    for (int f = 0; f < F; ++f) {
      se[f] = block_sum_nt<NT>(se[f], red);
      sq[f] = block_sum_nt<NT>(sq[f], red);
    }
    if (tid == 0) {
      for (int f = 0; f < nf; ++f) {
        const double lppd = mx[f] + log(se[f]) - log_n;
        const double p = sq[f] * inv_n1;
        lppd_out[j0 + f] = lppd;
        p_out[j0 + f] = p;
        elpd_sum += lppd - p;
        p_sum += p;
        n_high += p > 0.4 ? 1 : 0;
      }
    }
    __syncthreads();                                // the tile's shared constants are rewritten next
  }

  if (tid != 0) return;
  // se_elpd_waic = sqrt(N var_j(elpd, ddof=1)), two-pass over the pointwise values this thread wrote
  const double nan_v = __longlong_as_double(0x7ff8000000000000LL);
  double ss = 0.0;
  const double em = elpd_sum / (double)N;
  for (int j = 0; j < N; ++j) {
    const double dv = (lppd_out[j] - p_out[j]) - em;
    ss = fma(dv, dv, ss);
  }
  if (any_nan) {
    for (int j = 0; j < N; ++j) { lppd_out[j] = nan_v; p_out[j] = nan_v; }
    elpd_sum = p_sum = ss = nan_v;
    n_high = 0;
  }
  P.elpd_out[b] = elpd_sum;
  P.p_waic_out[b] = p_sum;
  P.se_out[b] = sqrt((double)N * (ss / (double)(N - 1)));
  P.n_high_p_out[b] = n_high;
}

}  // namespace bisip
