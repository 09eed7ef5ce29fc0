/*
 * bisip_b200 — C ABI of the B200-native BISIP MCMC likelihood hot path.
 *
 * This header is the drop-in boundary (SURVEY.md §8b): a shared library
 * (bisip_b200/csrc/libbisip_b200.so) with `extern "C"` entry points that take plain
 * pointers, sizes and a CUDA stream handle — no torch / C++ types.  All data pointers are
 * DEVICE pointers to float64 (unless stated); the library never allocates, frees or copies
 * caller memory and keeps no global state besides a thread-local last-error string.
 * Every function returns 0 on success, a negative BISIP_ERR_* otherwise.
 *
 * Reference interfaces replaced (paths relative to /root/reference/src/bisip/):
 *   bisip_forward            <- ColeCole_cyth / Dias2000_cyth / Decomp_cyth / Shin2015_cyth
 *                               (cython_funcs.pyx:49, :64, :75, :96), called from
 *                               Model.forward (models.py:228, :267, :305, :345)
 *   bisip_log_probability    <- Inversion._log_probability/_log_prior/_log_likelihood
 *                               (models.py:59-76)
 *   bisip_decomp_build_kernel<- the theta-independent term of C_Debye (cython_funcs.pyx:46-47)
 *   bisip_ensemble_run       <- emcee.EnsembleSampler(...).run_mcmc as driven by
 *                               Inversion.fit (models.py:111-118); chain layout/slicing of
 *                               sampler.get_chain (models.py:137)
 *   bisip_column_stats       <- np.percentile / np.mean / np.std over the flat chain
 *                               (utils.py:35, :53, :69, :85)
 *   bisip_model_percentile   <- utils.get_model_percentile (utils.py:17-35)
 *   bisip_autocorr_time      <- emcee autocorr.integrated_time, reached through
 *                               sampler.get_autocorr_time (models.py:154-159)
 *   bisip_rtd_stats          <- relaxation_time_distribution / total_m of decomposition.ipynb
 *                               cells 25-29 over the chain, then np.percentile / mean / std
 *   bisip_waic               <- (no counterpart: the tutorials compare models by eye with plot_fit)
 *   bisip_psis_loo           <- (no counterpart: the reference has no leave-one-out cross-validation)
 *
 * Layouts (all row-major, float64):
 *   theta   [n_spectra][n_theta][ndim]      parameter vectors (order as the reference's
 *                                           params dicts: models.py:212-213, :249-252,
 *                                           :287-291, :325-331)
 *   w       [n_freq] (w_stride==0: shared by all spectra) or [n_spectra][w_stride]
 *   taus    [n_tau], log_taus [n_coef][n_tau]   (tau_stride==0: shared) or per spectrum
 *           taus + b*tau_stride, log_taus + b*tau_stride*n_coef   (models.py:204-209)
 *   y, yerr [n_spectra][2][n_freq]          zn / zn_err: rows = [real; imag] (utils.py:141-142)
 *   bounds  [2][ndim]                       row 0 lower, row 1 upper (models.py:176-179)
 *   Z       [n_spectra][n_theta][2][n_freq] forward output, rows = [real; imag]
 */
#ifndef BISIP_B200_H
#define BISIP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BISIP_ABI_VERSION 2

enum bisip_model {
  BISIP_MODEL_COLECOLE = 0, /* PeltonColeCole, models.py:232 */
  BISIP_MODEL_DIAS = 1,     /* Dias2000,       models.py:274 */
  BISIP_MODEL_SHIN = 2,     /* Shin2015,       models.py:308 */
  BISIP_MODEL_DECOMP = 3    /* PolynomialDecomposition, models.py:182 */
};

enum bisip_precision {
  BISIP_PREC_FP64 = 0,  /* FP64 DMMA tensor tiles (decomposition) / FP64 pipe (others) */
  BISIP_PREC_TF32 = 1,  /* decomposition stage 2 on TF32 tensor cores, FP32 accumulate: tcgen05.mma with
                           operands / accumulators in tensor memory when one 128-row tile holds a half-step
                           (<= 256 walkers, n_freq <= 64, K planes fit in shared memory), mma.sync tiles otherwise */
  BISIP_PREC_3XTF32 = 2,     /* error-compensated 3xTF32 split, same dispatch */
  BISIP_PREC_TF32_MMA = 3,   /* TF32, always the mma.sync tile kernel (kept for the comparison study) */
  BISIP_PREC_3XTF32_MMA = 4, /* 3xTF32, always the mma.sync tile kernel */
  BISIP_PREC_FP64_COLLAPSED = 5 /* FP64, decomposition re-associated to z = (L K) a: the theta-independent product
                                   G = L K ((poly_deg+1) x 2N) is built once per spectrum (compensated sums), one
                                   evaluation is 2N (poly_deg+3) FMAs: FP64 DMMA tiles of 16 proposals x 8 columns up to
                                   256 walkers, the FP64 vector pipe above.  Same 1e-12 parity bar as BISIP_PREC_FP64,
                                   ~10x fewer flops; the two-stage DMMA contraction stays the default (n_coef <= 8) */
};

enum bisip_status {
  BISIP_OK = 0,
  BISIP_ERR_BAD_ARG = -1,     /* null pointer, non-positive size, inconsistent ndim ... */
  BISIP_ERR_UNSUPPORTED = -2, /* shape outside what the kernels are built for */
  BISIP_ERR_CUDA = -3,        /* a CUDA runtime call failed; see bisip_last_error() */
  BISIP_ERR_NO_DEVICE = -4    /* no sm_100 device visible */
};

typedef struct bisip_model_desc {
  int32_t model;     /* enum bisip_model */
  int32_t ndim;      /* ColeCole 1+3*n_modes; Dias 5; Shin 6; Decomp 1+n_coef */
  int32_t n_freq;    /* N */
  int32_t n_modes;   /* ColeCole only */
  int32_t n_tau;     /* Decomp only: S */
  int32_t n_coef;    /* Decomp only: poly_deg+1 */
  int32_t precision; /* enum bisip_precision */
  int32_t reserved;
  double c_exp;      /* Decomp only: 1.0 Debye, 0.5 Warburg */
} bisip_model_desc;

/* ABI version / diagnostics ------------------------------------------------------------ */
int bisip_abi_version(void);
const char *bisip_last_error(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t bisip_launch_count(void);

/* Which decomposition kernel bisip_ensemble_run will launch for (desc, n_walkers): every one of them is a CUDA
 * kernel of this library (there is no CPU path); the choice depends on precision, tau-grid size and walker count. */
enum bisip_kernel_kind {
  BISIP_KERNEL_DMMA = 0,         /* FP64 mma.sync (DMMA) tiles, n_tau <= 64 */
  BISIP_KERNEL_DMMA_CLUSTER = 1, /* FP64 DMMA, stage-1 recompute, columns split over a CTA cluster (n_tau > 64) */
  BISIP_KERNEL_MMA_TF32 = 2,     /* TF32 / 3xTF32 mma.sync tiles */
  BISIP_KERNEL_TCGEN05 = 3,      /* TF32 / 3xTF32 tcgen05.mma, operands and accumulators in tensor memory */
  BISIP_KERNEL_TCGEN05_CLUSTER = 4, /* the same with the real | imaginary columns split over a 2-CTA cluster */
  BISIP_KERNEL_FP64_COLLAPSED = 5   /* collapsed form on the FP64 vector pipe (BISIP_PREC_FP64_COLLAPSED, any n_tau) */
};
int bisip_decomp_kernel_kind(const bisip_model_desc *desc, int n_walkers);

/* Forward model for n_spectra x n_theta parameter vectors.  Z as documented above. */
int bisip_forward(const bisip_model_desc *desc, int n_spectra, int n_theta,
                  const double *theta, const double *w, int64_t w_stride,
                  const double *taus, const double *log_taus, int64_t tau_stride,
                  double *Z, void *stream);

/* Fused prior + forward + Gaussian log-likelihood (models.py:59-76):
 *   lp = -inf                                       if not all(lo < theta < hi)  (strict)
 *   lp = -0.5*sum((y-Z)^2/yerr^2 + 2*ln(yerr^2))    otherwise
 * lp_out [n_spectra][n_theta]. */
int bisip_log_probability(const bisip_model_desc *desc, int n_spectra, int n_theta,
                          const double *theta, const double *w, int64_t w_stride,
                          const double *taus, const double *log_taus, int64_t tau_stride,
                          const double *y, const double *yerr, const double *bounds,
                          double *lp_out, void *stream);

/* Gaussian log-likelihood of caller-supplied model rows (the reference's `_log_likelihood(theta, f, x, y, yerr)` with a
 * user callable `f`, models.py:59-62: the callable runs where the user wrote it, on the host; the reduction runs here):
 *   ll_out[r] = -0.5*sum_c((y[c]-Z[r][c])^2/yerr[c]^2 + 2*ln(yerr[c]^2)),  Z [n_rows][2*n_freq], y / yerr [2*n_freq]. */
int bisip_gauss_loglike(const double *Z, const double *y, const double *yerr, int n_freq, int n_rows,
                        double *ll_out, void *stream);

/* Decomposition kernel matrix K[n_tau][2*n_freq] = 1 - 1/(1 + (i w tau)^c): columns
 * [0,N) real parts, [N,2N) imaginary parts. */
int bisip_decomp_build_kernel(const double *w, int n_freq, const double *taus, int n_tau,
                              double c_exp, double *K, void *stream);

/* Number of stored steps for (nsteps, discard, thin): emcee's
 * chain[discard+thin-1 : nsteps : thin] (SURVEY.md App. B.4). */
int bisip_n_keep(int nsteps, int discard, int thin);

/*
 * On-device affine-invariant ensemble sampler (emcee StretchMove semantics, SURVEY App. B):
 * one CTA owns one spectrum for all nsteps; walkers never leave the SM between steps.
 *
 *   coords   [n_spectra][n_walkers][ndim]  in: p0, out: final ensemble
 *   lp       [n_spectra][n_walkers]        out: final log-probabilities
 *   chain    [n_spectra][n_keep][n_walkers][ndim] or NULL   (emcee (nsteps,nwalkers,ndim) layout
 *                                                             per spectrum; only kept steps stored)
 *   logp     [n_spectra][n_keep][n_walkers] or NULL
 *   accepted [n_spectra][n_walkers] int32  accepted-move counts over all nsteps
 *   flags    [n_spectra] int32             bit 0: a NaN log-probability was produced
 *                                          (emcee raises ValueError), bit 1: NaN at p0
 * RNG: Philox4x32-10, key = seed, counter = (index, step0+step, spectrum0+b, purpose) —
 * results are independent of how spectra are batched or sharded over GPUs.
 * a: stretch scale (emcee default 2.0).
 */
int bisip_ensemble_run(const bisip_model_desc *desc, int n_spectra, int n_walkers, int nsteps,
                       int step0, uint64_t seed, uint32_t spectrum0, double a,
                       int discard, int thin,
                       const double *w, int64_t w_stride,
                       const double *taus, const double *log_taus, int64_t tau_stride,
                       const double *y, const double *yerr, const double *bounds,
                       double *coords, double *lp, double *chain, double *logp,
                       int32_t *accepted, int32_t *flags, void *stream);

/*
 * Column statistics of data[n_spectra][n_samples][n_cols] (a flat chain is
 * [n_keep*n_walkers][ndim]): exact order statistics with NumPy's default 'linear'
 * interpolation, mean and population std (ddof=0).  The data is read in place (one CTA per
 * column keeps it in shared memory when n_samples <= ~27,000, else strided global reads).
 *   pct_lo[n_pct] int64: floor of the virtual index q/100*(n_samples-1)
 *   pct_gamma[n_pct]   : its fractional part (both computed by the host exactly like NumPy)
 *   pct_out [n_spectra][n_pct][n_cols]; mean_out, std_out [n_spectra][n_cols] (may be NULL)
 *   workspace, workspace_bytes: unused since ABI 2 (pass NULL, 0); bisip_column_stats_workspace returns 0.
 */
int64_t bisip_column_stats_workspace(int n_spectra, int64_t n_samples, int n_cols);
int bisip_column_stats(const double *data, int n_spectra, int64_t n_samples, int n_cols,
                       int n_pct, const int64_t *pct_lo, const double *pct_gamma,
                       double *pct_out, double *mean_out, double *std_out,
                       void *workspace, int64_t workspace_bytes, void *stream);

/*
 * Percentiles of the forward model over a chain, fused (replaces utils.get_model_percentile,
 * utils.py:17-35: one forward() per flat-chain sample into an (n, 2, N) array, then
 * np.percentile over axis 0).  One CTA per model column evaluates it for all n_theta parameter
 * vectors into shared memory and selects there: the (n_theta, 2N) model matrix is never
 * written to memory.
 *   theta   [n_spectra][n_theta][ndim]
 *   pct_out [n_spectra][n_pct][2][n_freq]
 * The decomposition is evaluated in its collapsed FP64 column form for every desc->precision;
 * ColeCole n_modes and Decomp n_coef (<= 32) are not limited to the sampler kernels' tile shapes.
 * BISIP_ERR_UNSUPPORTED when n_theta exceeds one CTA's shared memory (~27,000): compose
 * bisip_forward + bisip_column_stats instead.
 */
int bisip_model_percentile(const bisip_model_desc *desc, int n_spectra, int64_t n_theta,
                           const double *theta, const double *w, int64_t w_stride,
                           const double *taus, const double *log_taus, int64_t tau_stride,
                           int n_pct, const int64_t *pct_lo, const double *pct_gamma,
                           double *pct_out, void *stream);

/*
 * emcee's integrated autocorrelation time (Sokal window, constant c) of every column of
 * data[n_spectra][n_keep][n_walkers][n_cols], read in place; tau_out[n_spectra][n_cols] in rows of `data`.
 * Reference: emcee autocorr.integrated_time, reached through sampler.get_autocorr_time (models.py:154-159).
 * Each walker's series is centred on its own mean, its linear ACF normalised by its lag-0 value, the walkers
 * averaged, tau(L) = 2 sum_{l<=L} rho(l) - 1, and the result is tau at emcee's automatic window (the first L
 * with L >= c tau(L)).  In steps of the kept chain: multiply by the thinning for steps of the run.
 * A column with a constant walker (this includes n_keep == 1) or a NaN gives NaN.  The result of a spectrum
 * depends on its own column only.  One launch; the lags stop at the window.
 * BISIP_ERR_BAD_ARG: null pointer, non-positive size, c not finite or <= 0;
 * BISIP_ERR_UNSUPPORTED: n_spectra > 65535.
 */
int bisip_autocorr_time(const double *data, int n_spectra, int n_keep, int n_walkers, int n_cols,
                        double c, double *tau_out, void *stream);

/*
 * Relaxation-time distribution and total chargeability of a polynomial decomposition over a chain, read in place
 * (replaces products.relaxation_time_distribution of every flat-chain sample + np.percentile / np.mean / np.std;
 * reference docs/tutorials/decomposition.ipynb cells 25-29).
 *   theta    [n_spectra][n_samples][ndim]   r0, a_0 .. a_{n_coef-1} (r0 is not used); ndim == 1 + n_coef
 *   log_taus [n_coef][n_tau] (tau_stride 0: shared) or per spectrum at b*tau_stride*n_coef, as in bisip_forward
 * Column l < n_tau: m_l = sum_i a_i log_taus[i][l], accumulated in ascending i from 0 with unfused multiply and add
 * (products.relaxation_time_distribution's arithmetic: every value equals NumPy's bit for bit).  Column n_tau: the
 * total chargeability sum_l m_l of the same sample, evaluated as sum_i a_i (sum_l log_taus[i][l]) (equal up to
 * rounding).  Statistics per column as bisip_column_stats: exact 'linear' percentiles (pct_lo / pct_gamma as there),
 * mean and population std; a NaN sample gives NaN percentiles.
 *   pct_out [n_spectra][n_pct][n_tau+1]; mean_out, std_out [n_spectra][n_tau+1] (each may be NULL, not all three)
 * One launch; columns longer than one CTA's shared memory (~27,000 samples) are read from global memory, with no
 * workspace and no length limit.
 * BISIP_ERR_BAD_ARG: null pointer, non-positive size, ndim != 1 + n_coef, tau_stride < 0, no output;
 * BISIP_ERR_UNSUPPORTED: n_pct > 16, n_spectra > 65535, n_coef > 32.
 */
int bisip_rtd_stats(int n_spectra, int64_t n_samples, int ndim, int n_coef, int n_tau,
                    const double *theta, const double *log_taus, int64_t tau_stride,
                    int n_pct, const int64_t *pct_lo, const double *pct_gamma,
                    double *pct_out, double *mean_out, double *std_out, void *stream);

/*
 * WAIC (Watanabe's widely applicable information criterion, as in Vehtari, Gelman & Gabry 2017) of every spectrum
 * from its chain, read in place, for comparing two models fitted to the same data.
 *   theta [n_spectra][n_theta][ndim] (n_theta >= 2), w / taus / log_taus as in bisip_forward, y / yerr [n_spectra][2][N]
 * One data point per frequency j (its real and imaginary part are one measurement):
 *   ll[s][j] = -0.5 sum_{p in re, im} ((y[p][j] - Z[p][j](theta_s))^2 / yerr[p][j]^2 + 2 ln yerr[p][j]^2)
 * (sum_j ll[s][j] is the reference's _log_likelihood, models.py:59-62), and
 *   lppd_out[b][j] = logsumexp_s ll[s][j] - ln n_theta        p_out[b][j] = var_s(ll[s][j], ddof=1)
 *   elpd_out[b]    = sum_j (lppd - p)                          p_waic_out[b] = sum_j p
 *   se_out[b]      = sqrt(N var_j(lppd - p, ddof=1))           n_high_p_out[b] = #{j : p[j] > 0.4}  (int32)
 * Z is evaluated in FP64 for every desc->precision (the decomposition in its collapsed column form, as
 * bisip_model_percentile).  A NaN anywhere in a spectrum's samples makes all its outputs NaN (n_high_p 0).  One launch,
 * one CTA per spectrum; fixed-order reductions: a spectrum's result depends on its own chain and data only.  No
 * workspace and no limit on n_theta.
 * BISIP_ERR_BAD_ARG: null pointer, non-positive size, n_theta < 2, bad ndim / n_coef, w_stride or tau_stride < 0;
 * BISIP_ERR_UNSUPPORTED: n_spectra > 65535, n_coef > 32.
 */
int bisip_waic(const bisip_model_desc *desc, int n_spectra, int64_t n_theta, const double *theta,
               const double *w, int64_t w_stride, const double *taus, const double *log_taus, int64_t tau_stride,
               const double *y, const double *yerr,
               double *lppd_out, double *p_out, double *elpd_out, double *p_waic_out, double *se_out,
               int32_t *n_high_p_out, void *stream);

/*
 * PSIS-LOO: leave-one-out cross-validation by Pareto-smoothed importance sampling (Vehtari, Gelman & Gabry 2017;
 * Vehtari, Simpson, Gelman, Yao & Gabry 2024), with the Pareto shape k of every frequency, of every spectrum from its
 * chain, read in place.  Arguments as bisip_waic; ll[s][j] is bisip_waic's pointwise log-likelihood and S = n_theta.
 * For each frequency j, as ArviZ's psislw / _gpdfit / _gpinv with r_eff = 1:
 *   x_s = -ll[s][j] - max_s(-ll[s][j]);  M = ceil(min(0.2 S, 3 sqrt(S)));  cutoff = max((M+1)-th largest x, ln DBL_MIN)
 *   tail T = {s : x_s > cutoff}, L = |T|.  L <= 4: k = +inf, xt = x.  Otherwise (k, sigma) = the Zhang & Stephens
 *   generalized Pareto fit of the ascending exp(x_T) - exp(cutoff) (with the weakly informative prior on k); if k is
 *   finite the i-th smallest tail sample gets xt = ln(gpinv((i + 0.5) / L, k, sigma) + exp(cutoff)), then
 *   xt = min(xt, 0); otherwise xt = x.
 *   elpd_i_out[b][j] = logsumexp_s(xt + ll) - logsumexp_s(xt)     p_i_out[b][j] = lppd_j - elpd_i_out[b][j]
 *   k_out[b][j]      = k                                          (lppd_j = logsumexp_s ll - ln S)
 *   elpd_out[b]      = sum_j elpd_i                               p_loo_out[b] = sum_j p_i   (ascending j)
 *   se_out[b]        = sqrt(N var_j(elpd_i, ddof=1))              n_high_k_out[b] = #{j : k_j > min(1 - 1/log10 S, 0.7)}
 * Z is evaluated in FP64 for every desc->precision.  A NaN anywhere in a spectrum's samples makes all its outputs NaN
 * (n_high_k 0).  Two launches: one CTA per (frequency, spectrum), then one thread per spectrum for the totals; fixed-order
 * reductions: a spectrum's result depends on its own chain and data only.  No workspace.  A chain that fits one CTA's
 * shared memory (S up to about 25,900 on a B200) is evaluated there once; a longer one is re-evaluated per pass, with
 * only its Pareto tail (2M doubles) in shared memory.
 * BISIP_ERR_BAD_ARG: as bisip_waic;
 * BISIP_ERR_UNSUPPORTED: n_spectra > 65535, n_coef > 32, a tail that does not fit in shared memory (S above about 2e7).
 */
int bisip_psis_loo(const bisip_model_desc *desc, int n_spectra, int64_t n_theta, const double *theta,
                   const double *w, int64_t w_stride, const double *taus, const double *log_taus, int64_t tau_stride,
                   const double *y, const double *yerr,
                   double *elpd_i_out, double *p_i_out, double *k_out, double *elpd_out, double *p_loo_out,
                   double *se_out, int32_t *n_high_k_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BISIP_B200_H */
