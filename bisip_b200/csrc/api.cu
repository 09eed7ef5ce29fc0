// extern "C" boundary of libbisip_b200.so — see include/bisip_b200.h for the contract.  The kernels are launched by
// the per-family translation units (ens_*.cu, batch_*.cu; declared in launch.cuh); this file validates arguments,
// plans the launch and holds the statistics entry points.
#include <atomic>
#include <cstdio>
#include <cmath>
#include <string>

#include "launch.cuh"
#include "stats.cuh"
#include "model_pct.cuh"
#include "autocorr.cuh"
#include "rtd_stats.cuh"
#include "waic.cuh"
#include "loo.cuh"

namespace bisip {

static thread_local std::string g_err;
static std::atomic<long long> g_launches{0};

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
void count_launches(int n) { g_launches.fetch_add(n); }

}  // namespace bisip

using namespace bisip;

namespace {

// Start delay of the second co-resident CTA of ensemble_kernel (sampler.cuh, stagger_start): a quarter of one
// ensemble step, estimated from the tile count.
constexpr unsigned long long kStaggerNs = 6000ull;

// The kernels must run on the device that owns the caller's buffers, whatever device is current in the calling
// thread (one host thread may drive several GPUs): the entry points switch to the device of their primary pointer
// and restore the previous one on return.  A host pointer / unknown pointer leaves the current device alone.
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(const void* p) {
    cudaPointerAttributes at;
    if (p == nullptr || cudaPointerGetAttributes(&at, p) != cudaSuccess) { (void)cudaGetLastError(); return; }
    if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) return;
    if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; return; }
    if (at.device != prev) switched = (cudaSetDevice(at.device) == cudaSuccess);
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

int check_desc(const bisip_model_desc* d) {
  if (!d) return fail(BISIP_ERR_BAD_ARG, "desc is null");
  if (d->n_freq <= 0) return fail(BISIP_ERR_BAD_ARG, "n_freq must be positive");
  switch (d->model) {
    case BISIP_MODEL_COLECOLE:
      if (d->n_modes < 1 || d->n_modes > kMaxModes)
        return fail(BISIP_ERR_UNSUPPORTED, "ColeCole n_modes must be in [1,16]");
      if (d->ndim != 1 + 3 * d->n_modes) return fail(BISIP_ERR_BAD_ARG, "ColeCole ndim != 1+3*n_modes");
      break;
    case BISIP_MODEL_DIAS:
      if (d->ndim != 5) return fail(BISIP_ERR_BAD_ARG, "Dias2000 ndim != 5");
      break;
    case BISIP_MODEL_SHIN:
      if (d->ndim != 6) return fail(BISIP_ERR_BAD_ARG, "Shin2015 ndim != 6");
      break;
    case BISIP_MODEL_DECOMP:
      if (d->n_tau <= 0 || d->n_coef <= 0) return fail(BISIP_ERR_BAD_ARG, "Decomp n_tau/n_coef must be positive");
      if (d->ndim != 1 + d->n_coef) return fail(BISIP_ERR_BAD_ARG, "Decomp ndim != 1+n_coef");
      // poly_deg > 7: the two-stage tiles hold at most 8 coefficients; the FP64 precisions run the collapsed form
      // (same 1e-12 parity) up to 30 coefficients, the TF32 modes have no such kernel
      if (d->n_coef > 30) return fail(BISIP_ERR_UNSUPPORTED, "Decomp poly_deg > 29 not supported");
      if (d->n_coef > 8 && d->precision != BISIP_PREC_FP64 && d->precision != BISIP_PREC_FP64_COLLAPSED)
        return fail(BISIP_ERR_UNSUPPORTED, "Decomp poly_deg > 7 needs precision 'fp64' or 'fp64-collapsed'");
      if (d->precision < BISIP_PREC_FP64 || d->precision > BISIP_PREC_FP64_COLLAPSED)
        return fail(BISIP_ERR_BAD_ARG, "unknown precision");
      break;
    default:
      return fail(BISIP_ERR_BAD_ARG, "unknown model id");
  }
  return BISIP_OK;
}

__global__ void build_kernel_matrix(const double* w, int N, const double* taus, int S, double c_exp, double* K) {
  double cs, sn;
  sincospi(0.5 * c_exp, &sn, &cs);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S * N; i += gridDim.x * blockDim.x) {
    const int k = i / N, j = i - k * N;
    double kre, kim;
    debye_kernel_term(w[j], taus[k], c_exp, cs, sn, kre, kim);
    K[(size_t)k * 2 * N + j] = kre;
    K[(size_t)k * 2 * N + N + j] = kim;
  }
}

// Gaussian log-likelihood of n model rows Z[n][2N] supplied by the caller (a user forward callable evaluated on the host,
// models.py:59-62): one warp per row, lanes stride the 2N columns, fixed-order shuffle reduction.
__global__ void gauss_loglike_kernel(const double* __restrict__ Z, const double* __restrict__ y,
                                     const double* __restrict__ yerr, int C, int n, double* __restrict__ out) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  const double* z = Z + (size_t)row * C;
  double acc = 0.0;
  for (int c = lane; c < C; c += 32) {
    const double e = yerr[c], s2 = e * e, r = y[c] - z[c];
    acc += r * r / s2 + 2.0 * log(s2);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[row] = -0.5 * acc;
}

// bisip_psis_loo: loo_kernel of one model, the column in shared memory or recomputed per pass
template <int MODEL>
int launch_loo(const LooParams& P, bool smem_path, size_t smem, cudaStream_t st) {
  const dim3 grid(P.d.n_freq, P.B);
  return smem_path ? launch(loo_kernel<MODEL, true>, grid, smem, st, "psis_loo", &P, kStatThreads)
                   : launch(loo_kernel<MODEL, false>, grid, smem, st, "psis_loo", &P, kThreads);
}

}  // namespace

extern "C" {

int bisip_abi_version(void) { return BISIP_ABI_VERSION; }
const char* bisip_last_error(void) { return bisip::g_err.c_str(); }
int64_t bisip_launch_count(void) { return bisip::g_launches.load(); }

int bisip_decomp_kernel_kind(const bisip_model_desc* desc, int n_walkers) {
  if (int rc = check_desc(desc)) return rc;
  if (desc->model != BISIP_MODEL_DECOMP || n_walkers < 2) return fail(BISIP_ERR_BAD_ARG, "bisip_decomp_kernel_kind: bad argument");
  const size_t other = sampler_smem_bytes(n_walkers, desc->ndim);
  if (desc->precision == BISIP_PREC_FP64_COLLAPSED || desc->n_coef > 8) return BISIP_KERNEL_FP64_COLLAPSED;
  {
    const UmmaPlan up = plan_umma(*desc, other, (n_walkers + 1) / 2, true);
    if (up.ok) return up.cluster ? BISIP_KERNEL_TCGEN05_CLUSTER : BISIP_KERNEL_TCGEN05;
  }
  if (!use_rc(*desc)) return BISIP_KERNEL_DMMA;
  RcPlan plan;
  if (int rc = plan_rc(*desc, other, sampler_rows_pad(n_walkers), &plan)) return rc;
  return desc->precision == BISIP_PREC_FP64 ? BISIP_KERNEL_DMMA_CLUSTER : BISIP_KERNEL_MMA_TF32;
}

int bisip_n_keep(int nsteps, int discard, int thin) {
  if (thin < 1 || discard < 0) return 0;
  const int first = discard + thin - 1;
  return nsteps <= first ? 0 : (nsteps - first + thin - 1) / thin;
}

int bisip_forward(const bisip_model_desc* desc, int n_spectra, int n_theta, const double* theta, const double* w,
                  int64_t w_stride, const double* taus, const double* log_taus, int64_t tau_stride, double* Z,
                  void* stream) {
  if (int rc = check_desc(desc)) return rc;
  if (n_spectra <= 0 || n_theta <= 0 || !theta || !w || !Z) return fail(BISIP_ERR_BAD_ARG, "bisip_forward: bad argument");
  if (desc->model == BISIP_MODEL_DECOMP && (!taus || !log_taus)) return fail(BISIP_ERR_BAD_ARG, "bisip_forward: taus/log_taus null");
  if (n_spectra > 65535) return fail(BISIP_ERR_UNSUPPORTED, "bisip_forward: n_spectra > 65535 per call");
  DeviceGuard guard(theta);
  BatchParams P{*desc, n_spectra, n_theta, theta, w, w_stride, taus, log_taus, tau_stride, nullptr, nullptr, nullptr, Z, nullptr};
  return desc->model == BISIP_MODEL_DECOMP ? run_batch_decomp(P, true, (cudaStream_t)stream)
                                           : run_batch_vec(P, true, (cudaStream_t)stream);
}

int bisip_log_probability(const bisip_model_desc* desc, int n_spectra, int n_theta, const double* theta,
                          const double* w, int64_t w_stride, const double* taus, const double* log_taus,
                          int64_t tau_stride, const double* y, const double* yerr, const double* bounds,
                          double* lp_out, void* stream) {
  if (int rc = check_desc(desc)) return rc;
  if (n_spectra <= 0 || n_theta <= 0 || !theta || !w || !y || !yerr || !bounds || !lp_out)
    return fail(BISIP_ERR_BAD_ARG, "bisip_log_probability: bad argument");
  if (desc->model == BISIP_MODEL_DECOMP && (!taus || !log_taus)) return fail(BISIP_ERR_BAD_ARG, "bisip_log_probability: taus/log_taus null");
  if (n_spectra > 65535) return fail(BISIP_ERR_UNSUPPORTED, "bisip_log_probability: n_spectra > 65535 per call");
  DeviceGuard guard(theta);
  BatchParams P{*desc, n_spectra, n_theta, theta, w, w_stride, taus, log_taus, tau_stride, y, yerr, bounds, nullptr, lp_out};
  return desc->model == BISIP_MODEL_DECOMP ? run_batch_decomp(P, false, (cudaStream_t)stream)
                                           : run_batch_vec(P, false, (cudaStream_t)stream);
}

int bisip_decomp_build_kernel(const double* w, int n_freq, const double* taus, int n_tau, double c_exp, double* K,
                              void* stream) {
  if (!w || !taus || !K || n_freq <= 0 || n_tau <= 0) return fail(BISIP_ERR_BAD_ARG, "bisip_decomp_build_kernel: bad argument");
  DeviceGuard guard(K);
  build_kernel_matrix<<<ceil_div(n_freq * n_tau, 256), 256, 0, (cudaStream_t)stream>>>(w, n_freq, taus, n_tau, c_exp, K);
  BISIP_CUDA(cudaGetLastError());
  count_launches(1);
  return BISIP_OK;
}

int bisip_gauss_loglike(const double* Z, const double* y, const double* yerr, int n_freq, int n_rows, double* ll_out,
                        void* stream) {
  if (!Z || !y || !yerr || !ll_out || n_freq <= 0 || n_rows <= 0) return fail(BISIP_ERR_BAD_ARG, "bisip_gauss_loglike: bad argument");
  DeviceGuard guard(Z);
  gauss_loglike_kernel<<<ceil_div(n_rows, 4), 128, 0, (cudaStream_t)stream>>>(Z, y, yerr, 2 * n_freq, n_rows, ll_out);
  BISIP_CUDA(cudaGetLastError());
  count_launches(1);
  return BISIP_OK;
}

int bisip_ensemble_run(const bisip_model_desc* desc, int n_spectra, int n_walkers, int nsteps, int step0,
                       uint64_t seed, uint32_t spectrum0, double a, int discard, int thin, const double* w,
                       int64_t w_stride, const double* taus, const double* log_taus, int64_t tau_stride,
                       const double* y, const double* yerr, const double* bounds, double* coords, double* lp,
                       double* chain, double* logp, int32_t* accepted, int32_t* flags, void* stream) {
  if (int rc = check_desc(desc)) return rc;
  if (n_spectra <= 0 || n_walkers < 2 || nsteps < 0 || thin < 1 || discard < 0 || !w || !y || !yerr || !bounds || !coords)
    return fail(BISIP_ERR_BAD_ARG, "bisip_ensemble_run: bad argument");
  if (desc->model == BISIP_MODEL_DECOMP && (!taus || !log_taus)) return fail(BISIP_ERR_BAD_ARG, "bisip_ensemble_run: taus/log_taus null");
  if (!(a > 1.0)) return fail(BISIP_ERR_BAD_ARG, "bisip_ensemble_run: stretch scale a must be > 1");
  DeviceGuard guard(coords);
  cudaStream_t st = (cudaStream_t)stream;
  EnsembleParams P;
  P.d = *desc; P.B = n_spectra; P.W = n_walkers; P.nsteps = nsteps; P.step0 = step0; P.seed = seed;
  P.spectrum0 = spectrum0; P.a = a; P.discard = discard; P.thin = thin;
  P.nkeep = bisip_n_keep(nsteps, discard, thin);
  P.w = w; P.w_stride = w_stride; P.taus = taus; P.log_taus = log_taus; P.tau_stride = tau_stride;
  P.y = y; P.yerr = yerr; P.bounds = bounds; P.coords = coords; P.lp = lp; P.chain = chain; P.logp = logp;
  P.accepted = accepted; P.flags = flags;
  {
    uint32_t km = 1;
    while ((int)km < n_walkers) km <<= 1;
    P.kmask = km - 1;
    int ex;
    P.a_pow2 = (frexp(a, &ex) == 0.5) ? 1 : 0;
    P.inv_a = 1.0 / a;
  }
  P.stagger_ns = kStaggerNs;
  if (flags) BISIP_CUDA(cudaMemsetAsync(flags, 0, sizeof(int32_t) * (size_t)n_spectra, st));
  const int rp = sampler_rows_pad(n_walkers);
  size_t smem = sampler_smem_bytes(n_walkers, desc->ndim);
  dim3 grid(n_spectra);
  // Warp-private sampler (sampler_wp.cuh) for the evaluators that have a warp-level form, up to 256 walkers; both
  // kernels follow the same stream.
  const bool big_poly = desc->model == BISIP_MODEL_DECOMP && desc->n_coef > 8;     // FP64 on the collapsed tiles only
  if (big_poly && n_walkers > 256)
    return fail(BISIP_ERR_UNSUPPORTED, "Decomp poly_deg > 7 is sampled by the warp-private kernel: at most 256 walkers");
  if (n_walkers <= 256) {
    if (desc->model == BISIP_MODEL_DECOMP && (desc->precision == BISIP_PREC_FP64_COLLAPSED || big_poly))
      return launch_ens_wp_collapsed(P, grid, st);
    if (desc->model == BISIP_MODEL_DECOMP && desc->precision == BISIP_PREC_FP64 && desc->n_tau > 32 && desc->n_tau <= 64)
      return launch_ens_wp_dmma(P, grid, st);
    // measured (profiles/r02_wp_sweep.md, r02c_vec_analysis.md): warp-private wins by 1.2-2x for <= 64 walkers or short
    // spectra and for 1-mode Cole-Cole everywhere; for Dias / Shin / 2-mode Cole-Cole with > 64 walkers and > 32
    // frequencies the block-synchronous kernel is 2-7 % faster (its serial phases run on full warps; the long frequency
    // loop dominates either way).
    const bool long_vec = n_walkers > 64 && desc->n_freq > 32;
    const bool wp_vec = desc->model == BISIP_MODEL_DIAS || desc->model == BISIP_MODEL_SHIN
                            ? !long_vec
                            : desc->model == BISIP_MODEL_COLECOLE && (desc->n_modes == 1 || (desc->n_modes == 2 && !long_vec));
    if (wp_vec)
      return launch_ens_wp_vec(P, grid, st);
  }
  switch (desc->model) {
    case BISIP_MODEL_COLECOLE:
      smem += vec_smem_doubles(desc->n_freq, rp, vec_row_consts(*desc)) * 8;
      return launch_ens_colecole(P, grid, smem, st);
    case BISIP_MODEL_DIAS:
      smem += VecEvaluator<DiasRow>::smem_doubles(*desc, rp) * 8;
      return launch_ens_dias_shin(P, grid, smem, st);
    case BISIP_MODEL_SHIN:
      smem += VecEvaluator<ShinRow>::smem_doubles(*desc, rp) * 8;
      return launch_ens_dias_shin(P, grid, smem, st);
    default: {
      if (desc->precision == BISIP_PREC_FP64_COLLAPSED) {
        smem += DecompCollapsedEvaluator::smem_doubles(*desc, rp) * 8;
        return launch_ens_collapsed(P, grid, smem, st);
      }
      {
        const UmmaPlan up = plan_umma(*desc, smem, (n_walkers + 1) / 2, true);
        if (up.ok && up.cluster) {
          if ((long long)n_spectra * 2 > 2147483647LL) return fail(BISIP_ERR_UNSUPPORTED, "too many spectra per call");
          return launch_ens_umma(P, dim3(n_spectra * 2), up, st);
        }
        if (up.ok) return launch_ens_umma(P, grid, up, st);
      }
      if (use_rc(*desc)) {
        RcPlan plan;
        if (int rc = plan_rc(*desc, smem, rp, &plan)) return rc;
        if ((long long)n_spectra * plan.cs > 2147483647LL) return fail(BISIP_ERR_UNSUPPORTED, "too many spectra per call");
        return launch_ens_rc(P, dim3(n_spectra * plan.cs), plan, st);
      }
      smem += DecompEvaluator<4>::smem_doubles(*desc, rp) * 8;
      return launch_ens_dmma(P, grid, smem, st);
    }
  }
}

int64_t bisip_column_stats_workspace(int, int64_t, int) { return 0; }   // ABI 1 needed a key workspace; the chain is now read in place

// launch one of the shared-memory statistics kernels if (n, R) fits in one CTA's shared memory, else report "does not fit"
static bool stats_fits_smem(int64_t n, int R, size_t* smem) {
  *smem = stats_smem_bytes(n, R);
  return n <= 0x7fffffff / 8 && *smem + kStatStaticSmem <= (size_t)device_smem_optin();
}

int bisip_column_stats(const double* data, int n_spectra, int64_t n_samples, int n_cols, int n_pct,
                       const int64_t* pct_lo, const double* pct_gamma, double* pct_out, double* mean_out,
                       double* std_out, void* /*workspace*/, int64_t /*workspace_bytes*/, void* stream) {
  if (!data || n_spectra <= 0 || n_samples <= 0 || n_cols <= 0 || n_pct < 0)
    return fail(BISIP_ERR_BAD_ARG, "bisip_column_stats: bad argument");
  if (n_pct > kMaxPct) return fail(BISIP_ERR_UNSUPPORTED, "bisip_column_stats: at most 16 percentiles per call");
  if (n_pct > 0 && (!pct_lo || !pct_gamma || !pct_out)) return fail(BISIP_ERR_BAD_ARG, "bisip_column_stats: percentile arrays null");
  if (n_spectra > 65535) return fail(BISIP_ERR_UNSUPPORTED, "bisip_column_stats: n_spectra > 65535 per call");
  DeviceGuard guard(data);
  cudaStream_t st = (cudaStream_t)stream;
  StatsParams P;
  P.data = data; P.n = n_samples; P.ncol = n_cols; P.B = n_spectra;
  P.npct = n_pct;
  for (int i = 0; i < n_pct; ++i) { P.lo[i] = pct_lo[i]; P.gamma[i] = pct_gamma[i]; }
  P.pct_out = pct_out; P.mean_out = mean_out; P.std_out = std_out;
  const dim3 grid(n_cols, n_spectra);
  size_t smem = 0;
  if (stats_fits_smem(n_samples, 2 * n_pct, &smem))
    return launch(column_stats_smem_kernel, grid, smem, st, "column_stats", &P, kStatThreads);
  column_stats_global_kernel<<<grid, kThreads, 0, st>>>(P);
  BISIP_CUDA(cudaGetLastError());
  count_launches(1);
  return BISIP_OK;
}

// model description of the kernels built on model_points (model_pct.cuh): the decomposition runs its collapsed FP64
// column form for every precision, and the loops over modes / coefficients do not have the sampler kernels' tile limits
static int check_point_desc(const bisip_model_desc* desc, bisip_model_desc* out, const char* name) {
  if (!desc) return fail(BISIP_ERR_BAD_ARG, "desc is null");
  bisip_model_desc d = *desc;
  if (d.model == BISIP_MODEL_DECOMP) d.precision = BISIP_PREC_FP64_COLLAPSED;   // the column form; FP64 for every mode
  bisip_model_desc chk = d;
  if (chk.model == BISIP_MODEL_COLECOLE && chk.n_modes > kMaxModes) { chk.n_modes = 1; chk.ndim = 4; }
  if (chk.model == BISIP_MODEL_DECOMP && chk.n_coef > 8) { chk.n_coef = 8; chk.ndim = 9; chk.precision = BISIP_PREC_FP64; }
  if (int rc = check_desc(&chk)) return rc;
  if (d.model == BISIP_MODEL_COLECOLE && (d.n_modes < 1 || d.ndim != 1 + 3 * d.n_modes))
    return fail(BISIP_ERR_BAD_ARG, "ColeCole ndim != 1+3*n_modes");
  if (d.model == BISIP_MODEL_DECOMP && (d.ndim != 1 + d.n_coef || d.n_coef > kMaxCoefPct))
    return fail(d.n_coef > kMaxCoefPct ? BISIP_ERR_UNSUPPORTED : BISIP_ERR_BAD_ARG, std::string(name) + ": bad n_coef");
  *out = d;
  return BISIP_OK;
}

int bisip_model_percentile(const bisip_model_desc* desc, int n_spectra, int64_t n_theta, const double* theta,
                           const double* w, int64_t w_stride, const double* taus, const double* log_taus,
                           int64_t tau_stride, int n_pct, const int64_t* pct_lo, const double* pct_gamma,
                           double* pct_out, void* stream) {
  bisip_model_desc d;
  if (int rc = check_point_desc(desc, &d, "bisip_model_percentile")) return rc;
  if (n_spectra <= 0 || n_theta <= 0 || !theta || !w || n_pct <= 0 || !pct_lo || !pct_gamma || !pct_out)
    return fail(BISIP_ERR_BAD_ARG, "bisip_model_percentile: bad argument");
  if (d.model == BISIP_MODEL_DECOMP && (!taus || !log_taus)) return fail(BISIP_ERR_BAD_ARG, "bisip_model_percentile: taus/log_taus null");
  if (n_pct > kMaxPct) return fail(BISIP_ERR_UNSUPPORTED, "bisip_model_percentile: at most 16 percentiles per call");
  if (n_spectra > 65535) return fail(BISIP_ERR_UNSUPPORTED, "bisip_model_percentile: n_spectra > 65535 per call");
  DeviceGuard guard(theta);
  size_t smem = 0;
  if (!stats_fits_smem(n_theta, 2 * n_pct, &smem))
    return fail(BISIP_ERR_UNSUPPORTED, "bisip_model_percentile: chain too long for one CTA's shared memory "
                                       "(use bisip_forward + bisip_column_stats)");
  ModelPctParams P;
  P.d = d; P.B = n_spectra; P.n = n_theta; P.theta = theta; P.w = w; P.w_stride = w_stride;
  P.taus = taus; P.log_taus = log_taus; P.tau_stride = tau_stride;
  P.st.data = nullptr; P.st.n = n_theta; P.st.ncol = 2 * d.n_freq; P.st.B = n_spectra; P.st.npct = n_pct;
  for (int i = 0; i < n_pct; ++i) { P.st.lo[i] = pct_lo[i]; P.st.gamma[i] = pct_gamma[i]; }
  P.st.pct_out = pct_out; P.st.mean_out = nullptr; P.st.std_out = nullptr;
  return launch(model_percentile_kernel, dim3(2 * d.n_freq, n_spectra), smem, (cudaStream_t)stream, "model_percentile", &P,
                kStatThreads);
}

int bisip_autocorr_time(const double* data, int n_spectra, int n_keep, int n_walkers, int n_cols, double c,
                        double* tau_out, void* stream) {
  if (!data || !tau_out || n_spectra <= 0 || n_keep <= 0 || n_walkers <= 0 || n_cols <= 0)
    return fail(BISIP_ERR_BAD_ARG, "bisip_autocorr_time: bad argument");
  if (!std::isfinite(c) || !(c > 0.0)) return fail(BISIP_ERR_BAD_ARG, "bisip_autocorr_time: c must be finite and > 0");
  if (n_spectra > 65535) return fail(BISIP_ERR_UNSUPPORTED, "bisip_autocorr_time: n_spectra > 65535 per call");
  DeviceGuard guard(data);
  AutocorrParams P;
  P.data = data; P.B = n_spectra; P.n = n_keep; P.W = n_walkers; P.ncol = n_cols; P.c = c; P.tau_out = tau_out;
  const dim3 grid(n_cols, n_spectra);
  // the column in shared memory when it fits (the same test as the statistics kernels), else strided global reads
  const long long nw = (long long)n_keep * n_walkers;
  const size_t smem = autocorr_smem_bytes(n_keep, n_walkers, true);
  const int optin = device_smem_optin();
  if (nw <= 0x7fffffff / 8 && smem + kAcfStaticSmem <= (size_t)optin)
    return launch(autocorr_kernel<true>, grid, smem, (cudaStream_t)stream, "autocorr_time", &P, kAcfThreads);
  const size_t gsmem = autocorr_smem_bytes(0, n_walkers, false);
  if (gsmem + kAcfStaticSmem > (size_t)optin)
    return fail(BISIP_ERR_UNSUPPORTED, "bisip_autocorr_time: too many walkers for one CTA's shared memory");
  return launch(autocorr_kernel<false>, grid, gsmem, (cudaStream_t)stream, "autocorr_time", &P, kAcfThreads);
}

int bisip_rtd_stats(int n_spectra, int64_t n_samples, int ndim, int n_coef, int n_tau, const double* theta,
                    const double* log_taus, int64_t tau_stride, int n_pct, const int64_t* pct_lo, const double* pct_gamma,
                    double* pct_out, double* mean_out, double* std_out, void* stream) {
  if (!theta || !log_taus || n_spectra <= 0 || n_samples <= 0 || ndim <= 0 || n_coef <= 0 || n_tau <= 0 ||
      tau_stride < 0 || n_pct < 0)
    return fail(BISIP_ERR_BAD_ARG, "bisip_rtd_stats: bad argument");
  if (n_coef > kMaxCoefPct) return fail(BISIP_ERR_UNSUPPORTED, "bisip_rtd_stats: n_coef > 32");
  if (ndim != 1 + n_coef) return fail(BISIP_ERR_BAD_ARG, "bisip_rtd_stats: ndim != 1 + n_coef");
  if (n_pct > 0 && (!pct_lo || !pct_gamma || !pct_out))
    return fail(BISIP_ERR_BAD_ARG, "bisip_rtd_stats: percentile arrays null");
  if (n_pct == 0 && !mean_out && !std_out) return fail(BISIP_ERR_BAD_ARG, "bisip_rtd_stats: no output requested");
  if (n_pct > kMaxPct) return fail(BISIP_ERR_UNSUPPORTED, "bisip_rtd_stats: at most 16 percentiles per call");
  if (n_spectra > 65535) return fail(BISIP_ERR_UNSUPPORTED, "bisip_rtd_stats: n_spectra > 65535 per call");
  if (n_tau > 0x7ffffffe) return fail(BISIP_ERR_UNSUPPORTED, "bisip_rtd_stats: n_tau + 1 columns exceed the grid");
  DeviceGuard guard(theta);
  RtdParams P;
  P.theta = theta; P.log_taus = log_taus; P.tau_stride = tau_stride;
  P.ndim = ndim; P.n_coef = n_coef; P.n_tau = n_tau;
  P.st.data = nullptr; P.st.n = n_samples; P.st.ncol = n_tau + 1; P.st.B = n_spectra; P.st.npct = n_pct;
  for (int i = 0; i < n_pct; ++i) { P.st.lo[i] = pct_lo[i]; P.st.gamma[i] = pct_gamma[i]; }
  P.st.pct_out = n_pct ? pct_out : nullptr; P.st.mean_out = mean_out; P.st.std_out = std_out;
  const dim3 grid(n_tau + 1, n_spectra);
  size_t smem = 0;
  if (stats_fits_smem(n_samples, 2 * n_pct, &smem))
    return launch(rtd_stats_smem_kernel, grid, smem, (cudaStream_t)stream, "rtd_stats", &P, kStatThreads);
  return launch(rtd_stats_global_kernel, grid, 0, (cudaStream_t)stream, "rtd_stats", &P, kThreads);
}

int bisip_waic(const bisip_model_desc* desc, int n_spectra, int64_t n_theta, const double* theta, const double* w,
               int64_t w_stride, const double* taus, const double* log_taus, int64_t tau_stride, const double* y,
               const double* yerr, double* lppd_out, double* p_out, double* elpd_out, double* p_waic_out,
               double* se_out, int32_t* n_high_p_out, void* stream) {
  bisip_model_desc d;
  if (int rc = check_point_desc(desc, &d, "bisip_waic")) return rc;
  if (n_spectra <= 0 || n_theta < 2 || !theta || !w || w_stride < 0 || tau_stride < 0 || !y || !yerr || !lppd_out ||
      !p_out || !elpd_out || !p_waic_out || !se_out || !n_high_p_out)
    return fail(BISIP_ERR_BAD_ARG, "bisip_waic: bad argument");
  if (d.model == BISIP_MODEL_DECOMP && (!taus || !log_taus)) return fail(BISIP_ERR_BAD_ARG, "bisip_waic: taus/log_taus null");
  if (n_spectra > 65535) return fail(BISIP_ERR_UNSUPPORTED, "bisip_waic: n_spectra > 65535 per call");
  DeviceGuard guard(theta);
  WaicParams P;
  P.d = d; P.n = n_theta; P.theta = theta; P.w = w; P.w_stride = w_stride;
  P.taus = taus; P.log_taus = log_taus; P.tau_stride = tau_stride; P.y = y; P.yerr = yerr;
  P.lppd_out = lppd_out; P.p_out = p_out; P.elpd_out = elpd_out; P.p_waic_out = p_waic_out; P.se_out = se_out;
  P.n_high_p_out = n_high_p_out;
  const dim3 grid(n_spectra);
  const cudaStream_t st = (cudaStream_t)stream;
  switch (d.model) {
    case BISIP_MODEL_DECOMP: return launch(waic_kernel<BISIP_MODEL_DECOMP>, grid, 0, st, "waic", &P, kWaicThreads);
    case BISIP_MODEL_COLECOLE: return launch(waic_kernel<BISIP_MODEL_COLECOLE>, grid, 0, st, "waic", &P, kWaicThreads);
    case BISIP_MODEL_DIAS: return launch(waic_kernel<BISIP_MODEL_DIAS>, grid, 0, st, "waic", &P, kWaicThreads);
    default: return launch(waic_kernel<BISIP_MODEL_SHIN>, grid, 0, st, "waic", &P, kWaicThreads);
  }
}

int bisip_psis_loo(const bisip_model_desc* desc, int n_spectra, int64_t n_theta, const double* theta, const double* w,
                   int64_t w_stride, const double* taus, const double* log_taus, int64_t tau_stride, const double* y,
                   const double* yerr, double* elpd_i_out, double* p_i_out, double* k_out, double* elpd_out,
                   double* p_loo_out, double* se_out, int32_t* n_high_k_out, void* stream) {
  bisip_model_desc d;
  if (int rc = check_point_desc(desc, &d, "bisip_psis_loo")) return rc;
  if (n_spectra <= 0 || n_theta < 2 || !theta || !w || w_stride < 0 || tau_stride < 0 || !y || !yerr || !elpd_i_out ||
      !p_i_out || !k_out || !elpd_out || !p_loo_out || !se_out || !n_high_k_out)
    return fail(BISIP_ERR_BAD_ARG, "bisip_psis_loo: bad argument");
  if (d.model == BISIP_MODEL_DECOMP && (!taus || !log_taus)) return fail(BISIP_ERR_BAD_ARG, "bisip_psis_loo: taus/log_taus null");
  if (n_spectra > 65535) return fail(BISIP_ERR_UNSUPPORTED, "bisip_psis_loo: n_spectra > 65535 per call");
  DeviceGuard guard(theta);
  const size_t optin = (size_t)device_smem_optin();
  // the ll column in shared memory when it fits, else recomputed per pass with only the tail buffer in shared memory
  size_t smem = loo_smem_bytes(n_theta);
  const bool smem_path = n_theta <= 0x7fffffff / 8 && smem + kStatStaticSmem <= optin;
  if (!smem_path) {
    smem = std::max(loo_tail_bytes(n_theta), (size_t)256 * 4);   // and the radix select's histogram before it
    if (smem + kStatStaticSmem > optin)
      return fail(BISIP_ERR_UNSUPPORTED, "bisip_psis_loo: the Pareto tail of the chain does not fit in shared memory");
  }
  LooParams P;
  P.d = d; P.n = n_theta; P.B = n_spectra; P.theta = theta; P.w = w; P.w_stride = w_stride;
  P.taus = taus; P.log_taus = log_taus; P.tau_stride = tau_stride; P.y = y; P.yerr = yerr;
  P.elpd_i_out = elpd_i_out; P.p_i_out = p_i_out; P.k_out = k_out;
  P.elpd_out = elpd_out; P.p_loo_out = p_loo_out; P.se_out = se_out; P.n_high_k_out = n_high_k_out;
  const cudaStream_t st = (cudaStream_t)stream;
  int rc;
  switch (d.model) {
    case BISIP_MODEL_DECOMP: rc = launch_loo<BISIP_MODEL_DECOMP>(P, smem_path, smem, st); break;
    case BISIP_MODEL_COLECOLE: rc = launch_loo<BISIP_MODEL_COLECOLE>(P, smem_path, smem, st); break;
    case BISIP_MODEL_DIAS: rc = launch_loo<BISIP_MODEL_DIAS>(P, smem_path, smem, st); break;
    default: rc = launch_loo<BISIP_MODEL_SHIN>(P, smem_path, smem, st); break;
  }
  if (rc) return rc;
  return launch(loo_totals_kernel, dim3((n_spectra + 127) / 128), 0, st, "psis_loo_totals", &P, 128);
}

}  // extern "C"
