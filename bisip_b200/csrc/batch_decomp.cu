// Batched forward / log-probability of the polynomial decomposition (same evaluators as the sampler).
#include "batch.cuh"

namespace bisip {

// More than 8 polynomial coefficients (poly_deg > 7): none of the evaluators' tile shapes holds the stage-1 operand.  The
// forward is evaluated in its collapsed FP64 form Z_c = R0 (delta_c - sum_i a_i G_ic), G = L K accumulated once per CTA
// in compensated (Dot2) arithmetic like decomp_c_init — plain loops, any n_coef <= 30: this is the API path of
// forward() / _log_probability() for large polynomials, not a sampled path.  Grid (rows, B): CTA (r, b) handles theta
// rows r, r + gridDim.x, ... of spectrum b.
constexpr int kBigD = 30;
template <bool WANT_Z>
__global__ void __launch_bounds__(kThreads) decomp_big_batch_kernel(const BatchParams P) {
  extern __shared__ __align__(16) double smem[];
  __shared__ double red[kWarps];
  const int b = blockIdx.y, ndim = P.d.ndim, N = P.d.n_freq, D = P.d.n_coef, S = P.d.n_tau, C = 2 * N;
  double* G = smem;                    // [C][D]   (scaled by 1/sigma_c in likelihood mode)
  double* ys = G + (size_t)C * D;      // [C] y/sigma
  double* ds = ys + C;                 // [C] delta/sigma
  const double* w = P.w + (size_t)b * P.w_stride;
  const double* taus = P.taus + (size_t)b * P.tau_stride;
  const double* lts = P.log_taus + (size_t)b * P.tau_stride * D;
  const double* y = WANT_Z ? nullptr : P.y + (size_t)b * 2 * N;
  const double* yerr = WANT_Z ? nullptr : P.yerr + (size_t)b * 2 * N;
  double csum = 0.0;
  for (int c = threadIdx.x; c < C; c += kThreads) {
    const double is = WANT_Z ? 1.0 : 1.0 / yerr[c];
    ys[c] = WANT_Z ? 0.0 : y[c] * is;
    ds[c] = c < N ? is : 0.0;
    if (!WANT_Z) csum += 2.0 * log(yerr[c] * yerr[c]);
  }
  double cs, sn;
  sincospi(0.5 * P.d.c_exp, &sn, &cs);
  for (int idx = threadIdx.x; idx < C * D; idx += kThreads) {
    const int c = idx / D, i = idx - c * D;
    const int j = c < N ? c : c - N;
    const double is = WANT_Z ? 1.0 : 1.0 / yerr[c];
    G[idx] = dot2_lk(lts + (size_t)i * S, taus, S, w[j], P.d.c_exp, cs, sn, c >= N, is);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) csum += __shfl_xor_sync(0xffffffffu, csum, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = csum;
  __syncthreads();
  double llc = 0.0;
  for (int i = 0; i < kWarps; ++i) llc += red[i];
  for (int r0 = blockIdx.x; r0 < P.n_theta; r0 += gridDim.x) {      // one theta row per CTA pass, threads over columns
    const double* th = P.theta + ((size_t)b * P.n_theta + r0) * ndim;
    const double R0 = th[0];
    double chi = 0.0;
    for (int c = threadIdx.x; c < C; c += kThreads) {
      const double* g = G + (size_t)c * D;
      double acc = 0.0;
      for (int i = 0; i < D; ++i) acc = fma(R0 * th[1 + i], g[i], acc);
      if (WANT_Z) {
        P.Z[((size_t)b * P.n_theta + r0) * C + c] = R0 * ds[c] - acc;
      } else {
        const double r = fma(-R0, ds[c], ys[c]) + acc;
        chi = fma(r, r, chi);
      }
    }
    if (!WANT_Z) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) chi += __shfl_xor_sync(0xffffffffu, chi, o);
      __syncthreads();
      if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = chi;
      __syncthreads();
      if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int i = 0; i < kWarps; ++i) tot += red[i];
        bool ok = true;
        for (int d = 0; d < ndim; ++d) ok = ok && (P.bounds[d] < th[d]) && (th[d] < P.bounds[ndim + d]);
        P.lp[(size_t)b * P.n_theta + r0] = ok ? -0.5 * (tot + llc) : neg_inf();
      }
    }
  }
}

template <bool WANT_Z>
static int run_batch_decomp_t(const BatchParams& P, cudaStream_t st) {
  if (P.d.n_coef > 8) {
    if (P.d.n_coef > kBigD) return fail(BISIP_ERR_UNSUPPORTED, "Decomp poly_deg > 29 not supported");
    const size_t smem = ((size_t)2 * P.d.n_freq * (P.d.n_coef + 2)) * 8;
    const int rows = max(1, min(P.n_theta, device_sm_count() * 8 / max(1, P.B)));
    return launch(decomp_big_batch_kernel<WANT_Z>, dim3(rows, P.B), smem, st, "decomp_big_batch", &P);
  }
  const size_t other = batch_other_bytes(P.d);
  const UmmaPlan up = plan_umma(P.d, other, kRows);
  if (up.ok) {
    if (prec_planes(P.d.precision) == 3)
      return launch_batch<DecompUmmaEvaluator<3>, WANT_Z>(P, 2, up.smem, st, "decomp_umma_3xtf32_batch");
    return launch_batch<DecompUmmaEvaluator<1>, WANT_Z>(P, 2, up.smem, st, "decomp_umma_tf32_batch");
  }
  if (P.d.precision == BISIP_PREC_FP64_COLLAPSED)
    return launch_batch<DecompCollapsedEvaluator, WANT_Z>(P, 4, batch_smem<DecompCollapsedEvaluator>(P.d), st,
                                                          "decomp_collapsed_batch");
  if (use_rc(P.d)) {
    RcPlan plan;
    if (int rc = plan_rc(P.d, other, kRows, &plan)) return rc;
    switch (prec_planes(P.d.precision)) {
      case 1: return launch_batch<DecompTF32Evaluator<1>, WANT_Z>(P, 2, plan.smem, st, "decomp_tf32_batch", plan.cs);
      case 3: return launch_batch<DecompTF32Evaluator<3>, WANT_Z>(P, 2, plan.smem, st, "decomp_3xtf32_batch", plan.cs);
      default: return launch_batch<DecompRCEvaluator, WANT_Z>(P, 2, plan.smem, st, "decomp_rc_batch", plan.cs);
    }
  }
  const size_t smem = batch_smem<DecompEvaluator<1>>(P.d);     // the same for every KC
  switch (ceil_div(P.d.n_tau, 16)) {
    case 1: return launch_batch<DecompEvaluator<1>, WANT_Z>(P, 8, smem, st, "decomp_batch");
    case 2: return launch_batch<DecompEvaluator<2>, WANT_Z>(P, 8, smem, st, "decomp_batch");
    case 3: return launch_batch<DecompEvaluator<3>, WANT_Z>(P, 8, smem, st, "decomp_batch");
    default: return launch_batch<DecompEvaluator<4>, WANT_Z>(P, 8, smem, st, "decomp_batch");
  }
}

int run_batch_decomp(const BatchParams& P, bool want_z, cudaStream_t st) {
  return want_z ? run_batch_decomp_t<true>(P, st) : run_batch_decomp_t<false>(P, st);
}

}  // namespace bisip
