// Percentiles of the forward model over a chain, fused: bisip_model_percentile.
//
// Replaces utils.get_model_percentile (reference utils.py:17-35): a Python loop of one forward() per flat-chain sample
// into a (n, 2, N) array, then np.percentile over axis 0.  Here one CTA owns one of the 2N model columns (real or
// imaginary part at one frequency) of one spectrum: it evaluates that column for all n parameter vectors straight into
// shared memory and selects the order statistics there (stats.cuh), so the (n, 2N) model matrix is never written to
// HBM: traffic is n * ndim * 8 bytes in (L2-resident across the 2N CTAs of a spectrum) and n_pct * 2N * 8 bytes out.
//   * Cole-Cole / Dias / Shin: the same expressions as the batched forward kernels (models.cuh, FAST = false); the
//     column values agree with bisip_forward's to the last bit or two (FMA contraction is the compiler's choice).
//   * Polynomial decomposition: a single column of Z = R0 (delta - sum_k M_k K_kc) is the collapsed form
//     z_c = sum_i (R0 a_i) G_ic with G_ic = sum_k L_ik K_kc accumulated once per CTA in compensated (Dot2) arithmetic
//     (decomp_collapsed.cuh) — FP64 for every `precision`, within 1e-12 of the two-stage forward.
#pragma once
#include "common.cuh"
#include "decomp_collapsed.cuh"
#include "models.cuh"
#include "stats.cuh"

namespace bisip {

struct ModelPctParams {
  bisip_model_desc d;
  int B;
  long long n;                      // parameter vectors per spectrum
  const double* theta;              // [B][n][ndim]
  const double* w; long long w_stride;
  const double* taus; const double* log_taus; long long tau_stride;
  StatsParams st;                   // lo / gamma / npct ; pct_out = [B][npct][2N]
};

constexpr int kMaxCoefPct = 32;     // decomposition coefficients (poly_deg + 1) this kernel holds

// one Cole-Cole column value (any number of modes), expression by expression ColeColeRowT::prepare + eval<false>
__device__ __forceinline__ void colecole_point(const double* __restrict__ th, int K, double lnw, double& zre, double& zim) {
  const double R0 = th[0];
  double sre = 0.0, sim = 0.0;
  for (int i = 0; i < K; ++i) {
    const double ci = th[1 + 2 * K + i];
    double sn_, cs_;
    sincospi(0.5 * ci, &sn_, &cs_);
    const double x = exp(ci * (lnw + th[1 + K + i]));
    const double u = x * cs_, v = x * sn_;
    const double d1 = 1.0 + u;
    const double den = d1 * d1 + v * v;
    const double mi = th[1 + i] / den;
    sre = fma(mi, u + x * x, sre);
    sim = fma(mi, v, sim);
  }
  zre = R0 * (1.0 - sre);
  zim = -R0 * sim;
}

// grid (2N, B), kStatThreads threads, dynamic shared memory stats_smem_bytes(n, 2 npct)
__global__ void __launch_bounds__(kStatThreads, 1) model_percentile_kernel(const ModelPctParams P) {
  extern __shared__ __align__(16) unsigned char stats_dyn[];
  __shared__ double red[32];
  __shared__ double s_g[kMaxCoefPct];
  __shared__ __align__(16) double s_fq[kFq];
  constexpr int NT = kStatThreads;
  const int c = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int N = P.d.n_freq, ndim = P.d.ndim;
  const int j = c < N ? c : c - N;
  const bool imag = c >= N;
  const int n = (int)P.n;
  double* vals = reinterpret_cast<double*>(stats_dyn);
  double* pool = vals + n;
  unsigned int* hist = reinterpret_cast<unsigned int*>(pool + kStatPool);
  const double wj = P.w[(size_t)b * P.w_stride + j];
  const double* theta = P.theta + (size_t)b * P.n * ndim;

  if (P.d.model == BISIP_MODEL_DECOMP) {
    const int D = P.d.n_coef, S = P.d.n_tau;
    const double* taus = P.taus + (size_t)b * P.tau_stride;
    const double* lts = P.log_taus + (size_t)b * P.tau_stride * D;
    if (tid < D) {
      double cs, sn;
      sincospi(0.5 * P.d.c_exp, &sn, &cs);
      s_g[tid] = dot2_lk(lts + (size_t)tid * S, taus, S, wj, P.d.c_exp, cs, sn, imag, 1.0);
    }
  } else if (tid == 0) {
    s_fq[0] = wj; s_fq[1] = sqrt(wj); s_fq[2] = log(wj); s_fq[3] = 0.0;
    for (int i = 4; i < kFq; ++i) s_fq[i] = 0.0;
  }
  __syncthreads();

  double s = 0.0, mn = __longlong_as_double(0x7ff0000000000000LL), mx = -mn;
  int nan = 0;
  for (int i = tid; i < n; i += NT) {
    const double* th = theta + (size_t)i * ndim;
    double zre, zim;
    switch (P.d.model) {
      case BISIP_MODEL_DECOMP: {
        const double R0 = th[0];
        double acc = 0.0;
        for (int q = 0; q < P.d.n_coef; ++q) acc = fma(R0 * th[1 + q], s_g[q], acc);
        zre = zim = (imag ? 0.0 : R0) - acc;           // decomp_c_eval_Z: R0 * delta_c - acc
        break;
      }
      case BISIP_MODEL_COLECOLE:
        colecole_point(th, P.d.n_modes, s_fq[2], zre, zim);
        break;
      case BISIP_MODEL_DIAS: {
        double rc[DiasRow::kRC];
        DiasRow::prepare(th, 0, rc);
        DiasRow rr;
        rr.R0 = rc[0]; rr.R0m = rc[1]; rr.tau = rc[2]; rr.tau_p = rc[3]; rr.sfac = rc[4];
        rr.eval<false>(s_fq, zre, zim);
        break;
      }
      default: {
        double rc[ShinRow::kRC];
        ShinRow::prepare(th, 0, rc);
        ShinRow rr;
#pragma unroll
        for (int e = 0; e < 2; ++e) { rr.iR[e] = rc[4 * e]; rr.n[e] = rc[4 * e + 1]; rr.qc[e] = rc[4 * e + 2]; rr.qs[e] = rc[4 * e + 3]; }
        rr.eval<false>(s_fq, zre, zim);
        break;
      }
    }
    const double v = imag ? zim : zre;
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
  const int C = 2 * N;
  smem_column_stats<NT>(vals, n, sum, mn, mx, has_nan, P.st, P.st.pct_out + (size_t)b * P.st.npct * C + c, C, nullptr,
                        nullptr, hist, pool, red);
}

}  // namespace bisip
