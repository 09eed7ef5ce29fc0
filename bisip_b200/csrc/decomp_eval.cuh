// PolynomialDecomposition (Debye / Warburg) evaluator: the two-stage real contraction
//   stage 1  M[row][k]  = sum_i a[row][i] * L[i][k]          (walker coefficients -> chargeability over tau grid)
//   stage 2  z[row][c]  = sum_k M[row][k] * K[k][c]          (chargeability -> 2N real/imag frequency columns)
//   epilogue Z = R0*(delta_re - z),  chi = sum_c ((y - Z)/sigma)^2
// on FP64 tensor tiles (mma.sync .f64 -> DMMA.8x8x4).  Restates reference Decomp_cyth
// (cython_funcs.pyx:75-94) + C_Debye (:46-47) + _log_likelihood (models.py:59-62); the
// theta-independent factor K = 1 - 1/(1+(i w tau)^c), which the reference recomputes with
// cpow on every call, is built once per spectrum in shared memory in B-fragment order.
//
// One warp owns a 16-row tile of proposals.  Stage 1 leaves M in accumulator layout, which is
// re-used directly as the stage-2 A fragment (tau order inside a 16-chunk is permuted to
// match; K is stored with the same permutation), so M never touches shared memory.
#pragma once
#include "common.cuh"

namespace bisip {

struct DecompShape {
  int N;     // frequencies
  int S;     // taus
  int D;     // coefficients (poly_deg+1), <= 8
  int NT2;   // stage-2 column tiles  = ceil(2N/8)
  int KC;    // stage-2 k chunks      = ceil(S/16)
  __host__ __device__ DecompShape(int n, int s, int d) : N(n), S(s), D(d), NT2(ceil_div(2 * n, 8)), KC(ceil_div(s, 16)) {}
  __host__ __device__ size_t kf_doubles() const { return (size_t)NT2 * KC * 128; }
  __host__ __device__ size_t l1_doubles() const { return (size_t)KC * 2 * 2 * 32; }
  __host__ __device__ size_t col_doubles() const { return (size_t)NT2 * 8; }
};

// Position of K[tau k][column c] inside the fragment-ordered shared array.
//   chunk kc = k>>4; inside: hh = (k>>3)&1, t = (k>>1)&3, e = k&1  (tau = 16kc + 8hh + 2t + e)
//   tile  nt = c>>3, g = c&7 ; lane = 4g + t ; one 16-byte slot per (nt,kc,hh,lane) holds e=0,1
__device__ __forceinline__ int kf_index(int k, int c, int KC) {
  const int kc = k >> 4, hh = (k >> 3) & 1, t = (k >> 1) & 3, e = k & 1;
  const int nt = c >> 3, g = c & 7;
  return ((((nt * KC + kc) * 2 + hh) * 32 + (g * 4 + t)) << 1) + e;
}

// K(w,tau,c) = 1 - 1/(1+z), z = (i w tau)^c = x*(cos(c pi/2) + i sin(c pi/2)), x = (w tau)^c.
// (D-1)/D form: re = (u + x^2)/|D|^2, im = v/|D|^2 with u = x cs, v = x sn, D = 1+u+iv.
__device__ __forceinline__ void debye_kernel_term(double w, double tau, double c_exp, double cs, double sn,
                                                  double& kre, double& kim) {
  const double wt = w * tau;
  const double x = (c_exp == 1.0) ? wt : pow(wt, c_exp);
  const double u = x * cs, v = x * sn;
  const double d1 = 1.0 + u;
  const double den = d1 * d1 + v * v;
  kre = (u + x * x) / den;
  kim = v / den;
}

struct DecompSmem {
  double* Kf;    // [NT2][KC][2][32][2]
  double* L1;    // [2KC][2][32]   stage-1 B fragments (powers of log_tau)
  double* ycol;  // [NT2*8]  y/sigma per column (real | imag | 0-pad)      [forward-only mode: unused]
  double* isig;  // [NT2*8]  delta_c/sigma per column: 1/sigma on real columns, 0 on imaginary / padding
  double* part;  // [NG][rows_pad] partial chi (only when column groups are split over warps)
  double llconst; // sum 2*ln(sigma^2)
};

__host__ __device__ inline size_t decomp_smem_doubles(const DecompShape& sh, int rows_pad) {
  return sh.kf_doubles() + sh.l1_doubles() + 2 * sh.col_doubles() + (size_t)kWarps * rows_pad;
}

__device__ inline double* decomp_carve(DecompSmem& s, double* base, const DecompShape& sh, int rows_pad) {
  s.Kf = base; base += sh.kf_doubles();
  s.L1 = base; base += sh.l1_doubles();
  s.ycol = base; base += sh.col_doubles();
  s.isig = base; base += sh.col_doubles();
  s.part = base; base += (size_t)kWarps * rows_pad;
  return base;
}

// Build the per-spectrum constants.  All threads; ends with __syncthreads().
// red: scratch double[kWarps] for the block reduction of the likelihood constant.
__device__ inline void decomp_init(DecompSmem& s, const DecompShape& sh, double c_exp,
                                   const double* __restrict__ w, const double* __restrict__ taus,
                                   const double* __restrict__ log_taus,
                                   const double* __restrict__ y, const double* __restrict__ yerr,
                                   double* red) {
  const int tid = threadIdx.x, nthr = blockDim.x;     // any CTA size (the warp-private sampler runs 32 ... 256 threads)
  const int N = sh.N, S = sh.S, KC = sh.KC;
  for (int i = tid; i < (int)sh.kf_doubles(); i += nthr) s.Kf[i] = 0.0;
  // stage-1 B fragments: tile j (8 taus), half q: power t+4q, tau 8j+g
  for (int i = tid; i < (int)sh.l1_doubles(); i += nthr) {
    const int lane = i & 31, q = (i >> 5) & 1, j = i >> 6;
    const int g = lane >> 2, t = lane & 3;
    const int p = t + 4 * q, k = 8 * j + g;
    s.L1[i] = (p < sh.D && k < S) ? log_taus[(size_t)p * S + k] : 0.0;
  }
  // Likelihood mode (y != nullptr): the residual is produced directly by the tiles,
  //   r_c/sigma_c = y_c/sigma_c - R0*delta_c/sigma_c + sum_k (R0*M_k) * (K_kc/sigma_c),
  // so K is stored pre-scaled by 1/sigma_c and the accumulators start at ys_c - R0*ds_c.
  const bool scaled = (y != nullptr);
  double csum = 0.0;
  for (int c = tid; c < (int)sh.col_doubles(); c += nthr) {
    double ys = 0.0, ds = 0.0;
    if (c < 2 * N && scaled) {
      const double e = yerr[c];
      const double is = 1.0 / e;
      ys = y[c] * is;
      ds = (c < N) ? is : 0.0;
      csum += 2.0 * log(e * e);
    }
    s.ycol[c] = ys;
    s.isig[c] = ds;
  }
  __syncthreads();   // Kf zero-fill complete before scatter
  double cs, sn;
  sincospi(0.5 * c_exp, &sn, &cs);
  for (int i = tid; i < S * N; i += nthr) {
    const int k = i / N, j = i - k * N;
    double kre, kim;
    debye_kernel_term(w[j], taus[k], c_exp, cs, sn, kre, kim);
    if (scaled) {
      kre *= 1.0 / yerr[j];
      kim *= 1.0 / yerr[N + j];
    }
    s.Kf[kf_index(k, j, KC)] = kre;
    s.Kf[kf_index(k, N + j, KC)] = kim;
  }
  // block-reduce the likelihood constant (fixed order -> deterministic)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) csum += __shfl_xor_sync(0xffffffffu, csum, o);
  if ((tid & 31) == 0) red[tid >> 5] = csum;
  __syncthreads();
  double tot = 0.0;
  for (int i = 0; i < (nthr >> 5); ++i) tot += red[i];
  s.llconst = tot;
  __syncthreads();
}

// Warp-level: stage 1 for row tile `r` -> A fragments of all KC chunks (registers).
template <int KC>
__device__ __forceinline__ void decomp_stage1(const DecompSmem& s, int D, const double* __restrict__ prop, int ndim,
                                              int r, int lane, double (&A)[KC][8], double& R0a, double& R0b) {
  const int g = lane >> 2, t = lane & 3;
  const double* q0 = prop + (size_t)(r * 16 + g) * ndim;
  const double* q1 = q0 + 8 * ndim;
  R0a = q0[0];
  R0b = q1[0];
  double a1[4];   // coefficients pre-multiplied by R0: stage 2 then yields R0*z directly
  a1[0] = (t < D) ? R0a * q0[1 + t] : 0.0;
  a1[1] = (t < D) ? R0b * q1[1 + t] : 0.0;
  a1[2] = (t + 4 < D) ? R0a * q0[5 + t] : 0.0;
  a1[3] = (t + 4 < D) ? R0b * q1[5 + t] : 0.0;
#pragma unroll
  for (int kc = 0; kc < KC; ++kc) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = 2 * kc + h;
      double b1[2] = {s.L1[(j * 2 + 0) * 32 + lane], s.L1[(j * 2 + 1) * 32 + lane]};
      double c[4] = {0.0, 0.0, 0.0, 0.0};
      dmma_16x8x8(c, a1, b1);
      A[kc][4 * h + 0] = c[0];
      A[kc][4 * h + 1] = c[2];
      A[kc][4 * h + 2] = c[1];
      A[kc][4 * h + 3] = c[3];
    }
  }
}

// Stage 2 for one column tile: c[16 rows][8 cols] += (R0*M) x K'.  The caller initialises c.
template <int KC>
__device__ __forceinline__ void decomp_stage2_tile(const DecompSmem& s, int nt, int lane, const double (&A)[KC][8],
                                                   double (&c)[4]) {
  const double2* kf = reinterpret_cast<const double2*>(s.Kf) + (size_t)nt * KC * 64 + lane;
#pragma unroll
  for (int kc = 0; kc < KC; ++kc) {
    const double2 b01 = kf[kc * 64];
    const double2 b23 = kf[kc * 64 + 32];
    const double b[4] = {b01.x, b01.y, b23.x, b23.y};
    dmma_16x8x16(c, A[kc], b);
  }
}

// chi[row] = sum_c ((y_c - R0*(delta_c - z_c)) / sigma_c)^2 for rows [0,nrows) of prop
// (likelihood mode of decomp_init: pre-scaled K, accumulators start at the data term).
// Block-level; prop must be visible; on return chi[] is written but NOT yet synchronised
// when NG==1, synchronised internally when the column tiles were split over warps.
// How the (row tile, column group) work items are laid out for `nrows` proposals.
__device__ __forceinline__ void decomp_work_split(const DecompShape& sh, int nrows, int& RT, int& NG, int& TPG) {
  RT = (nrows + 15) >> 4;
  NG = kWarps / RT;
  if (NG < 1) NG = 1;
  if (NG > sh.NT2) NG = sh.NT2;
  TPG = ceil_div(sh.NT2, NG);
  NG = ceil_div(sh.NT2, TPG);
}
// Column-tile iterations each warp executes in one evaluation (pacing of the interleaved side work).
__device__ __forceinline__ int decomp_iters_per_warp(const DecompShape& sh, int nrows) {
  int RT, NG, TPG;
  decomp_work_split(sh, nrows, RT, NG, TPG);
  return ceil_div(RT * NG, kWarps) * TPG;
}
struct NoSide {
  __device__ __forceinline__ void advance() {}
  __device__ __forceinline__ void finish() {}
};

template <int KC, class Side>
__device__ inline void decomp_eval_chi(const DecompSmem& s, const DecompShape& sh, const double* __restrict__ prop,
                                       int ndim, int nrows, int rows_pad, double* chi, Side& side) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  int RT, NG, TPG;
  decomp_work_split(sh, nrows, RT, NG, TPG);
  for (int item = warp; item < RT * NG; item += kWarps) {
    const int r = item % RT, cg = item / RT;
    double A[KC][8];
    double R0a, R0b;
    decomp_stage1<KC>(s, sh.D, prop, ndim, r, lane, A, R0a, R0b);
    double chi0 = 0.0, chi1 = 0.0;
    const int nt_end = min(sh.NT2, (cg + 1) * TPG);
#pragma unroll 2
    for (int nt = cg * TPG; nt < nt_end; ++nt) {
      const int col = nt * 8 + 2 * t;
      const double2 ys = *reinterpret_cast<const double2*>(s.ycol + col);
      double c[4];
      if (nt * 8 >= sh.N) {          // tile entirely in the imaginary block: delta = 0 (warp-uniform)
        c[0] = ys.x; c[1] = ys.y; c[2] = ys.x; c[3] = ys.y;
      } else {
        const double2 ds = *reinterpret_cast<const double2*>(s.isig + col);
        c[0] = fma(-R0a, ds.x, ys.x);
        c[1] = fma(-R0a, ds.y, ys.y);
        c[2] = fma(-R0b, ds.x, ys.x);
        c[3] = fma(-R0b, ds.y, ys.y);
      }
      decomp_stage2_tile<KC>(s, nt, lane, A, c);      // c = (y - Z)/sigma
      side.advance();                                  // integer side work rides along with the tiles
      chi0 = fma(c[0], c[0], chi0);
      chi0 = fma(c[1], c[1], chi0);
      chi1 = fma(c[2], c[2], chi1);
      chi1 = fma(c[3], c[3], chi1);
    }
    chi0 += __shfl_xor_sync(0xffffffffu, chi0, 1);
    chi0 += __shfl_xor_sync(0xffffffffu, chi0, 2);
    chi1 += __shfl_xor_sync(0xffffffffu, chi1, 1);
    chi1 += __shfl_xor_sync(0xffffffffu, chi1, 2);
    if (t == 0) {
      double* dst = (NG == 1) ? chi : s.part + (size_t)cg * rows_pad;
      dst[r * 16 + g] = chi0;
      dst[r * 16 + g + 8] = chi1;
    }
  }
  if (NG > 1) {
    __syncthreads();
    for (int p = threadIdx.x; p < RT * 16; p += kThreads) {
      double acc = 0.0;
      for (int cg = 0; cg < NG; ++cg) acc += s.part[(size_t)cg * rows_pad + p];
      chi[p] = acc;
    }
  }
}

// Forward only: Z[row][2][N] (global) for rows [0,nrows) of prop.
template <int KC>
__device__ inline void decomp_eval_Z(const DecompSmem& s, const DecompShape& sh, const double* __restrict__ prop,
                                     int ndim, int nrows, double* __restrict__ Zout) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int RT = (nrows + 15) >> 4;
  for (int item = warp; item < RT * sh.NT2; item += kWarps) {
    const int r = item % RT, nt = item / RT;
    double A[KC][8];
    double R0a, R0b;
    decomp_stage1<KC>(s, sh.D, prop, ndim, r, lane, A, R0a, R0b);
    double c[4] = {0.0, 0.0, 0.0, 0.0};
    decomp_stage2_tile<KC>(s, nt, lane, A, c);       // c = R0*z
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int col = nt * 8 + 2 * t + e;
      if (col < 2 * sh.N) {
        const double d = (col < sh.N) ? 1.0 : 0.0;
        const int row0 = r * 16 + g, row1 = row0 + 8;
        if (row0 < nrows) Zout[(size_t)row0 * 2 * sh.N + col] = R0a * d - c[e];
        if (row1 < nrows) Zout[(size_t)row1 * 2 * sh.N + col] = R0b * d - c[2 + e];
      }
    }
  }
}

}  // namespace bisip
