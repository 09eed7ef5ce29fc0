// PolynomialDecomposition (Debye / Warburg), collapsed form (precision = BISIP_PREC_FP64_COLLAPSED).
//
// The kernel matrix K = 1 - 1/(1+(i w tau)^c) of Decomp_cyth (cython_funcs.pyx:87-90) does not depend on
// theta, so the two-stage contraction  z_c = sum_k (sum_i a_i L_ik) K_kc  re-associates to
//     z_c = sum_i a_i G_ic ,   G = L K   ((poly_deg+1) x 2N, built once per spectrum),
// and one log-probability costs 2N (D + 2) FP64 FMAs instead of 2 S 2N + 2 D S flops (D = poly_deg+1):
// 1,792 instead of 17,792 at the C5 shape.  G is accumulated with a compensated (Dot2) sum, so the
// only rounding that differs from the two-stage path is the final D-term dot product; forward and
// log-probability meet the same 1e-12 parity bar against the reference (tests/test_gpu_collapsed.py).
// With D <= 8 the contraction is too thin for tensor tiles (an m16n8k8 DMMA tile pads D to 8 and runs
// on the same pipe at the same flop rate as DFMA), so it runs on the FP64 vector pipe: a thread owns
// kCRows proposals and one group of frequencies; the column records are warp-uniform broadcast loads.
//
// north_star grades the two-stage contraction on DMMA tiles, which therefore stays the default
// (decomp_eval.cuh); this evaluator is the opt-in fast path for users who only want the answer.
#pragma once
#include "common.cuh"
#include "decomp_eval.cuh"

namespace bisip {

constexpr int kCRec = 10;   // doubles per column record: y/sigma, delta/sigma, G[0..7]  (80 bytes, 16-byte aligned)

struct DecompCShape {
  int N, S, D, C;   // frequencies, taus, coefficients (<= 8), columns = 2N
  __host__ __device__ DecompCShape(int n, int s, int d) : N(n), S(s), D(d), C(2 * n) {}
  __host__ __device__ size_t rec_doubles() const { return (size_t)C * kCRec; }
};

struct DecompCSmem {
  double* rec;    // [2N][kCRec]
  double* part;   // [kWarps][rows_pad] partial chi^2 per column group
  double llconst; // sum 2 ln(sigma^2)
};

__host__ __device__ inline size_t decomp_c_smem_doubles(const DecompCShape& sh, int rows_pad) {
  return sh.rec_doubles() + (size_t)kWarps * rows_pad;
}

__device__ inline double* decomp_c_carve(DecompCSmem& s, double* base, const DecompCShape& sh, int rows_pad) {
  s.rec = base; base += sh.rec_doubles();
  s.part = base; base += (size_t)kWarps * rows_pad;
  return base;
}

// G_ic = sum_k L_ik K_kc * is for one column c: frequency wj, real part of K or the imaginary one (imag), lt = row i
// of L.  Compensated (Dot2, Ogita-Rump-Oishi) sum: sum + comp = the exact dot product to ~1 ulp.
__device__ __forceinline__ double dot2_lk(const double* __restrict__ lt, const double* __restrict__ taus, int S, double wj,
                                          double c_exp, double cs, double sn, bool imag, double is) {
  double sum = 0.0, comp = 0.0;
  for (int k = 0; k < S; ++k) {
    double kre, kim;
    debye_kernel_term(wj, taus[k], c_exp, cs, sn, kre, kim);
    const double kv = (imag ? kim : kre) * is;
    const double l = lt[k];
    const double p = __dmul_rn(l, kv);
    const double pe = __fma_rn(l, kv, -p);
    const double t = __dadd_rn(sum, p);
    const double bb = __dsub_rn(t, sum);
    const double se = __dadd_rn(__dsub_rn(sum, __dsub_rn(t, bb)), __dsub_rn(p, bb));
    sum = t;
    comp = __dadd_rn(comp, __dadd_rn(se, pe));
  }
  return sum + comp;
}

// Per-spectrum constants.  All threads of the CTA (any CTA size); ends with __syncthreads().
// Likelihood mode (y != nullptr): G and the data term are pre-scaled by 1/sigma_c exactly as
// decomp_init() pre-scales K, so the dot product yields the normalised residual directly.
__device__ inline void decomp_c_init(DecompCSmem& s, const DecompCShape& sh, double c_exp,
                                     const double* __restrict__ w, const double* __restrict__ taus,
                                     const double* __restrict__ log_taus,
                                     const double* __restrict__ y, const double* __restrict__ yerr,
                                     double* red) {
  const int tid = threadIdx.x, NT = blockDim.x;
  const int N = sh.N, S = sh.S, C = sh.C;
  const bool scaled = (y != nullptr);
  double csum = 0.0;
  for (int c = tid; c < C; c += NT) {
    double ys = 0.0, ds = (c < N) ? 1.0 : 0.0;
    if (scaled) {
      const double e = yerr[c];
      const double is = 1.0 / e;
      ys = y[c] * is;
      ds = (c < N) ? is : 0.0;
      csum += 2.0 * log(e * e);
    }
    s.rec[(size_t)c * kCRec + 0] = ys;
    s.rec[(size_t)c * kCRec + 1] = ds;
  }
  double cs, sn;
  sincospi(0.5 * c_exp, &sn, &cs);
  for (int idx = tid; idx < C * 8; idx += NT) {
    const int c = idx >> 3, i = idx & 7;
    double g = 0.0;
    if (i < sh.D) {
      const int j = c < N ? c : c - N;
      const double wj = w[j];
      const double is = scaled ? 1.0 / yerr[c] : 1.0;
      g = dot2_lk(log_taus + (size_t)i * S, taus, S, wj, c_exp, cs, sn, c >= N, is);
    }
    s.rec[(size_t)c * kCRec + 2 + i] = g;
  }
  // block-reduce the likelihood constant (fixed order -> deterministic)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) csum += __shfl_xor_sync(0xffffffffu, csum, o);
  if ((tid & 31) == 0) red[tid >> 5] = csum;
  __syncthreads();
  double tot = 0.0;
  for (int i = 0; i < (NT >> 5); ++i) tot += red[i];
  s.llconst = tot;
  __syncthreads();
}

// Rows (proposals) per thread of the register tile: every column record read from shared memory then feeds
// kCRows rows, which divides the LDS.128 traffic per FMA by kCRows (the broadcast loads, not the FP64 pipe, bound
// the one-row version: 4 LDS.128 per 7.5 DFMA).  Used when there are at least 32*kCRows rows; else one row per thread.
constexpr int kCRows = 2;

// Work split of an evaluation, a function of the largest number of rows the CTA evaluates (`rows_cap`) only:
// thread-rows (rpt proposals each) padded to a power of two >= 32 so that a warp works on ONE group, the N frequencies
// cut into `ngroups` (a power of two) groups of `fpg` frequencies — a group is the real columns AND the imaginary
// columns of its frequencies, so every warp has the same work (real columns cost one FMA more).  Thread t owns
// thread-rows tr0, tr0+tstep, ... and groups g0, g0+gstep, ...; an evaluation of fewer rows leaves the threads of the
// missing rows idle.  Shifts only (the CTA size is a power of two): it is rebuilt at every evaluation for ~20
// integer instructions — integer divisions here were 8 % of the kernel, and a plan kept across the sampler's phases
// was spilled and its reloads stalled the evaluation (long scoreboard, 5 % of the warp samples).
struct DecompCPlan {
  int rpt, trows, fpg, ngroups, tr0, tstep, g0, gstep;
  __device__ __forceinline__ void make(int rows_cap, int N) {
    const int NT = blockDim.x, tid = threadIdx.x;
    const int lg_nt = 31 - __clz(NT);
    rpt = (kCRows > 1 && rows_cap >= 32 * kCRows) ? kCRows : 1;
    trows = rpt > 1 ? (rows_cap + kCRows - 1) / kCRows : rows_cap;          // kCRows is a compile-time constant
    const int lg = trows <= 32 ? 5 : 32 - __clz(trows - 1);                 // rows_p = 2^lg >= max(32, trows)
    int lg_g = lg_nt - lg;                                                  // NT / rows_p groups fill the CTA
    if (lg_g < 0) lg_g = 0;
    const int lg_n = 31 - __clz(N);
    if (lg_g > lg_n) lg_g = lg_n;                                           // at most N groups
    ngroups = 1 << lg_g;                                                    // <= NT/32 <= kWarps
    fpg = (N + ngroups - 1) >> lg_g;                                        // trailing groups may be empty
    if (lg <= lg_nt) {      // NT / rows_p >= ngroups groups side by side: one pass
      gstep = NT >> lg;
      g0 = tid >> lg;
      tr0 = tid & ((1 << lg) - 1);
      tstep = 1 << lg;
    } else {                // more thread-rows than threads: every thread walks all groups
      gstep = 1; g0 = 0; tr0 = tid; tstep = NT;
    }
  }
};

// RPT proposals x a run of columns: chi[r] += sum_c ((y_c - Z_c)/sigma_c)^2 over columns [c0, c1)
template <int D, int RPT, bool REAL>
__device__ __forceinline__ void decomp_c_col(const double2 (&u)[(2 + D + 1) / 2], const double (&R0)[RPT],
                                             const double (&ra)[RPT][D], double (&chi)[RPT]) {
#pragma unroll
  for (int r = 0; r < RPT; ++r) {
    double a = REAL ? fma(-R0[r], u[0].y, u[0].x) : u[0].x;
#pragma unroll
    for (int i = 0; i < D; ++i) a = fma(ra[r][i], ((i & 1) ? u[1 + (i >> 1)].y : u[1 + (i >> 1)].x), a);
    chi[r] = fma(a, a, chi[r]);
  }
}

// explicit shared-memory load: through the struct-held generic pointer the compiler falls back to LD.E.128
__device__ __forceinline__ double2 lds_f64x2(uint32_t saddr) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(saddr));
  return v;
}

template <int D, int RPT, bool REAL>
__device__ __forceinline__ void decomp_c_rows(const double* __restrict__ rec, int c0, int c1, const double (&R0)[RPT],
                                              const double (&ra)[RPT][D], double (&chi)[RPT]) {
  const uint32_t r2 = (uint32_t)__cvta_generic_to_shared(rec);
  constexpr int kV = kCRec * 8;             // bytes per record
  constexpr int kL = (2 + D + 1) / 2;       // double2 actually needed
#pragma unroll 2
  for (int c = c0; c < c1; ++c) {
    double2 u[kL];
#pragma unroll
    for (int q = 0; q < kL; ++q) u[q] = lds_f64x2(r2 + c * kV + 16 * q);
    decomp_c_col<D, RPT, REAL>(u, R0, ra, chi);
  }
}

// Partial chi^2 of every (proposal, frequency group) into s.part[group][row].  No barrier.
template <int D, int RPT>
__device__ __forceinline__ void decomp_c_parts_dr(const DecompCSmem& s, const DecompCShape& sh, const DecompCPlan& pl,
                                                  const double* __restrict__ prop, int ndim, int nrows, int rows_pad) {
  for (int tr = pl.tr0; tr < pl.trows; tr += pl.tstep) {
    if (tr >= nrows) break;
    double R0[RPT], ra[RPT][D], x[RPT];
#pragma unroll
    for (int r = 0; r < RPT; ++r) {
      const int row = tr + r * pl.trows;
      const double* th = prop + (size_t)(row < nrows ? row : tr) * ndim;
      R0[r] = th[0];
#pragma unroll
      for (int i = 0; i < D; ++i) ra[r][i] = R0[r] * th[1 + i];
    }
    for (int grp = pl.g0; grp < pl.ngroups; grp += pl.gstep) {      // grp is warp-uniform
      const int f0 = grp * pl.fpg, f1 = min(sh.N, f0 + pl.fpg);
#pragma unroll
      for (int r = 0; r < RPT; ++r) x[r] = 0.0;
      decomp_c_rows<D, RPT, true>(s.rec, f0, f1, R0, ra, x);
      decomp_c_rows<D, RPT, false>(s.rec, sh.N + f0, sh.N + f1, R0, ra, x);
#pragma unroll
      for (int r = 0; r < RPT; ++r) {
        const int row = tr + r * pl.trows;
        if (row < nrows) s.part[(size_t)grp * rows_pad + row] = x[r];
      }
    }
  }
}

template <int D>
__device__ __forceinline__ void decomp_c_parts_d(const DecompCSmem& s, const DecompCShape& sh, const DecompCPlan& pl,
                                                 const double* __restrict__ prop, int ndim, int nrows, int rows_pad) {
  if (kCRows > 1 && pl.rpt == kCRows) decomp_c_parts_dr<D, kCRows>(s, sh, pl, prop, ndim, nrows, rows_pad);
  else decomp_c_parts_dr<D, 1>(s, sh, pl, prop, ndim, nrows, rows_pad);
}

// s.part[group][row] = sum over the group's columns of ((y_c - Z_c)/sigma_c)^2 for rows [0,nrows) of prop,
// nrows <= rows_cap; returns the number of groups.  Block-level; prop must be visible; s.part is written but not
// synchronised on return (the sampler's accept phase adds the groups behind its own barrier).
__device__ inline int decomp_c_eval_parts(const DecompCSmem& s, const DecompCShape& sh, int rows_cap,
                                          const double* __restrict__ prop, int ndim, int nrows, int rows_pad) {
  DecompCPlan pl;
  pl.make(rows_cap, sh.N);
  switch (sh.D) {
    case 1: decomp_c_parts_d<1>(s, sh, pl, prop, ndim, nrows, rows_pad); break;
    case 2: decomp_c_parts_d<2>(s, sh, pl, prop, ndim, nrows, rows_pad); break;
    case 3: decomp_c_parts_d<3>(s, sh, pl, prop, ndim, nrows, rows_pad); break;
    case 4: decomp_c_parts_d<4>(s, sh, pl, prop, ndim, nrows, rows_pad); break;
    case 5: decomp_c_parts_d<5>(s, sh, pl, prop, ndim, nrows, rows_pad); break;
    case 6: decomp_c_parts_d<6>(s, sh, pl, prop, ndim, nrows, rows_pad); break;
    case 7: decomp_c_parts_d<7>(s, sh, pl, prop, ndim, nrows, rows_pad); break;
    default: decomp_c_parts_d<8>(s, sh, pl, prop, ndim, nrows, rows_pad); break;
  }
  return pl.ngroups;
}

// number of column groups decomp_c_eval_parts() produces for this rows_cap (the reader's side of the plan)
__device__ __forceinline__ int decomp_c_ngroups(int rows_cap, int N) {
  DecompCPlan pl;
  pl.make(rows_cap, N);
  return pl.ngroups;
}

// Forward only (decomp_c_init with y == nullptr): Z[row][2][N] = R0*(delta_c - z_c), coalesced over columns.
__device__ inline void decomp_c_eval_Z(const DecompCSmem& s, const DecompCShape& sh, const double* __restrict__ prop,
                                       int ndim, int nrows, double* __restrict__ Zout) {
  const int C = sh.C;
  for (int idx = threadIdx.x; idx < nrows * C; idx += blockDim.x) {
    const int row = idx / C, c = idx - row * C;
    const double* th = prop + (size_t)row * ndim;
    const double* r = s.rec + (size_t)c * kCRec;
    const double R0 = th[0];
    double acc = 0.0;
    for (int i = 0; i < sh.D; ++i) acc = fma(R0 * th[1 + i], r[2 + i], acc);
    Zout[idx] = R0 * r[1] - acc;
  }
}

}  // namespace bisip
