// Batched forward / log-probability (batch_decomp.cu, batch_vec.cu): one kernel template over the sampler's evaluator
// adaptors (sampler.cuh), so the batch API runs exactly the evaluation code the sampler runs.
#pragma once
#include "launch.cuh"

namespace bisip {

// Grid (chunks * cs, B), cs = CTAs per cluster (1 unless Eval::kClustered): the CTA (cluster) at chunk c handles theta
// rows [c * kRows, ...) of spectrum blockIdx.y, striding by the number of chunks.  Shared memory: the evaluator's
// region, then prop [kRows][ndim], chi [kRows], bounds [2][ndim] and the reduction scratch [kWarps]
// (batch_other_bytes).
// Clustered evaluators: every CTA of the cluster evaluates the same rows (column split), rank 0 alone writes lp.
template <class Eval, bool WANT_Z>
__global__ void __launch_bounds__(kThreads) batch_kernel(const BatchParams P) {
  extern __shared__ __align__(16) double smem[];
  int cs = 1, crank = 0;
  if (Eval::kClustered) {
    cg::cluster_group cluster = cg::this_cluster();
    cs = (int)cluster.num_blocks();
    crank = (int)cluster.block_rank();
  }
  const int b = blockIdx.y, ndim = P.d.ndim, N = P.d.n_freq;
  // unsigned as in blockIdx: with int chunk indices the tcgen05 TF32 forward ran 3 % slower (B200, 1,000 W)
  const unsigned chunk0 = blockIdx.x / cs, nchunks = gridDim.x / cs;
  Eval ev(P.d, cs, crank);
  double* p = ev.carve(smem, kRows);
  double* prop = p; p += kRows * ndim;
  double* chi = p; p += kRows;
  double* bnd = p; p += 2 * ndim;
  double* red = p;
  if (!WANT_Z) for (int i = threadIdx.x; i < 2 * ndim; i += kThreads) bnd[i] = P.bounds[i];
  ev.init(P.d, P.w + (size_t)b * P.w_stride, P.taus + (size_t)b * P.tau_stride,
          P.log_taus + (size_t)b * P.tau_stride * P.d.n_coef,
          WANT_Z ? nullptr : P.y + (size_t)b * 2 * N, WANT_Z ? nullptr : P.yerr + (size_t)b * 2 * N, red);
  for (int r0 = chunk0 * kRows; r0 < P.n_theta; r0 += nchunks * kRows) {
    const int n = min(kRows, P.n_theta - r0);
    const double* th = P.theta + ((size_t)b * P.n_theta + r0) * ndim;
    for (int i = threadIdx.x; i < kRows * ndim; i += kThreads) prop[i] = (i < n * ndim) ? th[i] : 0.0;
    __syncthreads();
    if (Eval::kNeedsPrepare) {
      // blockDim.x, not kThreads: with kThreads the 3-mode Cole-Cole kernel took 89 registers (2 CTAs/SM, 13 % slower)
      for (int q = threadIdx.x; q < n; q += blockDim.x) ev.prepare_row(q, prop + q * ndim);
      __syncthreads();
    }
    if (WANT_Z) {
      ev.eval_Z(prop, ndim, n, P.Z + ((size_t)b * P.n_theta + r0) * 2 * N);
    } else {
      NoSide ns;
      ev.eval_chi(prop, ndim, n, chi, ns);
      __syncthreads();
      if (crank == 0)
        for (int q = threadIdx.x; q < n; q += kThreads)
          P.lp[(size_t)b * P.n_theta + r0 + q] =
              in_bounds(prop + q * ndim, bnd, ndim) ? -0.5 * (ev.chi_of(chi, q) + ev.llconst()) : neg_inf();
    }
    __syncthreads();
  }
  ev.release();
  if (Eval::kClustered && cs > 1) cg::this_cluster().sync();   // peers may still read our shared memory
}

// Shared memory of batch_kernel<Eval> for the evaluators sized by the problem shape alone (the clustered and tcgen05
// evaluators take theirs from plan_rc / plan_umma).
template <class Eval>
size_t batch_smem(const bisip_model_desc& d) {
  return batch_other_bytes(d) + Eval::smem_doubles(d, kRows) * 8;
}

// One CTA (cluster of cs CTAs) per chunk of kRows theta rows, capped at per_sm CTAs per SM over the whole grid: enough
// CTAs to fill the chip, no more.
template <class Eval, bool WANT_Z>
int launch_batch(const BatchParams& P, int per_sm, size_t smem, cudaStream_t st, const char* name, int cs = 1) {
  const int cap = max(1, device_sm_count() * per_sm / max(1, P.B * cs));
  const dim3 grid(min(ceil_div(P.n_theta, kRows), cap) * cs, P.B);
  if (Eval::kClustered) return launch_cluster(batch_kernel<Eval, WANT_Z>, grid, cs, smem, st, name, &P);
  return launch(batch_kernel<Eval, WANT_Z>, grid, smem, st, name, &P);
}

}  // namespace bisip
