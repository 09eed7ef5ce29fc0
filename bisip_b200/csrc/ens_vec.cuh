// Vector-model ensemble kernels: CTA size and resident CTAs per SM.  Their evaluation phase is short, so
// the serial phases of the stretch move (proposals, accept, split) are about half of a step: many co-resident
// spectra hide them, and for <= 128 walkers 128-thread CTAs (8 or 6 per SM instead of 4 x 256) keep fewer
// lanes idle in those phases.  Values from the sweeps in profiles/r01c_vec_occupancy.md and
// profiles/r01d_vec_kernels.md (W=128, N=64).
#pragma once
#include "launch.cuh"

namespace bisip {

constexpr int kMinBVec = 4;      // 256-thread CTAs, 64 registers
constexpr int kVecSmallW = 128;  // walkers up to which the 128-thread variant is used

// launch ensemble_kernel<VecEvaluator<Row>> in the shape picked for W walkers; MB128 = CTAs/SM of the
// 128-thread variant (8 -> 64 registers, 6 -> 80 registers), ILP128 = its frequencies in flight per thread
template <class Row, int MB128, int ILP128 = 2>
int launch_vec_ensemble(const EnsembleParams& P, dim3 grid, size_t smem, cudaStream_t st, const char* name) {
  if (P.W <= kVecSmallW)
    return launch(ensemble_kernel<VecEvaluator<Row, ILP128>, MB128, 128>, grid, smem, st, name, &P, 128);
  return launch(ensemble_kernel<VecEvaluator<Row>, kMinBVec, kThreads>, grid, smem, st, name, &P, kThreads);
}

}  // namespace bisip
