// ensemble_kernel<DecompCollapsedEvaluator>: precision 'fp64-collapsed' (decomp_collapsed.cuh) with more than 256
// walkers; up to 256 the warp-private kernel runs (ens_wp_collapsed.cu).
#include "launch.cuh"

namespace bisip {

constexpr int kMinBCollapsed = 3;   // 256-thread CTAs: 80 registers and no spills; at 4 per SM (64 registers) the spill
                                    // reloads cost more than the fourth CTA hides (-4 %)

// Never launched: with <= 256 walkers the warp-private kernel runs.  Compiled all the same, because without them in
// this translation unit the compiler builds the 256-thread kernel differently (120 more instructions), and on a B200
// at 1,000 W it ran 0.8 % slower (512 walkers).
template __global__ void ensemble_kernel<DecompCollapsedEvaluator, 8, 128>(const EnsembleParams);
template __global__ void ensemble_kernel<DecompCollapsedEvaluator, 6, 128>(const EnsembleParams);

int launch_ens_collapsed(const EnsembleParams& P, dim3 grid, size_t smem, cudaStream_t st) {
  return launch(ensemble_kernel<DecompCollapsedEvaluator, kMinBCollapsed, kThreads>, grid, smem, st,
                "ensemble_decomp_collapsed", &P, kThreads);
}

}  // namespace bisip
