// ensemble_wp_kernel<CollapsedMmaEvaluator<KS>>: precision 'fp64-collapsed' on FP64 tensor tiles, W <= 256.
#include "ens_wp.cuh"

namespace bisip {

int launch_ens_wp_collapsed(const EnsembleParams& P, dim3 grid, cudaStream_t st) {
  const int KS = (P.d.n_coef + 2 + 7) / 8;
  const size_t other = wp_smem_bytes(P.W, P.d.ndim);
  switch (KS) {
    case 1: return launch_wp<CollapsedMmaEvaluator<1>, 64>(P, grid, other + CollapsedMmaEvaluator<1>::smem_doubles(P.d) * 8, st, "ensemble_wp_decomp_collapsed");
    case 2: return launch_wp<CollapsedMmaEvaluator<2>, 64>(P, grid, other + CollapsedMmaEvaluator<2>::smem_doubles(P.d) * 8, st, "ensemble_wp_decomp_collapsed");
    default: return launch_wp<CollapsedMmaEvaluator<4>, 80>(P, grid, other + CollapsedMmaEvaluator<4>::smem_doubles(P.d) * 8, st, "ensemble_wp_decomp_collapsed");
  }
}

}  // namespace bisip
