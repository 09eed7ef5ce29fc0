// ensemble_kernel<VecEvaluator<DiasRow | ShinRow>>.
#include "ens_vec.cuh"

namespace bisip {

// 128-thread kernels (profiles/r02c_vec_analysis.md): with the branch-free frequency loop four frequencies in flight at
// 80 registers (6 CTAs/SM) beat two at 64 (8 CTAs/SM) for Dias by 2 %, not for Shin
int launch_ens_dias_shin(const EnsembleParams& P, dim3 grid, size_t smem, cudaStream_t st) {
  if (P.d.model == BISIP_MODEL_DIAS) return launch_vec_ensemble<DiasRow, 6, 4>(P, grid, smem, st, "ensemble_dias");
  return launch_vec_ensemble<ShinRow, 6>(P, grid, smem, st, "ensemble_shin");
}

}  // namespace bisip
