// ensemble_kernel<VecEvaluator<ColeColeRowT<K>>>: Pelton Cole-Cole, 1..kMaxModes modes.
#include "ens_vec.cuh"

namespace bisip {

int launch_ens_colecole(const EnsembleParams& P, dim3 grid, size_t smem, cudaStream_t st) {
  switch (P.d.n_modes) {
    // 1 mode with <= 256 walkers runs the warp-private kernel (ens_wp_vec.cu)
    case 1: return launch(ensemble_kernel<VecEvaluator<ColeColeRowT<1>>, kMinBVec, kThreads>, grid, smem, st, "ensemble_colecole", &P, kThreads);
    case 2: return launch_vec_ensemble<ColeColeRowT<2>, 6>(P, grid, smem, st, "ensemble_colecole");
    case 3: return launch(ensemble_kernel<VecEvaluator<ColeColeRowT<3>>, 2>, grid, smem, st, "ensemble_colecole", &P);
    case 4: return launch(ensemble_kernel<VecEvaluator<ColeColeRowT<4>>, 1>, grid, smem, st, "ensemble_colecole", &P);
    default:
      if (P.d.n_modes <= 8) return launch(ensemble_kernel<VecEvaluator<ColeColeRow>, 1>, grid, smem, st, "ensemble_colecole", &P);
      return launch(ensemble_kernel<VecEvaluator<ColeColeRowBig>, 1>, grid, smem, st, "ensemble_colecole", &P);
  }
}

}  // namespace bisip
