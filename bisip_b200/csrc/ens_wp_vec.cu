// ensemble_wp_kernel<VecWarpEvaluator<Row>>: Dias, Shin and 1-2 mode Cole-Cole, W <= 256.
#include "ens_wp.cuh"

namespace bisip {

// frequencies in flight and register caps: the measured best (profiles/r02_wp_sweep.md, r02c_vec_analysis.md)
using DiasEval = VecWarpEvaluator<DiasRow, 4>;
using ShinEval = VecWarpEvaluator<ShinRow, 2>;

int launch_ens_wp_vec(const EnsembleParams& P, dim3 grid, cudaStream_t st) {
  const int rp = wp_rows_pad(P.W);
  const size_t other = wp_smem_bytes(P.W, P.d.ndim);
  switch (P.d.model) {
    case BISIP_MODEL_DIAS:
      return launch_wp<DiasEval, 80>(P, grid, other + DiasEval::smem_doubles(P.d, rp) * 8, st, "ensemble_wp_dias");
    case BISIP_MODEL_SHIN:
      return launch_wp<ShinEval, 80>(P, grid, other + ShinEval::smem_doubles(P.d, rp) * 8, st, "ensemble_wp_shin");
    default:
      if (P.d.n_modes == 1)
        return launch_wp<VecWarpEvaluator<ColeColeRowT<1>>, 80>(P, grid, other + VecWarpEvaluator<ColeColeRowT<1>>::smem_doubles(P.d, rp) * 8, st, "ensemble_wp_colecole");
      return launch_wp<VecWarpEvaluator<ColeColeRowT<2>>, 80>(P, grid, other + VecWarpEvaluator<ColeColeRowT<2>>::smem_doubles(P.d, rp) * 8, st, "ensemble_wp_colecole");
  }
}

}  // namespace bisip
