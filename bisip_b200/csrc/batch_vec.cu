// Batched forward / log-probability of the Cole-Cole / Dias / Shin models (same evaluators as the sampler).
#include "batch.cuh"

namespace bisip {

template <class Row, bool WANT_Z>
static int launch_vec(const BatchParams& P, cudaStream_t st, const char* name) {
  return launch_batch<VecEvaluator<Row>, WANT_Z>(P, 8, batch_smem<VecEvaluator<Row>>(P.d), st, name);
}

template <bool WANT_Z>
static int run_batch_vec_t(const BatchParams& P, cudaStream_t st) {
  switch (P.d.model) {
    case BISIP_MODEL_COLECOLE:
      switch (P.d.n_modes) {
        case 1: return launch_vec<ColeColeRowT<1>, WANT_Z>(P, st, "colecole_batch");
        case 2: return launch_vec<ColeColeRowT<2>, WANT_Z>(P, st, "colecole_batch");
        case 3: return launch_vec<ColeColeRowT<3>, WANT_Z>(P, st, "colecole_batch");
        case 4: return launch_vec<ColeColeRowT<4>, WANT_Z>(P, st, "colecole_batch");
        default:
          if (P.d.n_modes <= 8) return launch_vec<ColeColeRow, WANT_Z>(P, st, "colecole_batch");
          return launch_vec<ColeColeRowBig, WANT_Z>(P, st, "colecole_batch");
      }
    case BISIP_MODEL_DIAS: return launch_vec<DiasRow, WANT_Z>(P, st, "dias_batch");
    default: return launch_vec<ShinRow, WANT_Z>(P, st, "shin_batch");
  }
}

int run_batch_vec(const BatchParams& P, bool want_z, cudaStream_t st) {
  return want_z ? run_batch_vec_t<true>(P, st) : run_batch_vec_t<false>(P, st);
}

}  // namespace bisip
