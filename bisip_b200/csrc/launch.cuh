// Host-side helpers shared by the translation units of libbisip_b200.so: error reporting, launch wrappers and the
// kernel plans (which kernel / cluster size / shared memory a problem shape gets).  The library is split into several
// .cu files only so that they compile in parallel; the kernels themselves live in the .cuh headers.
#pragma once
#include <atomic>
#include <string>

#include "common.cuh"
#include "sampler.cuh"

namespace bisip {

int fail(int code, const std::string& msg);        // api.cu: stores the thread-local last-error string
void count_launches(int n);                        // api.cu: bisip_launch_count()

#define BISIP_CUDA(expr)                                                                      \
  do {                                                                                        \
    cudaError_t e_ = (expr);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(BISIP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));        \
  } while (0)

inline int device_smem_optin() {
  int dev = 0, v = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  return v;
}

inline int device_sm_count() {
  int dev = 0, v = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
  return v;
}

template <typename K>
int launch(K kernel, dim3 grid, size_t smem, cudaStream_t st, const char* name, const void* params_ptr,
           int threads = kThreads) {
  if ((int)smem > device_smem_optin())
    return fail(BISIP_ERR_UNSUPPORTED, std::string(name) + ": problem does not fit in shared memory");
  BISIP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  void* args[] = {const_cast<void*>(params_ptr)};
  BISIP_CUDA(cudaLaunchKernel((const void*)kernel, grid, dim3(threads), args, smem, st));
  count_launches(1);
  return BISIP_OK;
}

template <typename K>
int launch_cluster(K kernel, dim3 grid, int cluster, size_t smem, cudaStream_t st, const char* name,
                   const void* params_ptr) {
  if ((int)smem > device_smem_optin())
    return fail(BISIP_ERR_UNSUPPORTED, std::string(name) + ": problem does not fit in shared memory");
  BISIP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  void* args[] = {const_cast<void*>(params_ptr)};
  BISIP_CUDA(cudaLaunchKernelExC(&cfg, (const void*)kernel, args));
  count_launches(1);
  return BISIP_OK;
}

// ---- batched forward / log-probability (batch_*.cu) ---------------------------------------------------------------
constexpr int kRows = 128;     // theta rows per CTA pass

struct BatchParams {
  bisip_model_desc d;
  int B, n_theta;
  const double* theta;
  const double* w; long long w_stride;
  const double* taus; const double* log_taus; long long tau_stride;
  const double* y; const double* yerr; const double* bounds;
  double* Z; double* lp;
};

inline size_t batch_other_bytes(const bisip_model_desc& d) {
  return ((size_t)kRows * d.ndim + kRows + 2 * d.ndim + kWarps) * 8;
}

// ---- kernel plans --------------------------------------------------------------------------------------------------
// 0 = FP64, 1 = TF32, 3 = 3xTF32 (operand planes per product)
inline int prec_planes(int precision) {
  switch (precision) {
    case BISIP_PREC_TF32: case BISIP_PREC_TF32_MMA: return 1;
    case BISIP_PREC_3XTF32: case BISIP_PREC_3XTF32_MMA: return 3;
    default: return 0;
  }
}

// Large tau grids: pick the cluster size (column split) so that K fits; prefer two CTAs per SM.
struct RcPlan { int cs; bool two_per_sm; size_t smem; };
inline size_t rc_eval_doubles(const bisip_model_desc& d, int rows_pad, int cs) {
  switch (prec_planes(d.precision)) {
    case 1: return DecompTF32Evaluator<1>::smem_doubles(d, rows_pad, cs);
    case 3: return DecompTF32Evaluator<3>::smem_doubles(d, rows_pad, cs);
    default: return DecompRCEvaluator::smem_doubles(d, rows_pad, cs);
  }
}
inline int plan_rc(const bisip_model_desc& d, size_t other_bytes, int rows_pad, RcPlan* out) {
  // Smallest cluster first; for a given cluster size two CTAs per SM if they fit, else one.  A wider cluster is
  // worse than a lower occupancy: every CTA of a cluster repeats the sampler's serial phases, and measured on
  // B200 (W=256, N=64) a 2-CTA cluster at one CTA/SM runs n_tau=256 at 24.7 TFLOP/s while 4-CTA clusters at two
  // CTAs/SM reach 20.6-22.0 TFLOP/s for n_tau=160..240 (profiles/r01e_cluster_plan.md).
  const size_t two = 113 * 1024, one = (size_t)device_smem_optin();
  const int cands[3] = {1, 2, 4};
  for (int i = 0; i < 3; ++i) {
    const size_t smem = other_bytes + rc_eval_doubles(d, rows_pad, cands[i]) * 8;
    if (smem <= two) { *out = {cands[i], true, smem}; return BISIP_OK; }
    if (smem <= one) { *out = {cands[i], false, smem}; return BISIP_OK; }
  }
  return fail(BISIP_ERR_UNSUPPORTED, "Decomp: n_tau x n_freq too large for a 4-CTA cluster's shared memory");
}
// the clustered ("rc") layout serves every mma.sync reduced-precision run and every FP64 run with n_tau > 64
inline bool use_rc(const bisip_model_desc& d) {
  return d.model == BISIP_MODEL_DECOMP && d.precision != BISIP_PREC_FP64_COLLAPSED &&
         (d.n_tau > 64 || d.precision != BISIP_PREC_FP64);
}

// tcgen05 path (decomp_umma.cuh): BISIP_PREC_TF32 / _3XTF32 whenever one M = 128 tile holds a half-step
// (rows <= 128), 2N <= 128 columns, and the B planes fit in shared memory next to `other_bytes`.
// n_tau <= 64: 256 tensor-memory columns per CTA, two CTAs per SM — the request is padded so that a third CTA
// (which would spin in tcgen05.alloc) never becomes resident.  n_tau > 64: 512 columns, so the request is padded
// past half an SM's shared memory and exactly one CTA is resident.
struct UmmaPlan { bool ok; bool two_per_sm; size_t smem; bool cluster; };
inline UmmaPlan plan_umma(const bisip_model_desc& d, size_t other_bytes, int rows, bool allow_cluster = false) {
  UmmaPlan pl{false, false, 0, false};
  const int planes = prec_planes(d.precision);
  if (d.model != BISIP_MODEL_DECOMP || (d.precision != BISIP_PREC_TF32 && d.precision != BISIP_PREC_3XTF32)) return pl;
  if (rows > kUmmaRows || !DecompUmmaShape::fits(d.n_freq, d.n_tau)) return pl;
  const DecompUmmaShape sh(d.n_freq, d.n_tau, d.n_coef);
  size_t smem = other_bytes + decomp_umma_smem_doubles(sh, planes) * 8;
  if (smem > (size_t)device_smem_optin()) {
    // K planes too large for one CTA: a 2-CTA cluster splits the real | imaginary columns (sampler kernel only)
    if (!allow_cluster) return pl;
    const DecompUmmaShape shc(d.n_freq, d.n_tau, d.n_coef, 1, 0);
    smem = other_bytes + decomp_umma_smem_doubles(shc, planes) * 8;
    if (smem > (size_t)device_smem_optin()) return pl;
    pl.ok = true;
    pl.cluster = true;
    pl.smem = smem < 116 * 1024 ? 116 * 1024 : smem;      // 512 tensor-memory columns: one CTA per SM
    return pl;
  }
  pl.ok = true;
  pl.two_per_sm = sh.nchunks == 1 && smem <= 113 * 1024;
  const size_t floor_bytes = pl.two_per_sm ? 77 * 1024 : 116 * 1024;
  pl.smem = smem < floor_bytes ? floor_bytes : smem;
  return pl;
}

// per-proposal constants of the vector-model kernel that the launchers pick
inline int vec_row_consts(const bisip_model_desc& d) {
  switch (d.model) {
    case BISIP_MODEL_DIAS: return DiasRow::kRC;
    case BISIP_MODEL_SHIN: return ShinRow::kRC;
    default:
      switch (d.n_modes) {
        case 1: return ColeColeRowT<1>::kRC;
        case 2: return ColeColeRowT<2>::kRC;
        case 3: return ColeColeRowT<3>::kRC;
        case 4: return ColeColeRowT<4>::kRC;
        default: return d.n_modes <= 8 ? ColeColeRow::kRC : ColeColeRowBig::kRC;
      }
  }
}

// ---- launchers, one translation unit per kernel family --------------------------------------------------------------
int launch_ens_dmma(const EnsembleParams& P, dim3 grid, size_t smem, cudaStream_t st);                       // ens_dmma.cu
int launch_ens_rc(const EnsembleParams& P, dim3 grid, const RcPlan& plan, cudaStream_t st);                  // ens_rc.cu
int launch_ens_umma(const EnsembleParams& P, dim3 grid, const UmmaPlan& plan, cudaStream_t st);              // ens_umma.cu
int launch_ens_collapsed(const EnsembleParams& P, dim3 grid, size_t smem, cudaStream_t st);                  // ens_collapsed.cu
int launch_ens_colecole(const EnsembleParams& P, dim3 grid, size_t smem, cudaStream_t st);                   // ens_colecole.cu
int launch_ens_dias_shin(const EnsembleParams& P, dim3 grid, size_t smem, cudaStream_t st);                  // ens_dias_shin.cu
int launch_ens_wp_collapsed(const EnsembleParams& P, dim3 grid, cudaStream_t st);                            // ens_wp_collapsed.cu
int launch_ens_wp_dmma(const EnsembleParams& P, dim3 grid, cudaStream_t st);                                 // ens_wp_dmma.cu
int launch_ens_wp_vec(const EnsembleParams& P, dim3 grid, cudaStream_t st);                                  // ens_wp_vec.cu
int run_batch_decomp(const BatchParams& P, bool want_z, cudaStream_t st);                                    // batch_decomp.cu
int run_batch_vec(const BatchParams& P, bool want_z, cudaStream_t st);                                       // batch_vec.cu

}  // namespace bisip
