// Integrated autocorrelation time of every column of data[B][n][W][ncol] (a kept chain: n steps x W walkers x ncol
// parameters per spectrum): emcee's estimator (autocorr.integrated_time, reached through sampler.get_autocorr_time,
// reference models.py:154-159), the same one sampler.integrated_time / integrated_time_batch compute with FFTs:
//   x_w(t)   = walker w's series centred on its own mean
//   acf_w(L) = sum_{t < n-L} x_w(t) x_w(t+L)                (the zero-padded linear ACF, as direct sums)
//   rho(L)   = (1/W) sum_w acf_w(L) / acf_w(0)              (normalised per walker, then averaged)
//   tau(L)   = 2 sum_{l <= L} rho(l) - 1
// and the result is tau(window), window = emcee's _auto_window: the first L with !(L < c tau(L)).  Where every lag
// passes (which needs c tau(n-1) > n-1; tau(n-1) is 0 in exact arithmetic) emcee's argmin picks lag 0.
//
// For a centred series sum_L acf(L) = acf(0)/2, so the window always closes, usually after a few tau.  The CTA therefore
// works through the lags in chunks of kAcfChunk and stops after the chunk in which the window closed: the work is
// W x n x (lags up to the window), not W x n^2.
//
// One CTA per (column, spectrum), as column_stats_smem_kernel: the ncol CTAs of a spectrum read the same sectors
// together.  The column goes to shared memory in its natural [t][w] order (lanes on consecutive walkers: conflict-free)
// and is centred there.  A thread owns one walker and kAcfLags consecutive lags and slides a register window over t,
// so each shared-memory load feeds kAcfLags / 2 FMAs.  Columns longer than shared memory run the same arithmetic on
// strided global loads (centred on the fly), so both paths give the same bits.  Walker averages are fixed-order
// reductions (no atomics): the result of a column depends on that column only, never on batch composition.
#pragma once
#include "common.cuh"

namespace bisip {

constexpr int kAcfThreads = 512;
constexpr int kAcfLags = 8;                                    // lags per thread (register window)
constexpr int kAcfGroups = 2;                                  // lag groups per chunk
constexpr int kAcfChunk = kAcfGroups * kAcfLags;               // lags per chunk
constexpr int kAcfGroupThreads = kAcfThreads / kAcfGroups;     // threads (walker slots) per lag group
constexpr int kAcfLoadUnroll = 16;                             // independent loads in flight per thread
static_assert(kAcfGroupThreads % 32 == 0, "a lag group is whole warps");

struct AutocorrParams {
  const double* data;
  int B, n, W, ncol;
  double c;
  double* tau_out;   // [B][ncol]
};

// dynamic shared memory: the centred column [n][W] (shared-memory path only), then mean[W] and acf0[W]
__host__ __device__ inline size_t autocorr_smem_bytes(long long n, int W, bool column) {
  return ((column ? (size_t)n * W : 0) + 2 * (size_t)W) * 8;
}
constexpr size_t kAcfStaticSmem = 2048;   // upper bound of the kernel's static shared memory (red + flags)

template <bool SMEM>
__global__ void __launch_bounds__(kAcfThreads, 1) autocorr_kernel(const AutocorrParams P) {
  extern __shared__ __align__(16) unsigned char acf_dyn[];
  __shared__ double red[kAcfGroups][kAcfGroupThreads / 32][kAcfLags];
  __shared__ double s_rho[kAcfChunk];
  __shared__ double s_tau;
  __shared__ int s_done;
  const int col = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int n = P.n, W = P.W;
  const size_t nw = (size_t)n * W;
  double* vals = reinterpret_cast<double*>(acf_dyn);           // SMEM: [n][W]
  double* mean = vals + (SMEM ? nw : 0);
  double* acf0 = mean + W;
  const double* src = P.data + (size_t)b * nw * P.ncol + col;

  if (SMEM) {
    for (size_t i0 = tid; i0 < nw; i0 += (size_t)kAcfThreads * kAcfLoadUnroll) {
      double v[kAcfLoadUnroll];
#pragma unroll
      for (int u = 0; u < kAcfLoadUnroll; ++u) {
        const size_t i = i0 + (size_t)u * kAcfThreads;
        v[u] = i < nw ? __ldg(src + i * P.ncol) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < kAcfLoadUnroll; ++u) {
        const size_t i = i0 + (size_t)u * kAcfThreads;
        if (i < nw) vals[i] = v[u];
      }
    }
    __syncthreads();
  }
  // value of walker w at step t, centred (SMEM: centred in place below)
  auto at = [&](int t, int w) -> double {
    if (SMEM) return vals[t * W + w];                           // n W < 2^28 on this path
    return __ldg(src + ((size_t)t * W + w) * P.ncol) - mean[w];
  };
  // per walker, sequentially in t: mean (np.mean: sum / n), centring, acf(0)
  for (int w = tid; w < W; w += kAcfThreads) {
    double s = 0.0;
    for (int t = 0; t < n; ++t) s += SMEM ? vals[(size_t)t * W + w] : __ldg(src + ((size_t)t * W + w) * P.ncol);
    const double m = s / (double)n;
    mean[w] = m;
    double a0 = 0.0;
    for (int t = 0; t < n; ++t) {
      double x;
      if (SMEM) {
        x = vals[(size_t)t * W + w] - m;
        vals[(size_t)t * W + w] = x;
      } else {
        x = __ldg(src + ((size_t)t * W + w) * P.ncol) - m;
      }
      a0 = fma(x, x, a0);
    }
    acf0[w] = a0;
  }
  if (tid == 0) { s_done = 0; s_tau = 0.0; }
  __syncthreads();

  const int g = tid / kAcfGroupThreads, slot = tid % kAcfGroupThreads;
  const int warp_in_group = slot >> 5, lane = tid & 31;
  double cum = 0.0, tau0 = 0.0;                                // thread 0's running sum and tau(0)
  for (int base = 0; base < n; base += kAcfChunk) {
    const int L0 = base + g * kAcfLags;
    double rs[kAcfLags];
#pragma unroll
    for (int j = 0; j < kAcfLags; ++j) rs[j] = 0.0;
    if (L0 < n) {
      for (int w = slot; w < W; w += kAcfGroupThreads) {
        // acc[j] = sum_t x(t) x(t + L0 + j), t ascending, in blocks of kAcfLags steps: win[] holds x(t0 + L0 + j),
        // nxt[] the next kAcfLags values; values past the end are 0, so the padded steps add exact zeros
        double acc[kAcfLags], win[kAcfLags];
#pragma unroll
        for (int j = 0; j < kAcfLags; ++j) {
          acc[j] = 0.0;
          win[j] = L0 + j < n ? at(L0 + j, w) : 0.0;
        }
        const int tmax = n - L0;                              // t < n - L0 for the group's first lag
        for (int t0 = 0; t0 < tmax; t0 += kAcfLags) {
          double xs[kAcfLags], nxt[kAcfLags];
#pragma unroll
          for (int s = 0; s < kAcfLags; ++s) {
            xs[s] = t0 + s < n ? at(t0 + s, w) : 0.0;
            const int i = t0 + L0 + kAcfLags + s;
            nxt[s] = i < n ? at(i, w) : 0.0;
          }
#pragma unroll
          for (int s = 0; s < kAcfLags; ++s)
#pragma unroll
            for (int j = 0; j < kAcfLags; ++j)
              acc[j] = fma(xs[s], s + j < kAcfLags ? win[s + j] : nxt[s + j - kAcfLags], acc[j]);
#pragma unroll
          for (int j = 0; j < kAcfLags; ++j) win[j] = nxt[j];
        }
        const double a0 = acf0[w];
#pragma unroll
        for (int j = 0; j < kAcfLags; ++j) rs[j] += acc[j] / a0;
      }
    }
    // sum over the walkers of the group: lanes by xor-shuffle, then the warps in index order
#pragma unroll
    for (int j = 0; j < kAcfLags; ++j) {
      double v = rs[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[g][warp_in_group][j] = v;
    }
    __syncthreads();
    if (tid < kAcfChunk) {
      double s = 0.0;
      for (int q = 0; q < kAcfGroupThreads / 32; ++q) s += red[tid / kAcfLags][q][tid % kAcfLags];
      s_rho[tid] = s / (double)W;
    }
    __syncthreads();
    if (tid == 0) {                                            // the cumulative sum in lag order, the window test
      for (int k = 0; k < kAcfChunk && !s_done; ++k) {
        const int L = base + k;
        cum += s_rho[k];
        const double tau = 2.0 * cum - 1.0;
        if (L == 0) tau0 = tau;
        if (!((double)L < P.c * tau)) { s_tau = tau; s_done = 1; }
        else if (L == n - 1) { s_tau = tau0; s_done = 1; }
      }
    }
    __syncthreads();
    if (s_done) break;
  }
  if (tid == 0) P.tau_out[(size_t)b * P.ncol + col] = s_tau;
}

}  // namespace bisip
