// Reduced-precision decomposition on the 5th-generation tensor cores (tcgen05 / TMEM), the Blackwell-native
// form of the "TF32 / 3xTF32 variant" of north_star (BASELINE config 4 compares it with FP64 DMMA).
// Both contractions of the two-stage forward run as tcgen05.mma.cta_group::1.kind::tf32 with M = 128: the
// <= 128 proposals of one half-step of one spectrum are ONE tile, operands and accumulators live in TENSOR MEMORY.
//
//   stage 1  M[row][k] = R0 sum_i a[row][i] L[i][k].  The power table L (log_tau^i) is badly conditioned, so at
//            init its rows are orthonormalised once per spectrum in FP64 (modified Gram-Schmidt, two passes):
//            L = R^T Q.  Per proposal only b = R (R0 a) is FP64 (<= 36 FMAs); b is split exactly into three TF32
//            planes and stored to tensor memory (tcgen05.st, lane = row), Q is held in shared memory as three TF32
//            planes, and M = b Q is six K = 8 MMAs (all plane products above 2^-33) with FP32 accumulation:
//            |b_j q_jk| <= rms(M), nothing cancels any more, M is FP32-accurate.
//   stage 2  D[128][NC] = M x (K / sigma).  M is read back (tcgen05.ld), split into TF32 hi / lo planes and stored
//            to tensor memory as the A operand; B = K/sigma sits in shared memory as hi / lo planes in the
//            canonical K-major no-swizzle core-matrix layout; PREC = 3 issues A_lo B_hi + A_hi B_lo + A_hi B_hi
//            ("3xTF32", 24 instructions per column block for 64 taus), PREC = 1 the hi product only.  One extra K
//            step (A from shared memory) adds the residual constants (y - R0 delta)/sigma, see kUmmaR0c below.
//            The real and the imaginary columns are two blocks with their own mbarriers: the epilogue of the first
//            runs under the MMAs of the second.
//   epilogue tcgen05.ld (lane = row: one thread owns a row, no shuffles): the accumulators ARE the weighted
//            residuals, chi^2 is their sum of squares (FP32 partial sums, combined in FP64).
//
// One elected lane of warp 7 issues every MMA from the uniform datapath (tcgen05.commit only tracks the issuing
// thread's instructions); completion arrives on mbarriers.  Tensor memory per CTA: 128 accumulator columns + 128
// operand columns = 256, so two CTAs share an SM's 512 (the stage-1 result aliases the accumulator columns, the b
// planes alias the A columns).  n_tau > 64 runs in 64-tau chunks with separate stage-1 columns (512 columns, one CTA
// per SM; api.cu guarantees it); when the K planes exceed one CTA's shared memory a 2-CTA cluster splits the real |
// imaginary columns and exchanges the partial chi^2 through distributed shared memory (cluster mode).
// Polling the mbarriers from one warp per group (the others parked in a hardware barrier) was measured: no change.
// The operand conventions (descriptor fields, A-in-TMEM layout) are pinned on hardware by tools/umma_probe.cu.
// Restates reference Decomp_cyth (cython_funcs.pyx:75-94) + _log_likelihood (models.py:59-62) at TF32 precision.
#pragma once
#include "decomp_eval.cuh"
#include "decomp_rc.cuh"   // cooperative-groups cluster handle (cg::)

namespace bisip {

static_assert(kThreads == 256, "decomp_umma.cuh maps 256 threads onto 128 TMEM lanes x 2 halves");
#ifdef BISIP_PHASE_TIMING
#define UMMA_T0 long long ut_ = clock64();
#define UMMA_MARK(i) { long long n_ = clock64(); s.ph[i] += n_ - ut_; ut_ = n_; }
#else
#define UMMA_T0
#define UMMA_MARK(i)
#endif
constexpr int kUmmaRows = 128;      // MMA M: proposals per tile (>= rows of a half-step: W <= 256)
constexpr int kUmmaChunk = 64;      // taus per A buffer
// The residual constant (y - R0 delta)/sigma is produced by the tensor core as well: expanded about R0 = kUmmaR0c,
//   (y - R0 delta)/sigma = c0 - dR0 g,   c0 = (y - kUmmaR0c delta)/sigma,  g = delta/sigma,  dR0 = R0 - kUmmaR0c,
// it is one extra K step of 8 products  [1, 1, 1, -d_hi, -d_hi, -d_mid, -d_mid, -d_lo] x [c0_hi, c0_mid, c0_lo, g_hi,
// g_mid, g_hi, g_mid, g_hi]  (three-way TF32 splits: c0 enters exactly to 2^-33, the product to ~2^-22 of |dR0 g|)
// that initialises the accumulators, so the epilogue is a bare sum of squares.  BISIP normalises every spectrum by
// max|Z| (utils.py:138-142) and bounds r0 to [0.9, 1.1] (models.py:212): |dR0| <= 0.1 and the dropped cross terms
// (~2e-6 for sigma = 1 %) stay below the FP32 accumulators' own rounding of the O(10-50) partial sums.
constexpr double kUmmaR0c = 1.0;

struct DecompUmmaShape {
  int N, S, D;
  int NCH;     // columns per part (real | imag), multiple of 16
  int NC;      // columns held by this CTA = stage-2 MMA N: 2 NCH, or NCH when a 2-CTA cluster splits real | imag
  int cl;      // 1: cluster mode (K planes too large for one CTA): CTA `part` of the pair owns the real (0) or imaginary (1) columns
  int part;
  int SP;      // taus padded to a multiple of 8 (stage-2 K steps)
  int SQ;      // taus padded to a multiple of 16 (stage-1 MMA N)
  int nchunks; // chunks of <= 64 taus
  __host__ __device__ DecompUmmaShape(int n, int s, int d, int cluster = 0, int rank = 0)
      : N(n), S(s), D(d), NCH(ceil_div(n, 16) * 16), NC((cluster ? 1 : 2) * ceil_div(n, 16) * 16), cl(cluster), part(rank),
        SP(ceil_div(s, 8) * 8),
        SQ(ceil_div(s, 16) * 16), nchunks(ceil_div(ceil_div(s, 8) * 8, kUmmaChunk)) {}
  __host__ __device__ size_t plane_bytes() const { return (size_t)NC * SP * 4; }    // K/sigma lo plane
  // hi plane: one more K step of 8 columns holding the residual constants (see the epilogue note below)
  __host__ __device__ size_t hiplane_bytes() const { return (size_t)NC * (SP + 8) * 4; }
  __host__ __device__ size_t lk_bytes() const { return SQ * 64 > 4096 ? (size_t)SQ * 64 : 4096; }   // also holds A_ext (4 KB)
  __host__ __device__ size_t qplane_bytes() const { return (size_t)SQ * 32; }       // one Q plane: SQ taus x 8 coefficients
  __host__ __device__ int tmem_cols() const { return nchunks > 1 ? 512 : 256; }
  __host__ __device__ static bool fits(int n_freq, int n_tau) { return n_freq <= 64 && n_tau <= 512; }
};

// Shared-memory block of the evaluator.  Only the base pointer is kept (the sampler kernel is register-bound at two
// CTAs per SM); the sub-arrays are addressed by offsets recomputed from the shape:
//   Bhi  [NC x (SP + 8)] TF32, canonical K-major core matrices (8 columns x 16 bytes); K step SP/8 = residual constants
//   Blo  [NC x SP] the low plane (PREC == 3)
//   Q    [3][SQ x 8] TF32 planes of the orthonormalised tau basis (stage-1 B operand)
//   Lk   [SQ][8] doubles: init scratch, log_tau powers per tau, orthonormalised in place; afterwards its first 4 KB
//        hold A_ext [128 rows x 8] TF32, the per-proposal A operand of the residual-constant K step
//   R    [8][8] doubles:  L_i = sum_{j<=i} R[i][j] q_j
//   part [128] doubles: partial chi^2 of the second thread half;  xsum [2][128] (cluster mode): this CTA's chi^2 for the peer
//   bar  [5] mbarriers (stage-1 MMAs, column blocks of the stage-2 MMAs; 3 in use);  tmem: base address from tcgen05.alloc
struct DecompUmmaSmem {
  uint8_t* p0;        // 128-byte aligned start (= Bhi)
  double llconst;
  uint32_t tbase;
  uint32_t phase;     // bit i: parity of the next completion of bar[i]; bit 8: buffer of the cluster exchange
#ifdef BISIP_PHASE_TIMING
  long long ph[8];    // per-thread cycle counters of the evaluation sub-phases (registers)
#endif
};
struct DecompUmmaOff {
  uint32_t Blo, Q, Lk, R, part, xsum, bar, tmem;
  template <int PREC>
  static __device__ __forceinline__ DecompUmmaOff make(const DecompUmmaShape& sh) {
    DecompUmmaOff o;
    o.Blo = (uint32_t)sh.hiplane_bytes();
    o.Q = o.Blo + (PREC == 3 ? (uint32_t)sh.plane_bytes() : 0u);
    o.Lk = o.Q + 3u * (uint32_t)sh.qplane_bytes();
    o.R = o.Lk + (uint32_t)sh.lk_bytes();
    o.part = o.R + 512u;
    o.xsum = o.part + kUmmaRows * 8u;
    o.bar = o.xsum + (sh.cl ? 2u * kUmmaRows * 8u : 0u);
    o.tmem = o.bar + 40u;
    return o;
  }
};

__host__ __device__ inline size_t decomp_umma_smem_doubles(const DecompUmmaShape& sh, int prec) {
  const size_t planes = prec == 3 ? 2 : 1;
  return 16 + (sh.hiplane_bytes() + (planes - 1) * sh.plane_bytes() + 3 * sh.qplane_bytes() + sh.lk_bytes()) / 8 + 64 +
         kUmmaRows + (sh.cl ? 2 * kUmmaRows : 0) + 8;
}

template <int PREC>
__device__ inline double* decomp_umma_carve(DecompUmmaSmem& s, double* base, const DecompUmmaShape& sh) {
  s.p0 = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(base) + 127) & ~uintptr_t(127));
  s.phase = 0;
#ifdef BISIP_PHASE_TIMING
  for (int i = 0; i < 8; ++i) s.ph[i] = 0;
#endif
  return base + decomp_umma_smem_doubles(sh, PREC);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Canonical K-major no-swizzle operand tile: core matrix = 8 rows x 16 bytes (4 TF32), 128 contiguous bytes;
// K-adjacent core matrices contiguous (LBO = 128 B), row-group-adjacent ones `sbo` bytes apart.
//   K/sigma plane: rows = frequency columns n, K = taus:  sbo = 32 SP
//   Q plane:       rows = taus,               K = 8 coefficients: sbo = 256
__device__ __forceinline__ int umma_tile_off(int row, int k, int sbo) {
  return (row & 7) * 16 + (row >> 3) * sbo + (k >> 2) * 128 + (k & 3) * 4;
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, int sbo) {
  return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)((sbo >> 4) & 0x3fff) << 32) |
         ((uint64_t)1 << 46);     // version 1, no swizzle, base offset 0
}
// instruction descriptor: D = F32, A = B = TF32, both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t umma_idesc(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kUmmaRows >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32_ts(uint32_t tD, uint32_t tA, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tD), "r"(tA), "l"(bdesc), "r"(idesc),
      "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_ss(uint32_t tD, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tD), "l"(adesc), "l"(bdesc), "r"(idesc),
      "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar_saddr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_saddr) : "memory");
}
// one lane of a converged warp (warp-uniform call site): lets the compiler keep the MMA operands in uniform registers
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// suspend-time hint of mbarrier.try_wait: the waiting warps sleep instead of re-issuing the poll (the polls were 5 % of
// all issued instructions of the sampler kernel)
constexpr uint32_t kUmmaWaitHintNs = 2000;
__device__ __forceinline__ void mbar_wait(uint32_t baddr, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(baddr), "r"(parity), "r"(kUmmaWaitHintNs) : "memory");
  }
}

// round-to-nearest TF32 image of an FP32 value (magnitude + half ulp, masked: cvt.rna without inf / nan handling)
__device__ __forceinline__ uint32_t tf32_rn(float x) { return (__float_as_uint(x) + 0x1000u) & 0xffffe000u; }

// three-way TF32 split of a double (33 mantissa bits): x = hi + mid + lo + O(2^-33 |x|).  The double is first
// written as two floats (the only FP64 <-> FP32 conversions, which are slow); the rest is exact FP32 arithmetic.
__device__ __forceinline__ void split3_tf32(double x, uint32_t& hi, uint32_t& mid, uint32_t& lo) {
  const float xh = (float)x;
  const float xl = (float)(x - (double)xh);
  hi = tf32_rn(xh);
  const float r1 = xh - __uint_as_float(hi);          // exact: <= 13 significant bits
  mid = tf32_rn(r1);
  lo = tf32_rn((r1 - __uint_as_float(mid)) + xl);
}
// two-way split of an FP32 value (22 bits).  The re-pack of M runs this on 64 values per proposal and half-step: it was
// 20 % of all instructions of the 3xTF32 sampler kernel, most of them integer (half rate on B200).  Three splits were
// compared; split2_tf32 is variant 1:
//   0  hi = rn(x), lo = rn(x - hi)                      5 instructions (round 1)
//   1  hi = rn(x), lo = x - hi left in FP32            3: the tensor core ignores the low 13 mantissa bits of a tf32
//                                                         operand, i.e. truncates lo itself
//   2  hi = x with the low 13 bits cleared, lo = x - hi  2: truncation on both levels
// Measured (profiles/r02d_barriers.md): forward error of 3xTF32 8.3e-8 / 8.4e-8 / 1.2e-7, sampler 6.53e9 / 6.62e9 / 6.58e9
// evals/s for 0 / 1 / 2; variant 2 also truncates the only plane of plain TF32 (5.6e-5 -> 1.9e-4), so 1 it is.
__device__ __forceinline__ void split2_tf32_rn(float x, uint32_t& hi, uint32_t& lo) {      // init-time planes: always rounded
  hi = tf32_rn(x);
  lo = tf32_rn(x - __uint_as_float(hi));
}
__device__ __forceinline__ void split2_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = tf32_rn(x);
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// Per-spectrum constants; allocates tensor memory.  All threads; ends with __syncthreads().
template <int PREC>
__device__ inline void decomp_umma_init(DecompUmmaSmem& s, const DecompUmmaShape& sh, double c_exp,
                                        const double* __restrict__ w, const double* __restrict__ taus,
                                        const double* __restrict__ log_taus, const double* __restrict__ y,
                                        const double* __restrict__ yerr, double* red) {
  const int tid = threadIdx.x, lane = tid & 31;
  const int N = sh.N, S = sh.S, SP = sh.SP, NCH = sh.NCH, D = sh.D;
  const DecompUmmaOff o = DecompUmmaOff::make<PREC>(sh);
  struct { uint8_t *Bhi, *Blo, *Q; double *Lk, *R; uint64_t* bar; uint32_t* tmem; } l;
  l.Bhi = s.p0; l.Blo = s.p0 + o.Blo; l.Q = s.p0 + o.Q;
  l.Lk = reinterpret_cast<double*>(s.p0 + o.Lk); l.R = reinterpret_cast<double*>(s.p0 + o.R);
  l.bar = reinterpret_cast<uint64_t*>(s.p0 + o.bar); l.tmem = reinterpret_cast<uint32_t*>(s.p0 + o.tmem);
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(l.tmem)), "r"(sh.tmem_cols())
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 32) {
    for (int i = 0; i < 5; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(l.bar + i)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {
    uint32_t* z = reinterpret_cast<uint32_t*>(l.Bhi);      // K/sigma planes and the Q planes are contiguous
    const int nw = (int)(o.Lk / 4);
    for (int i = tid; i < nw; i += kThreads) z[i] = 0u;
  }
  for (int i = tid; i < sh.SQ * 8; i += kThreads) {
    const int k = i >> 3, p = i & 7;
    l.Lk[i] = (p < D && k < S) ? log_taus[(size_t)p * S + k] : 0.0;
  }
  if (tid < 64) l.R[tid] = 0.0;
  const bool scaled = (y != nullptr);
  double csum = 0.0;
  for (int c = tid; c < 2 * N; c += kThreads)
    if (scaled) csum += 2.0 * log(yerr[c] * yerr[c]);
  __syncthreads();
  // ---- warp 0: orthonormalise the D rows of the tau table in place (modified Gram-Schmidt, every projection twice);
  //      the other warps build the K/sigma planes meanwhile -----------------------------------------------------
  if (tid < 32) {
    for (int i = 0; i < D; ++i) {
      for (int pass = 0; pass < 2; ++pass)
        for (int j = 0; j < i; ++j) {
          double dot = 0.0;
          for (int k = lane; k < S; k += 32) dot = fma(l.Lk[k * 8 + j], l.Lk[k * 8 + i], dot);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
          for (int k = lane; k < S; k += 32) l.Lk[k * 8 + i] = fma(-dot, l.Lk[k * 8 + j], l.Lk[k * 8 + i]);
          if (lane == 0) l.R[i * 8 + j] += dot;
          __syncwarp();
        }
      double nn = 0.0;
      for (int k = lane; k < S; k += 32) nn = fma(l.Lk[k * 8 + i], l.Lk[k * 8 + i], nn);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) nn += __shfl_xor_sync(0xffffffffu, nn, o);
      const double nrm = sqrt(nn);
      const double inv = nrm > 1e-290 ? 1.0 / nrm : 0.0;       // a dependent row contributes nothing new
      for (int k = lane; k < S; k += 32) l.Lk[k * 8 + i] *= inv;
      if (lane == 0) l.R[i * 8 + i] = inv != 0.0 ? nrm : 0.0;
      __syncwarp();
    }
  } else {
    const int sbo_hi = 32 * (SP + 8);
    // residual constants: K step SP/8 of the hi plane, column n: [c0_hi, c0_mid, c0_lo, g_hi, g_mid, g_hi, g_mid, g_hi]
    for (int n = tid - 32; n < sh.NC; n += kThreads - 32) {
      const int part = sh.cl ? sh.part : (n >= NCH), j = sh.cl ? n : n - part * NCH;
      double c0 = 0.0, g = 0.0;
      if (j < N && scaled) {
        const double is = 1.0 / yerr[part * N + j];
        g = part ? 0.0 : is;
        c0 = y[part * N + j] * is - kUmmaR0c * g;
      }
      uint32_t c[3], q[3];
      split3_tf32(c0, c[0], c[1], c[2]);
      split3_tf32(g, q[0], q[1], q[2]);
      const uint32_t ext[8] = {c[0], c[1], c[2], q[0], q[1], q[0], q[1], q[0]};
      for (int e = 0; e < 8; ++e) *reinterpret_cast<uint32_t*>(l.Bhi + umma_tile_off(n, SP + e, sbo_hi)) = ext[e];
    }
    double cs, sn;
    sincospi(0.5 * c_exp, &sn, &cs);
    for (int i = tid - 32; i < S * N; i += kThreads - 32) {
      const int k = i / N, j = i - k * N;
      double kre, kim;
      debye_kernel_term(w[j], taus[k], c_exp, cs, sn, kre, kim);
      if (scaled) {
        kre *= 1.0 / yerr[j];
        kim *= 1.0 / yerr[N + j];
      }
      uint32_t hi, lo;
      if (!sh.cl || sh.part == 0) {
        split2_tf32_rn((float)kre, hi, lo);
        *reinterpret_cast<uint32_t*>(l.Bhi + umma_tile_off(j, k, sbo_hi)) = hi;
        if (PREC == 3) *reinterpret_cast<uint32_t*>(l.Blo + umma_tile_off(j, k, 32 * SP)) = lo;
      }
      if (!sh.cl || sh.part == 1) {
        const int n = sh.cl ? j : NCH + j;
        split2_tf32_rn((float)kim, hi, lo);
        *reinterpret_cast<uint32_t*>(l.Bhi + umma_tile_off(n, k, sbo_hi)) = hi;
        if (PREC == 3) *reinterpret_cast<uint32_t*>(l.Blo + umma_tile_off(n, k, 32 * SP)) = lo;
      }
    }
  }
  __syncthreads();
  for (int i = tid; i < S * D; i += kThreads) {             // Q planes: row = tau, K = coefficient
    const int k = i / D, p = i - k * D;
    uint32_t q0, q1, q2;
    split3_tf32(l.Lk[k * 8 + p], q0, q1, q2);
    const int off = umma_tile_off(k, p, 256);
    *reinterpret_cast<uint32_t*>(l.Q + off) = q0;
    *reinterpret_cast<uint32_t*>(l.Q + sh.qplane_bytes() + off) = q1;
    *reinterpret_cast<uint32_t*>(l.Q + 2 * sh.qplane_bytes() + off) = q2;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) csum += __shfl_xor_sync(0xffffffffu, csum, o);
  if ((tid & 31) == 0) red[tid >> 5] = csum;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // operand planes -> visible to the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  double tot = 0.0;
  for (int i = 0; i < kWarps; ++i) tot += red[i];
  s.llconst = tot;
  s.tbase = *l.tmem;
  __syncthreads();
}

// All TMEM traffic of this CTA is complete (callers end their last evaluation with a barrier).
__device__ inline void decomp_umma_release(DecompUmmaSmem& s, const DecompUmmaShape& sh) {
#ifdef BISIP_PHASE_TIMING
  if (blockIdx.x == 0 && threadIdx.x == 0 && gridDim.y == 1 && s.ph[2] + s.ph[4] > 100000)
    printf("umma eval cycles (thread 0, whole run): b=R.a %lld  split+st %lld  wait-st+barrier %lld | mma1-wait %lld  repack+barrier %lld  "
           "mma2-issue(warp 7 only) %lld  mma2-wait+epilogue %lld  tail %lld\n", s.ph[6], s.ph[7], s.ph[0], s.ph[1], s.ph[2], s.ph[3], s.ph[4], s.ph[5]);
#endif
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s.tbase), "r"(sh.tmem_cols()) : "memory");
}

// Evaluate nrows <= 128 proposals.  WANT_Z = false: chi[q] = sum_c ((y_c - Z_c)/sigma_c)^2 (caller barriers
// before reading); WANT_Z = true: Zout[q][2][N] (forward only; init was called with y == nullptr).
// 256 threads: thread = (row r = tid & 127, half h = tid >> 7); h splits the tau groups when M is re-packed and the
// real | imaginary columns in the epilogue.  Warp w may touch TMEM lanes [32 (w & 3), +32) only — exactly its rows.
template <int PREC, bool WANT_Z>
__device__ inline void decomp_umma_eval(DecompUmmaSmem& s, const DecompUmmaShape& sh, const double* __restrict__ prop,
                                        int ndim, int nrows, double* __restrict__ chi, double* __restrict__ Zout) {
  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);               // warp-uniform by construction
  const int r = tid & (kUmmaRows - 1), h = warp >> 2;
  const uint32_t lane_base = (uint32_t)(32 * (warp & 3)) << 16;
  const bool warp_live = 32 * (warp & 3) < nrows;
  const uint32_t tbase = __shfl_sync(0xffffffffu, s.tbase, 0);
  const bool chunked = sh.nchunks > 1;
  const uint32_t tD = tbase, tA = tbase + 128;                          // accumulators | A planes: hi at tA, lo at tA + 64
  const uint32_t tM = chunked ? tbase + 256 : tbase;                    // stage-1 result (aliases D when there is one chunk)
  const uint32_t tB = chunked ? tbase + 320 : tbase + 128;              // b planes: 3 x 8 columns (alias A when one chunk)
  const DecompUmmaOff o = DecompUmmaOff::make<PREC>(sh);
  const uint32_t sb = smem_u32(s.p0);
  const uint32_t barS = sb + o.bar, barD = barS + 8;
  UMMA_T0
  // ---- b = R (R0 a): the proposal in the orthonormal tau basis, three TF32 planes -> tensor memory ----------------
  double R0 = 0.0;
  if (warp_live) {
    double a[8], b[8];
    if (r < nrows) {
      const double* q = prop + (size_t)r * ndim;
      R0 = q[0];
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = (i < sh.D) ? R0 * q[1 + i] : 0.0;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = 0.0;
    }
    const uint32_t ra = sb + o.R;
#pragma unroll
    for (int j = 0; j < 8; ++j) b[j] = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i < sh.D) {
#pragma unroll
        for (int j = 0; j <= i; ++j) {
          double rij;
          asm volatile("ld.shared.f64 %0, [%1];" : "=d"(rij) : "r"(ra + (i * 8 + j) * 8));
          b[j] = fma(rij, a[i], b[j]);
        }
      }
    }
    UMMA_MARK(6)
    // half h converts and stores coefficients [4h, 4h+4) of all three planes (conversions dominate this phase)
    uint32_t p0[4], p1[4], p2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double bj = h ? b[4 + j] : b[j];
      p0[j] = p1[j] = p2[j] = 0u;
      if (4 * h + j < sh.D) split3_tf32(bj, p0[j], p1[j], p2[j]);
    }
    tmem_st4(tB + lane_base + 4 * h, p0);
    tmem_st4(tB + lane_base + 8 + 4 * h, p1);
    UMMA_MARK(7)
    tmem_st4(tB + lane_base + 16 + 4 * h, p2);
    if (h == 1) {     // A_ext row r = [1, 1, 1, -d_hi, -d_hi, -d_mid, -d_mid, -d_lo], d = R0 - kUmmaR0c (shared memory, SS-mode MMA)
      uint32_t d0, d1, d2;
      split3_tf32(r < nrows ? kUmmaR0c - R0 : 0.0, d0, d1, d2);
      const uint32_t ax = sb + o.Lk + (uint32_t)umma_tile_off(r, 0, 256);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(ax), "r"(0x3f800000u), "r"(0x3f800000u), "r"(0x3f800000u), "r"(d0) : "memory");
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(ax + 128u), "r"(d0), "r"(d1), "r"(d1), "r"(d2) : "memory");
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // A_ext -> visible to the tensor core
  tc_fence_before();
  __syncthreads();
  UMMA_MARK(0)
  // stage-2 column blocks: the real and the imaginary columns (N = NCH each).  Measured on B200 (C5 shape, 3xTF32):
  // one N = 128 block 5.36e9 evals/s, two blocks 6.00e9, four N = 32 blocks 5.11e9 (short instructions pay a fixed cost).
  const int nblk = sh.cl ? 1 : 2, bw = sh.NCH;
  const uint32_t idescb = umma_idesc(bw);
  const uint32_t q0a = sb + o.Q, qpb = (uint32_t)sh.qplane_bytes();
  for (int c = 0; c < sh.nchunks; ++c) {
    const int k0 = c * kUmmaChunk, kt = min(kUmmaChunk, sh.SP - k0);      // taus of this chunk (multiple of 8)
    const int nq = min(kUmmaChunk, sh.SQ - k0);                           // stage-1 N (multiple of 16)
    const int ng = kt >> 3;
    // ---- stage 1: M = b Q (six plane products, smallest first) -> tM.  Issued by the same lane as stage 2:
    //      tcgen05.commit only tracks the issuing thread's MMAs, and the wait below must also cover stage 2 of
    //      the previous chunk before its A planes are overwritten ------------------------------------------------------
    if (warp == 7) {
      tc_fence_after();
      if (elect_one()) {
        const uint32_t id1 = umma_idesc(nq);
        const uint64_t d0 = umma_desc(q0a + 32 * k0, 256), d1 = umma_desc(q0a + qpb + 32 * k0, 256),
                       d2 = umma_desc(q0a + 2 * qpb + 32 * k0, 256);
        umma_tf32_ts(tM, tB + 16, d0, id1, 0u);      // lo  x hi
        umma_tf32_ts(tM, tB, d2, id1, 1u);           // hi  x lo
        umma_tf32_ts(tM, tB + 8, d1, id1, 1u);       // mid x mid
        umma_tf32_ts(tM, tB + 8, d0, id1, 1u);       // mid x hi
        umma_tf32_ts(tM, tB, d1, id1, 1u);           // hi  x mid
        umma_tf32_ts(tM, tB, d0, id1, 1u);           // hi  x hi
        umma_commit(barS);
      }
      __syncwarp();
    }
    mbar_wait(barS, s.phase & 1u);
    s.phase ^= 1u;
    tc_fence_after();
    UMMA_MARK(1)
    // ---- re-pack: M (FP32, lane = row) -> TF32 hi / lo A planes; half h takes the 8-tau groups g = h, h+2, ... ------
    if (warp_live) {
      uint32_t m[4][8];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (h + 2 * i < ng) tmem_ld8(tM + lane_base + 8 * (h + 2 * i), m[i]);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (h + 2 * i < ng) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) split2_tf32(__uint_as_float(m[i][e]), hi[e], lo[e]);
          tmem_st8(tA + lane_base + 8 * (h + 2 * i), hi);
          if (PREC == 3) tmem_st8(tA + 64 + lane_base + 8 * (h + 2 * i), lo);
        }
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    UMMA_MARK(2)
    // ---- stage 2: D (+)= M (K/sigma); 256 bytes of each plane per K step of 8 taus.  The columns are issued as two
    //      blocks (real, imaginary), each committed to its own mbarrier, so the epilogue of the real block (half 0)
    //      runs under the MMAs of the imaginary one.  Warp 7 issues: it belongs to the half whose block finishes last.
    if (warp == 7) {
      tc_fence_after();
      if (elect_one()) {
        for (int blk = 0; blk < nblk; ++blk) {
          const int n0 = blk * sh.NCH;                                   // first column of the block
          const int sbo_hi = 32 * (sh.SP + 8), sbo_lo = 32 * sh.SP;
          const uint32_t rhi = (uint32_t)(n0 >> 3) * (uint32_t)sbo_hi, rlo = (uint32_t)(n0 >> 3) * (uint32_t)sbo_lo;
          const uint64_t dhi = umma_desc(sb + rhi + 32u * k0, sbo_hi), dlo = umma_desc(sb + o.Blo + rlo + 32u * k0, sbo_lo);
          // the residual constants initialise the accumulators (K step SP/8 of the hi plane x A_ext from shared memory)
          if (c == 0) umma_tf32_ss(tD + n0, umma_desc(sb + o.Lk, 256), umma_desc(sb + rhi + 32u * sh.SP, sbo_hi), idescb, 0u);
          if (PREC == 3) {
            for (int j = 0; j < ng; ++j) umma_tf32_ts(tD + n0, tA + 64 + 8 * j, dhi + 16u * j, idescb, 1u);
            for (int j = 0; j < ng; ++j) umma_tf32_ts(tD + n0, tA + 8 * j, dlo + 16u * j, idescb, 1u);
          }
          for (int j = 0; j < ng; ++j) umma_tf32_ts(tD + n0, tA + 8 * j, dhi + 16u * j, idescb, 1u);
          if (c + 1 == sh.nchunks) umma_commit(barD + 8 * blk);
        }
      }
      __syncwarp();
    }
  }
  UMMA_MARK(3)
  // ---- epilogue: D row r; half h owns column block h (columns [h NCH, (h+1) NCH)); in cluster mode the CTA has one
  //      block and the halves share it (when NCH/2 is still a multiple of the 16-column load) ---------------------------
  // The accumulators already hold the weighted residual (y - Z)/sigma (see kUmmaR0c): chi^2 is their sum of squares.
  double acc = 0.0;
  {
    const int blk = sh.cl ? 0 : h;
    const bool halves = sh.cl && (sh.NCH & 31) == 0;
    const int cw = !sh.cl ? sh.NCH : (halves ? sh.NCH / 2 : (h == 0 ? sh.NCH : 0));      // columns of this thread
    const int cfirst = !sh.cl ? h * sh.NCH : (halves ? h * (sh.NCH / 2) : 0);
    mbar_wait(barD + 8 * blk, (s.phase >> (1 + blk)) & 1u);
    s.phase ^= 2u << blk;
    tc_fence_after();
    float ch[4] = {0.f, 0.f, 0.f, 0.f};
    if (warp_live) {
      const uint32_t td = tD + lane_base + (uint32_t)cfirst;
      for (int c0 = 0; c0 < cw; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(td + c0, v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (WANT_Z) {
          if (r < nrows) {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const int j = c0 + e;
              if (j < sh.N) Zout[(size_t)r * 2 * sh.N + h * sh.N + j] = (h ? 0.0 : R0) - (double)__uint_as_float(v[e]);
            }
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const float res = __uint_as_float(v[e]);
            ch[e & 3] = fmaf(res, res, ch[e & 3]);
          }
        }
      }
    }
    acc = ((double)ch[0] + (double)ch[1]) + ((double)ch[2] + (double)ch[3]);
  }
  tc_fence_before();
  UMMA_MARK(4)
  if (!WANT_Z) {
    double* part = reinterpret_cast<double*>(s.p0 + o.part);
    if (h == 1) part[r] = acc;
    __syncthreads();
    if (!sh.cl) {
      if (h == 0 && r < nrows) chi[r] = acc + part[r];
    } else {
      // both CTAs of the pair run the sampler on identical walkers: exchange the per-proposal partial sums through
      // distributed shared memory and add them in rank order, so both take bit-identical accept decisions
      cg::cluster_group cluster = cg::this_cluster();
      double* mine = reinterpret_cast<double*>(s.p0 + o.xsum) + ((s.phase >> 8) & 1u) * kUmmaRows;
      if (h == 0) mine[r] = acc + part[r];
      cluster.sync();
      if (h == 0 && r < nrows) chi[r] = cluster.map_shared_rank(mine, 0)[r] + cluster.map_shared_rank(mine, 1)[r];
      s.phase ^= 0x100u;
    }
  }
  UMMA_MARK(5)
}

}  // namespace bisip
