// On-device affine-invariant ensemble sampler: one persistent CTA per spectrum runs all
// nsteps of emcee's red/blue stretch move (SURVEY.md App. B.3; emcee is third-party and not
// vendored in the reference — call sites models.py:111-118) with the walkers, their
// log-probabilities and the per-spectrum model constants resident in shared memory.
//
// Stream layout (identical to oracle/bisip_oracle.c::oracle_ensemble_run):
//   Philox4x32-10, key = seed, counter = (index, step, spectrum, purpose)
//   purpose 0      shuffle keys: walker i <- word (i&3) of index (i>>2), low bits replaced by i so
//                  that keys are unique: key = (word & ~mask) | i, mask = 2^ceil(log2 W) - 1;
//                  walkers ranked by key; ranks [0,H0) = split 0, [H0,W) = split 1, H0 = (W+1)/2
//   purpose 1+s    proposal p of split s, ONE call for all its draws: u = u53(x,y) -> zz = ((a-1)u+1)^2/a ;
//                  partner = mulhi(z, Nc) ; acceptance draw u2 = u53(w, (z << 16) | 0x8000): 43 random bits (w and
//                  the low half of z, which the partner index does not depend on), centred so that u2 > 0
#pragma once
#include "common.cuh"
#include "decomp_eval.cuh"
#include "decomp_rc.cuh"
#include "decomp_tf32.cuh"
#include "decomp_umma.cuh"
#include "decomp_collapsed.cuh"
#include "models.cuh"

namespace bisip {

// Developer build (-DBISIP_PHASE_TIMING, `make dbg`): block 0 accumulates SM cycles per phase and
// prints them at the end.  Compiled out of the product library.
#ifdef BISIP_PHASE_TIMING
#define PHASE_DECL long long ph_[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; long long ph_t_ = clock64(); long long fq_ = 0;
#define FINE_START { fq_ = clock64(); }
#define FINE_MARK(i) { long long n_ = clock64(); ph_[i] += n_ - fq_; fq_ = n_; }
#define PHASE_MARK(i) { long long n_ = clock64(); ph_[i] += n_ - ph_t_; ph_t_ = n_; }
#define PHASE_PRINT if (blockIdx.x == 0 && threadIdx.x == 0) printf("phase cycles/step: split %.0f  propose %.0f  eval %.0f  accept %.0f  store %.0f\n", \
    (double)ph_[0] / P.nsteps, (double)ph_[1] / P.nsteps, (double)ph_[2] / P.nsteps, (double)ph_[3] / P.nsteps, (double)ph_[4] / P.nsteps); \
  if (blockIdx.x == 0 && threadIdx.x == 0) printf("fine (thread 0) cycles/step: propose-body %.0f  propose-barrier %.0f  eval-body %.0f  eval-barrier %.0f  accept-body %.0f  accept-tail(keys) %.0f ; %.0f\n", (double)ph_[6] / P.nsteps, (double)ph_[7] / P.nsteps, (double)ph_[8] / P.nsteps, (double)ph_[9] / P.nsteps, (double)ph_[10] / P.nsteps, (double)ph_[11] / P.nsteps, 0.0);
#else
#define FINE_START
#define FINE_MARK(i)
#define PHASE_DECL
#define PHASE_MARK(i)
#define PHASE_PRINT
#endif

struct EnsembleParams {
  bisip_model_desc d;
  int B, W, nsteps, step0;
  unsigned long long seed;
  uint32_t spectrum0;
  double a;
  int discard, thin, nkeep;
  const double* w; long long w_stride;
  const double* taus; const double* log_taus; long long tau_stride;
  const double* y; const double* yerr; const double* bounds;
  double* coords; double* lp; double* chain; double* logp;
  int* accepted; int* flags;
  unsigned long long stagger_ns;   // start delay of every second CTA on an SM (0 = off)
  // host-precomputed constants (kept in the parameter bank, not in registers)
  uint32_t kmask;                  // 2^ceil(log2 W) - 1
  int a_pow2;                      // a is a power of two: zr*zr/a == zr*zr*inv_a exactly
  double inv_a;
};

struct SamplerSmem {
  double* coords;  // [W][ndim]
  double* lp;      // [W]
  double* prop;    // [rows_pad][ndim]
  double* chi;     // [rows_pad]
  double* zz;      // [2][rows_pad]  stretch factors, double-buffered by half-step parity
  double* bnd;     // [2][ndim]
  double* red;     // [kWarps]
  long long* bkey; // [2][ndim] ordered-integer image of bnd
  float* lf;       // [2][rows_pad]  (ndim-1) ln zz - ln u2 in FP32 (accept filter), by half-step parity; the acceptance
                   //                uniform itself is re-drawn from the Philox counter in the rare FP64 fallback
  uint32_t* keys;  // [Wpad4]        shuffle keys of the NEXT step
  int* list;       // [2][W]         walker at rank, double-buffered by step parity
  int* acc;        // [W]
  int* inb;        // [rows_pad]
  int* partner;    // [rows_pad]     index into the complementary half
  int* hist;       // [260]          bucket counters / starts of the key ranking (16-byte aligned)
  uint32_t* sorted;// [Wpad4]        keys grouped by bucket
};

__host__ __device__ inline int sampler_rows_pad(int W) { return ceil_div((W + 1) / 2, 16) * 16; }

__host__ __device__ inline size_t sampler_smem_bytes(int W, int ndim) {
  const int rp = sampler_rows_pad(W);
  size_t dbl = (size_t)W * ndim + W + (size_t)rp * ndim + rp + 2 * rp + rp + 4 * ndim + kWarps;
  size_t words = (size_t)(W + 4) + 2 * W + W + rp + rp + 260 + (W + 4);
  return dbl * 8 + words * 4 + 48;
}

__device__ inline void sampler_carve(SamplerSmem& s, double* base, int W, int ndim) {
  const int rp = sampler_rows_pad(W);
  s.coords = base; base += (size_t)W * ndim;
  s.lp = base; base += W;
  s.prop = base; base += (size_t)rp * ndim;
  s.chi = base; base += rp;
  s.zz = base; base += 2 * rp;
  s.lf = reinterpret_cast<float*>(base); base += rp;
  s.bnd = base; base += 2 * ndim;
  s.red = base; base += kWarps;
  s.bkey = reinterpret_cast<long long*>(base); base += 2 * ndim;
  s.keys = reinterpret_cast<uint32_t*>((reinterpret_cast<uintptr_t>(base) + 15) & ~uintptr_t(15));   // LDS.128
  s.list = reinterpret_cast<int*>(s.keys + ((W + 3) & ~3));
  s.acc = s.list + 2 * W;
  s.inb = s.acc + W;
  s.partner = s.inb + rp;
  s.hist = reinterpret_cast<int*>((reinterpret_cast<uintptr_t>(s.partner + rp) + 15) & ~uintptr_t(15));
  s.sorted = reinterpret_cast<uint32_t*>(s.hist + 260);
}

// strict box prior, models.py:64-69 (NaN -> outside)
__device__ __forceinline__ bool in_bounds(const double* th, const double* bnd, int ndim) {
  bool ok = true;
  for (int d = 0; d < ndim; ++d) ok = ok && (bnd[d] < th[d]) && (th[d] < bnd[ndim + d]);
  return ok;
}

// Same predicate on the integer pipe (FP64 compares would queue behind the other CTA's DMMA
// stream): doubles mapped to int64 keys that order like IEEE numbers (-0 canonicalised to +0).
// NaNs map beyond +/-inf, so `lo < x < hi` is false for them exactly as in IEEE arithmetic.
__device__ __forceinline__ long long ordered_key(double x) {
  long long b = __double_as_longlong(x);
  if ((b << 1) == 0) b = 0;
  return b ^ ((b >> 63) & 0x7fffffffffffffffLL);
}
__device__ __forceinline__ bool in_bounds_keys(const double* th, const long long* bkey, int ndim) {
  bool ok = true;
  for (int d = 0; d < ndim; ++d) {
    const long long k = ordered_key(th[d]);
    ok = ok & (bkey[d] < k) & (k < bkey[ndim + d]);
  }
  return ok;
}

// ndim is a run-time value (1+3K, 5, 6, 2+poly_deg): a plain loop over it serialises its shared-memory
// loads (one ~30-cycle round trip per dimension).  The proposal is therefore built by a fully unrolled
// body picked by a switch on ndim (2..9 cover poly_deg 0..7, Dias, Shin and 1-2 Cole-Cole modes), so all
// loads of a proposal are in flight together and no instruction is spent on absent dimensions — each FP64
// operation here queues behind the co-resident CTA's tensor-pipe stream.
constexpr int kDimUnroll = 8;

// q = c - (c - s) * zz (explicitly unfused, like the oracle) -> dst ; returns the strict-prior flag
template <int ND>
__device__ __forceinline__ bool propose_and_check_n(const double* __restrict__ cj, const double* __restrict__ sk,
                                                    double zz, double* __restrict__ dst,
                                                    const long long* __restrict__ bkey) {
  double c[ND], x[ND];
  long long lo[ND], hi[ND];
#pragma unroll
  for (int d = 0; d < ND; ++d) {
    c[d] = cj[d];
    x[d] = sk[d];
    lo[d] = bkey[d];
    hi[d] = bkey[ND + d];
  }
  bool ok = true;
#pragma unroll
  for (int d = 0; d < ND; ++d) {
    const double v = __dsub_rn(c[d], __dmul_rn(__dsub_rn(c[d], x[d]), zz));
    const long long k = ordered_key(v);
    dst[d] = v;
    ok = ok & (lo[d] < k) & (k < hi[d]);
  }
  return ok;
}

__device__ __forceinline__ bool propose_and_check(const double* __restrict__ cj, const double* __restrict__ sk,
                                                  double zz, double* __restrict__ dst, const long long* __restrict__ bkey,
                                                  int ndim) {
  switch (ndim) {
    case 2: return propose_and_check_n<2>(cj, sk, zz, dst, bkey);
    case 3: return propose_and_check_n<3>(cj, sk, zz, dst, bkey);
    case 4: return propose_and_check_n<4>(cj, sk, zz, dst, bkey);
    case 5: return propose_and_check_n<5>(cj, sk, zz, dst, bkey);
    case 6: return propose_and_check_n<6>(cj, sk, zz, dst, bkey);
    case 7: return propose_and_check_n<7>(cj, sk, zz, dst, bkey);
    case 8: return propose_and_check_n<8>(cj, sk, zz, dst, bkey);
    case 9: return propose_and_check_n<9>(cj, sk, zz, dst, bkey);
    default: break;
  }
  bool ok = true;
  for (int d = 0; d < ndim; ++d) {
    const double v = __dsub_rn(cj[d], __dmul_rn(__dsub_rn(cj[d], sk[d]), zz));
    dst[d] = v;
    const long long k = ordered_key(v);
    ok = ok & (bkey[d] < k) & (k < bkey[ndim + d]);
  }
  return ok;
}

// q = c - (c - s) * zz for the dimensions d = sub, sub + 2, ... of one proposal (the two lanes of a row share it);
// returns this lane's part of the strict-prior flag.  Fully unrolled per ndim like propose_and_check_n.
template <int ND>
__device__ __forceinline__ bool propose_pair_n(const double* __restrict__ cj, const double* __restrict__ sk, double zz,
                                               double* __restrict__ dst, const long long* __restrict__ bkey, int sub) {
  constexpr int H = (ND + 1) / 2;
  double c[H], x[H];
  long long lo[H], hi[H];
#pragma unroll
  for (int i = 0; i < H; ++i) {
    const int d = 2 * i + sub;
    const int dd = d < ND ? d : 0;
    c[i] = cj[dd];
    x[i] = sk[dd];
    lo[i] = bkey[dd];
    hi[i] = bkey[ND + dd];
  }
  bool ok = true;
#pragma unroll
  for (int i = 0; i < H; ++i) {
    const int d = 2 * i + sub;
    const double v = __dsub_rn(c[i], __dmul_rn(__dsub_rn(c[i], x[i]), zz));
    const long long k = ordered_key(v);
    if (d < ND) {
      dst[d] = v;
      ok = ok & (lo[i] < k) & (k < hi[i]);
    }
  }
  return ok;
}

__device__ __forceinline__ bool propose_pair(const double* __restrict__ cj, const double* __restrict__ sk, double zz,
                                             double* __restrict__ dst, const long long* __restrict__ bkey, int ndim, int sub) {
  switch (ndim) {
    case 2: return propose_pair_n<2>(cj, sk, zz, dst, bkey, sub);
    case 3: return propose_pair_n<3>(cj, sk, zz, dst, bkey, sub);
    case 4: return propose_pair_n<4>(cj, sk, zz, dst, bkey, sub);
    case 5: return propose_pair_n<5>(cj, sk, zz, dst, bkey, sub);
    case 6: return propose_pair_n<6>(cj, sk, zz, dst, bkey, sub);
    case 7: return propose_pair_n<7>(cj, sk, zz, dst, bkey, sub);
    case 8: return propose_pair_n<8>(cj, sk, zz, dst, bkey, sub);
    case 9: return propose_pair_n<9>(cj, sk, zz, dst, bkey, sub);
    default: break;
  }
  bool ok = true;
  for (int d = sub; d < ndim; d += 2) {
    const double v = __dsub_rn(cj[d], __dmul_rn(__dsub_rn(cj[d], sk[d]), zz));
    dst[d] = v;
    const long long k = ordered_key(v);
    ok = ok & (bkey[d] < k) & (k < bkey[ndim + d]);
  }
  return ok;
}

// Accept filter on the integer pipe.  est = (lp' - lp) + lf is the FP32-logarithm image of emcee's
// (ndim-1) ln zz + lp' - lp - ln u, whose error is < 1e-5 from the logarithms plus the FP64 rounding of the two
// log-probabilities (<= 2^-52 (|lp'| + |lp|)).  The FP64 decision is therefore already determined whenever
// |est| >= 2^-12 and |est| >= 2^-46 max(|lp'|, |lp|); both are comparisons of biased exponents.  NaN (inf - inf)
// is "determined" too: emcee's `nan > x` is False.  Returns true when determined and sets `accept`.
__device__ __forceinline__ bool accept_filter(double est, double lpn, double lpo, bool& accept) {
  const int he = __double2hiint(est);
  const unsigned ae = (unsigned)he & 0x7fffffffu;
  const unsigned e_est = ae >> 20;
  const unsigned e_n = ((unsigned)__double2hiint(lpn) >> 20) & 0x7ffu, e_o = ((unsigned)__double2hiint(lpo) >> 20) & 0x7ffu;
  const unsigned emax = e_n > e_o ? e_n : e_o;
  const bool is_nan = ae > 0x7ff00000u || (ae == 0x7ff00000u && __double2loint(est) != 0);
  accept = (he >= 0) && !is_nan;
  return e_est >= 1011u && e_est + 46u >= emax;
}

__device__ __forceinline__ void copy_dims(double* __restrict__ dst, const double* __restrict__ src, int ndim) {
#pragma unroll
  for (int d = 0; d < kDimUnroll; ++d) {
    const double v = src[d < ndim ? d : 0];
    if (d < ndim) dst[d] = v;
  }
  for (int d = kDimUnroll; d < ndim; ++d) dst[d] = src[d];
}

// All random draws of proposal rows of half-step (t, sp) from one Philox call per proposal (stream layout at the top of
// this file): stretch factor, partner index, and the FP32 image of the accept threshold (ndim-1) ln zz - ln u2.  It only
// depends on the Philox counter, so it may run anywhere before the next PROPOSE phase (the sampler gives it to the
// threads that have no proposal to accept).
struct DrawCtx {
  double* zz;          // [2][rows_pad]
  float* lf;           // [2][rows_pad]
  int* partner;        // [rows_pad]
  int rows_pad, W, H0, ndim;
  uint32_t spec, k0, k1;
  double a, inv_a;
  int a_pow2;
};

__device__ __forceinline__ void draw_rows(const DrawCtx& c, uint32_t t, int sp, int worker, int nworkers) {
  const int Hs = sp ? c.W - c.H0 : c.H0, Nc = c.W - Hs;
  double* zzb = c.zz + (size_t)sp * c.rows_pad;
  float* lfb = c.lf + (size_t)sp * c.rows_pad;
  const bool a_is2 = c.a == 2.0;
  const float am1f = (float)(c.a - 1.0), inv_af = (float)c.inv_a, nd1f = (float)(c.ndim - 1);
  for (int q = worker; q < Hs; q += nworkers) {
    const u32x4 r = philox4x32_10((uint32_t)q, t, c.spec, (uint32_t)(1 + sp), c.k0, c.k1);
    // the uniforms are assembled on the integer pipe (u53_int) and the accept threshold on the FP32 pipe: every
    // FP64-pipe instruction of this work would queue behind the co-resident warps' tensor / DFMA stream
    const double u = u53_int(r.x, r.y);
    double zz;
    if (a_is2) {                                    // ((a-1) u + 1)^2 / a with a = 2: (a-1) u = u and /2 are exact
      const double zr = __dadd_rn(u, 1.0);
      const double sq = __dmul_rn(zr, zr);          // in [1, 4): halving = one exponent step
      zz = __hiloint2double(__double2hiint(sq) - 0x00100000, __double2loint(sq));
    } else {
      const double zr = __dadd_rn(__dmul_rn(c.a - 1.0, u), 1.0);
      zz = c.a_pow2 ? __dmul_rn(__dmul_rn(zr, zr), c.inv_a) : __ddiv_rn(__dmul_rn(zr, zr), c.a);
    }
    const uint32_t zlow = (r.z << 16) | 0x8000u;
    zzb[q] = zz;
    c.partner[q] = (int)__umulhi(r.z, (uint32_t)Nc);
    // FP32 image of (ndim-1) ln zz - ln u2 straight from the random words: |error| < 1e-5, far inside the 2^-12
    // margin below which accept_filter() hands the decision to the FP64 logarithms
    const float uf = (float)(r.x >> 8) * 5.9604644775390625e-08f;                    // 2^-24
    const float zrf = fmaf(am1f, uf, 1.0f);
    const float zzf = zrf * zrf * inv_af;
    const float u2f = fmaf((float)(zlow >> 6), 1.1102230246251565e-16f,                // 2^-53
                           (float)(r.w >> 5) * 7.450580596923828e-09f);              // 2^-27
    lfb[q] = nd1f * __logf(zzf) - __logf(u2f);
  }
}

// Side work executed INSIDE the evaluation phase: ranking the shuffle keys of the next step.  It is
// pure integer/LDS work, so it fills issue slots that the tile loop leaves idle while its warps wait
// for the FP64 tensor pipe; the evaluators call advance() once per column-tile iteration.
// count of the 4 keys of shared-memory chunk `saddr` (32-bit shared address) that are below ki:
// one LDS.128 + (ISETP, predicated add) per key, four independent counters
__device__ __forceinline__ void rank_chunk(uint32_t saddr, uint32_t ki, int& r0, int& r1, int& r2, int& r3) {
  asm volatile(
      "{\n\t"
      ".reg .pred p0, p1, p2, p3;\n\t"
      ".reg .u32 k0, k1, k2, k3;\n\t"
      "ld.shared.v4.u32 {k0, k1, k2, k3}, [%4];\n\t"
      "setp.lt.u32 p0, k0, %5;\n\t"
      "setp.lt.u32 p1, k1, %5;\n\t"
      "setp.lt.u32 p2, k2, %5;\n\t"
      "setp.lt.u32 p3, k3, %5;\n\t"
      "@p0 add.s32 %0, %0, 1;\n\t"
      "@p1 add.s32 %1, %1, 1;\n\t"
      "@p2 add.s32 %2, %2, 1;\n\t"
      "@p3 add.s32 %3, %3, 1;\n\t"
      "}"
      : "+r"(r0), "+r"(r1), "+r"(r2), "+r"(r3)
      : "r"(saddr), "r"(ki));
}

struct RankSide {
  uint32_t kaddr;    // shared-memory address of the keys (4 per 16-byte chunk)
  const uint32_t* keys;
  int* list_out;
  int nchunks;       // Wpad4/4
  int W;
  int pos, step;
  int r0, r1, r2, r3;
  uint32_t ki;
  bool on;
  __device__ __forceinline__ void begin(const uint32_t* keys_, int* list, int W_, int iters) {
    keys = keys_;
    kaddr = (uint32_t)__cvta_generic_to_shared(keys_);
    list_out = list;
    W = W_;
    nchunks = ((W_ + 3) & ~3) >> 2;
    on = list != nullptr;
    pos = 0;
    r0 = r1 = r2 = r3 = 0;
    step = iters > 0 ? (nchunks + iters - 1) / iters : nchunks;
    ki = (on && (int)threadIdx.x < W_) ? keys_[threadIdx.x] : 0u;
  }
  __device__ __forceinline__ void advance() {
    if (!on) return;
    const int end = min(nchunks, pos + step);
    for (; pos < end; ++pos) rank_chunk(kaddr + 16u * pos, ki, r0, r1, r2, r3);
  }
  __device__ __forceinline__ void finish() {
    if (!on) return;
    if ((int)threadIdx.x < W) {                       // warps without walkers skip the count
#pragma unroll 4
      for (; pos < nchunks; ++pos) rank_chunk(kaddr + 16u * pos, ki, r0, r1, r2, r3);
      list_out[(r0 + r1) + (r2 + r3)] = threadIdx.x;
    }
    for (int i = threadIdx.x + blockDim.x; i < W; i += blockDim.x) {   // W > CTA size: remaining walkers, not interleaved
      const uint32_t k = keys[i];
      int a = 0, b = 0, c = 0, d = 0;
      for (int ch = 0; ch < nchunks; ++ch) rank_chunk(kaddr + 16u * ch, k, a, b, c, d);
      list_out[(a + b) + (c + d)] = i;
    }
    on = false;
  }
};

// Ranking of the shuffle keys in O(W): walkers are binned by the top 8 bits of their (uniform random) key, the 256
// bin counts are scanned by one warp, and each walker then only compares itself with the keys of its own bin (one
// on average).  rank = bin start + smaller keys in the bin — the same number the all-pairs count above produces, so
// chains stay bit-identical; the shared-memory atomics only decide where a key is parked inside its bin.
// All threads of the CTA; W <= NT.  Ends without a barrier (the caller synchronises before list_out is read).
// ZERO = false: the caller has zeroed hist[0, 256) behind a barrier already (the sampling loop does it in the first
// accept phase of the step, which saves one CTA barrier per step).
// rank_binned_rest: everything after the bin slots (key, bin, slot of this thread's walker, taken with atomicAdd on
// counters that were zero; a barrier lies between the last atomicAdd and this call): scan, placement, count.
template <int NT>
__device__ __forceinline__ void rank_binned_rest(int* __restrict__ list_out, int W, int* __restrict__ hist,
                                                 uint32_t* __restrict__ sorted, uint32_t key, int bin, int slot) {
  const int tid = threadIdx.x;
  if (tid < 32) {                                  // exclusive scan of the 256 counters, 8 per lane
    int4* h4 = reinterpret_cast<int4*>(hist);
    const int4 a = h4[2 * tid], c = h4[2 * tid + 1];
    const int s0 = a.x, s1 = s0 + a.y, s2 = s1 + a.z, s3 = s2 + a.w, s4 = s3 + c.x, s5 = s4 + c.y, s6 = s5 + c.z;
    const int tot = s6 + c.w;
    int inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, inc, o);
      if (tid >= o) inc += n;
    }
    const int base = inc - tot;
    h4[2 * tid] = make_int4(base, base + s0, base + s1, base + s2);
    h4[2 * tid + 1] = make_int4(base + s3, base + s4, base + s5, base + s6);
    if (tid == 31) hist[256] = inc;
  }
  __syncthreads();
  int start = 0;
  if (tid < W) {
    start = hist[bin];
    sorted[start + slot] = key;
  }
  __syncthreads();
  if (tid < W) {
    const int end = hist[bin + 1];
    int cnt = 0;
    for (int j = start; j < end; ++j) cnt += sorted[j] < key ? 1 : 0;
    list_out[start + cnt] = tid;
  }
}

template <int NT>
__device__ __forceinline__ void rank_keys_binned(const uint32_t* __restrict__ keys, int* __restrict__ list_out, int W,
                                                 int* __restrict__ hist, uint32_t* __restrict__ sorted) {
  const int tid = threadIdx.x;
  for (int i = tid; i < 256; i += NT) hist[i] = 0;
  __syncthreads();
  uint32_t key = 0;
  int bin = 0, slot = 0;
  if (tid < W) {
    key = keys[tid];
    bin = (int)(key >> 24);
    slot = atomicAdd(&hist[bin], 1);
  }
  __syncthreads();
  rank_binned_rest<NT>(list_out, W, hist, sorted, key, bin, slot);
}

// Binned key ranking (rank_keys_binned above) cut at its barriers so that the warp-private sampler can place the pieces
// between the barriers it has anyway.  `counts` must be zero on entry of part A and is left intact by B and C.
//   A  slot of every key inside its bin                       (needs: keys visible)          -> (key, bin, slot)
//   -- barrier --
//   B  every warp scans the 256 bin counts itself (8 per lane + a shuffle scan) and hands each of its threads the start of
//      its bin by shuffle — no shared array of starts, nothing written but sorted[start + slot] = key
//   -- barrier --
//   C  rank = start + smaller keys in the own bin ; list_out[rank] = walker
template <int NT>
__device__ __forceinline__ void rank_part_a(const uint32_t* __restrict__ keys, int W, int* __restrict__ counts,
                                            uint32_t& key, int& bin, int& slot) {
  const int tid = threadIdx.x;
  key = 0; bin = 0; slot = 0;
  if (tid < W) {
    key = keys[tid];
    bin = (int)(key >> 24);
    slot = atomicAdd(&counts[bin], 1);
  }
}
template <int NT>
__device__ __forceinline__ int rank_part_b(int W, const int* __restrict__ counts, uint32_t* __restrict__ sorted,
                                           uint32_t key, int bin, int slot) {
  const int tid = threadIdx.x, lane = tid & 31;
  int pre[8];                                      // exclusive prefix of bins 8 lane ... 8 lane + 7
  {
    const int4* h4 = reinterpret_cast<const int4*>(counts);
    const int4 a = h4[2 * lane], c = h4[2 * lane + 1];
    const int s0 = a.x, s1 = s0 + a.y, s2 = s1 + a.z, s3 = s2 + a.w, s4 = s3 + c.x, s5 = s4 + c.y, s6 = s5 + c.z;
    const int tot = s6 + c.w;
    int inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += n;
    }
    const int base = inc - tot;
    pre[0] = base; pre[1] = base + s0; pre[2] = base + s1; pre[3] = base + s2;
    pre[4] = base + s3; pre[5] = base + s4; pre[6] = base + s5; pre[7] = base + s6;
  }
  int start = 0;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int v = __shfl_sync(0xffffffffu, pre[e], bin >> 3);
    if ((bin & 7) == e) start = v;
  }
  if (tid < W) sorted[start + slot] = key;
  return start;
}
template <int NT>
__device__ __forceinline__ void rank_part_c(int W, const int* __restrict__ counts, const uint32_t* __restrict__ sorted,
                                            int* __restrict__ list_out, uint32_t key, int bin, int start) {
  const int tid = threadIdx.x;
  if (tid < W) {
    const int end = start + counts[bin];
    int cnt = 0;
    for (int j = start; j < end; ++j) cnt += sorted[j] < key ? 1 : 0;
    list_out[start + cnt] = tid;
  }
}

// Evaluator adaptors -------------------------------------------------------------------
template <int KC>
struct DecompEvaluator {
  static constexpr bool kClustered = false;
  static constexpr bool kRankInAccept = true;
  static constexpr bool kLegacyRank = false;
  static constexpr bool kNeedsPrepare = false;
  __device__ __forceinline__ void prepare_row(int, const double*) {}
  __device__ __forceinline__ void release() {}
  DecompSmem sm;
  DecompShape sh;
  int rows_pad;
  __device__ DecompEvaluator(const bisip_model_desc& d, int, int) : sh(d.n_freq, d.n_tau, d.n_coef) {}
  static __host__ size_t smem_doubles(const bisip_model_desc& d, int rows_pad) {
    return decomp_smem_doubles(DecompShape(d.n_freq, d.n_tau, d.n_coef), rows_pad);
  }
  __device__ double* carve(double* base, int rp) { rows_pad = rp; return decomp_carve(sm, base, sh, rp); }
  __device__ void init(const bisip_model_desc& d, const double* w, const double* taus, const double* log_taus,
                       const double* y, const double* yerr, double* red) {
    decomp_init(sm, sh, d.c_exp, w, taus, log_taus, y, yerr, red);
  }
  __device__ double llconst() const { return sm.llconst; }
  __device__ __forceinline__ double chi_of(const double* chi, int q) const { return chi[q]; }
  __device__ int iters_per_warp(int nrows) const { return decomp_iters_per_warp(sh, nrows); }
  template <class Side>
  __device__ void eval_chi(const double* prop, int ndim, int nrows, double* chi, Side& side) {
    decomp_eval_chi<KC>(sm, sh, prop, ndim, nrows, rows_pad, chi, side);
  }
  __device__ void eval_Z(const double* prop, int ndim, int nrows, double* Z) {
    decomp_eval_Z<KC>(sm, sh, prop, ndim, nrows, Z);
  }
};

// Large tau grids: stage 1 recomputed per k chunk, frequency columns split over a CTA cluster.
struct DecompRCEvaluator {
  static constexpr bool kClustered = true;
  static constexpr bool kRankInAccept = false;     // measured: 3.712e8 vs 3.691e8 at 256 taus (profiles/r02d_barriers.md)
  static constexpr bool kLegacyRank = false;
  static constexpr bool kNeedsPrepare = false;
  __device__ __forceinline__ void prepare_row(int, const double*) {}
  __device__ __forceinline__ void release() {}
  DecompRCSmem sm;
  DecompRCShape sh;
  int rows_pad;
  __device__ DecompRCEvaluator(const bisip_model_desc& d, int cs, int rank) : sh(d.n_freq, d.n_tau, d.n_coef, cs, rank) {}
  static __host__ size_t smem_doubles(const bisip_model_desc& d, int rows_pad, int cs) {
    return decomp_rc_smem_doubles(DecompRCShape(d.n_freq, d.n_tau, d.n_coef, cs, 0), rows_pad);
  }
  __device__ double* carve(double* base, int rp) { rows_pad = rp; return decomp_rc_carve(sm, base, sh, rp); }
  __device__ void init(const bisip_model_desc& d, const double* w, const double* taus, const double* log_taus,
                       const double* y, const double* yerr, double* red) {
    decomp_rc_init(sm, sh, d.c_exp, w, taus, log_taus, y, yerr, red);
  }
  __device__ double llconst() const { return sm.llconst; }
  __device__ __forceinline__ double chi_of(const double* chi, int q) const { return chi[q]; }
  __device__ int iters_per_warp(int) const { return 0; }
  template <class Side>
  __device__ void eval_chi(const double* prop, int ndim, int nrows, double* chi, Side& side) {
    side.finish();
    decomp_rc_eval_chi(sm, sh, prop, ndim, nrows, rows_pad, chi);
  }
  __device__ void eval_Z(const double* prop, int ndim, int nrows, double* Z) {
    decomp_rc_eval_Z(sm, sh, prop, ndim, nrows, Z);
  }
};

// TF32 (PREC=1) / 3xTF32 (PREC=3) stage 2, FP64 stage 1; same clustered work split.
template <int PREC>
struct DecompTF32Evaluator {
  static constexpr bool kClustered = true;
  static constexpr bool kRankInAccept = true;
  static constexpr bool kLegacyRank = false;
  static constexpr bool kNeedsPrepare = false;
  __device__ __forceinline__ void prepare_row(int, const double*) {}
  __device__ __forceinline__ void release() {}
  DecompTF32Smem sm;
  DecompRCShape sh;
  int rows_pad;
  __device__ DecompTF32Evaluator(const bisip_model_desc& d, int cs, int rank) : sh(d.n_freq, d.n_tau, d.n_coef, cs, rank) {}
  static __host__ size_t smem_doubles(const bisip_model_desc& d, int rows_pad, int cs) {
    return decomp_tf32_smem_doubles(DecompRCShape(d.n_freq, d.n_tau, d.n_coef, cs, 0), rows_pad, PREC);
  }
  __device__ double* carve(double* base, int rp) { rows_pad = rp; return decomp_tf32_carve<PREC>(sm, base, sh, rp); }
  __device__ void init(const bisip_model_desc& d, const double* w, const double* taus, const double* log_taus,
                       const double* y, const double* yerr, double* red) {
    decomp_tf32_init<PREC>(sm, sh, d.c_exp, w, taus, log_taus, y, yerr, red);
  }
  __device__ double llconst() const { return sm.llconst; }
  __device__ __forceinline__ double chi_of(const double* chi, int q) const { return chi[q]; }
  __device__ int iters_per_warp(int) const { return 0; }
  template <class Side>
  __device__ void eval_chi(const double* prop, int ndim, int nrows, double* chi, Side& side) {
    side.finish();
    decomp_tf32_eval_chi<PREC>(sm, sh, prop, ndim, nrows, rows_pad, chi);
  }
  __device__ void eval_Z(const double* prop, int ndim, int nrows, double* Z) {
    decomp_tf32_eval_Z<PREC>(sm, sh, prop, ndim, nrows, Z);
  }
};

// TF32 (PREC=1) / 3xTF32 (PREC=3) stage 2 on tcgen05 tensor cores: A (chargeability) and the FP32 accumulators
// live in tensor memory, one M = 128 tile per half-step (<= 256 walkers, <= 64 frequencies).
template <int PREC, bool CL = false>
struct DecompUmmaEvaluator {
  static constexpr bool kClustered = CL;
  static constexpr bool kRankInAccept = true;      // TF32 8.38e9 vs 8.32e9, 3xTF32 equal
  static constexpr bool kLegacyRank = false;
  static constexpr bool kNeedsPrepare = false;
  __device__ __forceinline__ void prepare_row(int, const double*) {}
  DecompUmmaSmem sm;
  DecompUmmaShape sh;
  __device__ DecompUmmaEvaluator(const bisip_model_desc& d, int, int rank) : sh(d.n_freq, d.n_tau, d.n_coef, CL ? 1 : 0, rank) {}
  static __host__ size_t smem_doubles(const bisip_model_desc& d, int) {
    return decomp_umma_smem_doubles(DecompUmmaShape(d.n_freq, d.n_tau, d.n_coef, CL ? 1 : 0, 0), PREC);
  }
  __device__ double* carve(double* base, int) { return decomp_umma_carve<PREC>(sm, base, sh); }
  __device__ void init(const bisip_model_desc& d, const double* w, const double* taus, const double* log_taus,
                       const double* y, const double* yerr, double* red) {
    decomp_umma_init<PREC>(sm, sh, d.c_exp, w, taus, log_taus, y, yerr, red);
  }
  __device__ double llconst() const { return sm.llconst; }
  __device__ __forceinline__ double chi_of(const double* chi, int q) const { return chi[q]; }
  __device__ int iters_per_warp(int) const { return 0; }
  template <class Side>
  __device__ void eval_chi(const double* prop, int ndim, int nrows, double* chi, Side& side) {
    side.finish();
    decomp_umma_eval<PREC, false>(sm, sh, prop, ndim, nrows, chi, nullptr);
  }
  __device__ void eval_Z(const double* prop, int ndim, int nrows, double* Z) {
    decomp_umma_eval<PREC, true>(sm, sh, prop, ndim, nrows, nullptr, Z);
  }
  __device__ void release() { decomp_umma_release(sm, sh); }   // frees the tensor memory
};

// Collapsed form z = (L K) a on the FP64 vector pipe (decomp_collapsed.cuh): precision 'fp64-collapsed'.
struct DecompCollapsedEvaluator {
  static constexpr bool kClustered = false;
  static constexpr bool kRankInAccept = true;
  static constexpr bool kLegacyRank = false;
  static constexpr bool kNeedsPrepare = false;
  __device__ __forceinline__ void prepare_row(int, const double*) {}
  __device__ __forceinline__ void release() {}
  DecompCSmem sm;
  DecompCShape sh;
  int rows_pad;
  __device__ DecompCollapsedEvaluator(const bisip_model_desc& d, int, int) : sh(d.n_freq, d.n_tau, d.n_coef) {}
  static __host__ size_t smem_doubles(const bisip_model_desc& d, int rows_pad) {
    return decomp_c_smem_doubles(DecompCShape(d.n_freq, d.n_tau, d.n_coef), rows_pad);
  }
  // rp = sampler_rows_pad(W) >= the rows of either half-step
  __device__ double* carve(double* base, int rp) { rows_pad = rp; return decomp_c_carve(sm, base, sh, rp); }
  __device__ void init(const bisip_model_desc& d, const double* w, const double* taus, const double* log_taus,
                       const double* y, const double* yerr, double* red) {
    decomp_c_init(sm, sh, d.c_exp, w, taus, log_taus, y, yerr, red);
  }
  __device__ double llconst() const { return sm.llconst; }
  // the per-column-group partial sums are added here, in group order, by the thread that takes the accept
  // decision: no reduction pass and no extra barrier inside the evaluation
  __device__ __forceinline__ double chi_of(const double*, int q) const {
    const int ngroups = decomp_c_ngroups(rows_pad, sh.N);
    double acc = 0.0;
    for (int g = 0; g < ngroups; ++g) acc += sm.part[(size_t)g * rows_pad + q];
    return acc;
  }
  __device__ int iters_per_warp(int) const { return 0; }
  template <class Side>
  __device__ void eval_chi(const double* prop, int ndim, int nrows, double* chi, Side& side) {
    side.finish();
    decomp_c_eval_parts(sm, sh, rows_pad, prop, ndim, nrows, rows_pad);
  }
  __device__ void eval_Z(const double* prop, int ndim, int nrows, double* Z) {
    decomp_c_eval_Z(sm, sh, prop, ndim, nrows, Z);
  }
};

template <class Row, int ILP = 2>
struct VecEvaluator {
  static constexpr bool kClustered = false;
  static constexpr bool kRankInAccept = Row::kRankInAccept;
  static constexpr bool kLegacyRank = Row::kLegacyRank;
  static constexpr bool kNeedsPrepare = true;
  VecSmem sm;
  int N, n_modes;
  __device__ VecEvaluator(const bisip_model_desc& d, int, int) : N(d.n_freq), n_modes(d.n_modes) {}
  static __host__ size_t smem_doubles(const bisip_model_desc& d, int rows_pad) {
    return vec_smem_doubles(d.n_freq, rows_pad, Row::kRC);
  }
  __device__ double* carve(double* base, int rp) { return vec_carve(sm, base, N, rp, Row::kRC); }
  __device__ void init(const bisip_model_desc&, const double* w, const double*, const double*, const double* y,
                       const double* yerr, double* red) {
    vec_init(sm, N, w, y, yerr, red);
  }
  __device__ double llconst() const { return sm.llconst; }
  __device__ __forceinline__ double chi_of(const double* chi, int q) const { return chi[q]; }
  __device__ int iters_per_warp(int) const { return 0; }
  // theta-only constants of proposal q (exp / sincospi / divisions), by the thread that built it
  __device__ __forceinline__ void prepare_row(int q, const double* th) {
    Row::prepare(th, n_modes, sm.rowc + (size_t)q * Row::kRC);
  }
  __device__ __forceinline__ void release() {}
  template <class Side>
  __device__ void eval_chi(const double*, int, int nrows, double* chi, Side& side) {
    side.finish();
    vec_eval_chi<Row, ILP>(sm, N, n_modes, nrows, chi);
  }
  __device__ void eval_Z(const double*, int, int nrows, double* Z) { vec_eval_Z<Row>(sm, N, n_modes, nrows, Z); }
};

// Co-resident CTAs that start together stay phase-locked: both run their serial phases
// (split, proposals, accept) at the same time and then fight for the math pipe at the same time.
// The second CTA to arrive on an SM therefore starts a fraction of a step late, after which the two
// alternate (one samples/accepts while the other owns the FP64 tensor pipe).  The arrival order
// comes from a per-SM counter that is never reset (only its parity matters).
__device__ unsigned int g_sm_arrivals[1024];

__device__ __forceinline__ void stagger_start(unsigned long long delay_ns) {
  __shared__ unsigned int slot_s;
  if (threadIdx.x == 0) {
    unsigned int smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    slot_s = atomicAdd(&g_sm_arrivals[smid & 1023], 1u);
  }
  __syncthreads();
  if ((slot_s & 1u) && delay_ns) {
    if (threadIdx.x == 0) {
      unsigned long long t0, t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      do {
        __nanosleep(1000);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      } while (t1 - t0 < delay_ns);
    }
    __syncthreads();
  }
}

// NT = CTA size: 256, or 128 for the vector models with <= 128 walkers (twice as many, half as wide
// CTAs per SM: their serial phases keep fewer lanes idle and interleave better; api.cu picks).
template <class Eval, int MINB, int NT = kThreads>
__global__ void __launch_bounds__(NT, MINB) ensemble_kernel(const EnsembleParams P) {
  extern __shared__ __align__(16) double smem[];
  const int tid = threadIdx.x;
  if (MINB > 1 && !Eval::kClustered) stagger_start(P.stagger_ns);
  // clustered evaluators: the CTAs of a cluster own one spectrum together (column split); all of
  // them run the sampler on identical state, rank 0 alone writes the results
  int cs = 1, crank = 0;
  if (Eval::kClustered) {
    cg::cluster_group cluster = cg::this_cluster();
    cs = (int)cluster.num_blocks();
    crank = (int)cluster.block_rank();
  }
  const int b = blockIdx.x / cs;
  const bool writer = (crank == 0);
  const int W = P.W, ndim = P.d.ndim;
  const int rows_pad = sampler_rows_pad(W);
  const int H0 = (W + 1) / 2;

  Eval ev(P.d, cs, crank);
  SamplerSmem s;
  double* p = ev.carve(smem, rows_pad);
  sampler_carve(s, p, W, ndim);

  // ---- per-spectrum constants + initial ensemble ---------------------------------------
  for (int i = tid; i < 2 * ndim; i += NT) {
    s.bnd[i] = P.bounds[i];
    s.bkey[i] = ordered_key(P.bounds[i]);
  }
  const double* gc = P.coords + (size_t)b * W * ndim;
  for (int i = tid; i < W * ndim; i += NT) s.coords[i] = gc[i];
  for (int i = tid; i < W; i += NT) s.acc[i] = 0;
  for (int i = tid; i < rows_pad * ndim; i += NT) s.prop[i] = 0.0;
  ev.init(P.d, P.w + (size_t)b * P.w_stride, P.taus + (size_t)b * P.tau_stride,
          P.log_taus + (size_t)b * P.tau_stride * P.d.n_coef, P.y + (size_t)b * 2 * P.d.n_freq,
          P.yerr + (size_t)b * 2 * P.d.n_freq, s.red);   // ends with __syncthreads()
  const double llc = ev.llconst();
  int flag = 0;

  // log-probability of p0, in two passes of <= H0 rows
  RankSide side;
  side.begin(s.keys, nullptr, W, 0);
  for (int pass = 0; pass < 2; ++pass) {
    const int off = pass ? H0 : 0, n = pass ? W - H0 : H0;
    for (int i = tid; i < n * ndim; i += NT) s.prop[i] = s.coords[off * ndim + i];
    __syncthreads();
    if (Eval::kNeedsPrepare) {
      for (int q = tid; q < n; q += NT) ev.prepare_row(q, s.prop + q * ndim);
      __syncthreads();
    }
    ev.eval_chi(s.prop, ndim, n, s.chi, side);
    __syncthreads();
    for (int q = tid; q < n; q += NT) {
      const double v = in_bounds(s.prop + q * ndim, s.bnd, ndim) ? -0.5 * (ev.chi_of(s.chi, q) + llc) : neg_inf();
      if (v != v) flag |= 2;
      s.lp[off + q] = v;
    }
    __syncthreads();
  }

  const uint32_t k0 = (uint32_t)P.seed, k1 = (uint32_t)(P.seed >> 32);
  const uint32_t spec = P.spectrum0 + (uint32_t)b;
  const int first = P.discard + P.thin - 1;
  const int Wpad4 = (W + 3) & ~3;
  int kept = 0;

  // ---- work that depends only on the Philox stream runs one phase AHEAD of its use, on threads that
  //      would otherwise idle, so that the serial phases between two evaluations stay short ----------
  // shuffle keys of step t (emcee: shuffle(arange(W) % 2)): one Philox call feeds 4 walkers
  auto gen_keys = [&](uint32_t t, int worker, int nworkers) {
    for (int c = worker; c < Wpad4 / 4; c += nworkers) {
      const u32x4 r = philox4x32_10((uint32_t)c, t, spec, 0u, k0, k1);
      const uint32_t wd[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int i = 4 * c + e;
        s.keys[i] = i < W ? ((wd[e] & ~P.kmask) | (uint32_t)i) : 0xffffffffu;   // padding sorts last
      }
    }
  };
  DrawCtx dctx;
  dctx.zz = s.zz; dctx.lf = s.lf; dctx.partner = s.partner; dctx.rows_pad = rows_pad; dctx.W = W; dctx.H0 = H0; dctx.ndim = ndim;
  dctx.spec = spec; dctx.k0 = k0; dctx.k1 = k1; dctx.a = P.a; dctx.inv_a = P.inv_a; dctx.a_pow2 = P.a_pow2;
  const bool binned = W <= NT;                       // binned ranking (one key per thread); else the all-pairs side work

  // prologue: split of step 0 and the draws of its first half-step
  gen_keys((uint32_t)P.step0, tid, NT);
  __syncthreads();
  if (binned) {
    rank_keys_binned<NT>(s.keys, s.list, W, s.hist, s.sorted);
  } else {
    side.begin(s.keys, s.list, W, 0);
    side.finish();
  }
  draw_rows(dctx, (uint32_t)P.step0, 0, tid, NT);
  __syncthreads();

  uint32_t rk_key = 0;
  int rk_bin = 0, rk_slot = 0;
  // The Dias and Cole-Cole kernels (6-8 CTAs per SM) are FASTER with the round-1 sequence of 12 barriers per step, the
  // doubled one included (same-box A/B, profiles/r02d_barriers.md: Dias, 128 walkers, 7.01e9 vs 6.95e9 on full waves, 6.30e9
  // vs 6.06e9 on the 1,024 spectra of BASELINE config 3; Shin is 0.6 % faster with the short one): their barriers are free
  // (other CTAs fill them) and apparently keep the co-resident CTAs out of phase.
  constexpr bool kLegacyRank = Eval::kLegacyRank;
  constexpr bool kPairPropose = Eval::kClustered;   // same-box A/B (profiles/r02d_barriers.md): clustered evaluators +0.4-1 %, TF32 tcgen05 -2 %
  // bin slots of the key ranking inside the second accept phase (one CTA barrier less per step) or in a phase of their
  // own: +-1-2 % either way depending on the evaluator and the CTA size (profiles/r02d_barriers.md)
  constexpr bool kRankInAccept = Eval::kRankInAccept && (NT == 128 || Eval::kClustered || !Eval::kNeedsPrepare);
  PHASE_DECL
  for (int it = 0; it < P.nsteps; ++it) {
    const uint32_t t = (uint32_t)(P.step0 + it);
    const int* list = s.list + (size_t)(it & 1) * W;          // this step's split
    int* list_next = s.list + (size_t)((it + 1) & 1) * W;
    PHASE_MARK(5)
    for (int sp = 0; sp < 2; ++sp) {
      const int off = sp ? H0 : 0, Hs = sp ? W - H0 : H0;
      const int coff = sp ? 0 : H0;
      const double* zzb = s.zz + (size_t)sp * rows_pad;
      const float* lfb = s.lf + (size_t)sp * rows_pad;
      // ---- PROPOSE: threads [0,Hs) build q = c_j - (c_j - s_k) zz (the random draws of this half-step were produced
      //      under the previous evaluation).  Second half-step: every thread also takes the bin slot of its key of the
      //      NEXT step's split (keys drawn in the first accept phase) — the ranking rides on the barriers that exist ----
      FINE_START
      if (kPairPropose && 2 * Hs <= NT && !Eval::kNeedsPrepare) {
        // two threads per proposal, the dimensions interleaved between them (round 2d: the threads beyond Hs idled here
        // and the dependent chain of one thread per proposal was ~1,400 cycles for six dimensions); same arithmetic per
        // dimension, so positions stay bit-identical.  Used by the clustered evaluators only (kPairPropose); never for the
        // vector models: their row constants (exp, sincospi, divisions) would be prepared on half-filled warps.
        const int q = tid >> 1, sub = tid & 1;
        bool ok = true;
        if (q < Hs) {
          const int j = list[coff + s.partner[q]];
          const int k = list[off + q];
          ok = propose_pair(s.coords + j * ndim, s.coords + k * ndim, zzb[q], s.prop + q * ndim, s.bkey, ndim, sub);
        }
        const unsigned okm = __ballot_sync(0xffffffffu, ok);
        if (q < Hs && sub == 0) s.inb[q] = ((okm >> ((tid & 31) & ~1)) & 3u) == 3u ? 1 : 0;
      } else {
        for (int q = tid; q < Hs; q += NT) {
          const int j = list[coff + s.partner[q]];
          const int k = list[off + q];
          s.inb[q] = propose_and_check(s.coords + j * ndim, s.coords + k * ndim, zzb[q], s.prop + q * ndim, s.bkey, ndim) ? 1 : 0;
          ev.prepare_row(q, s.prop + q * ndim);
        }
      }
      FINE_MARK(6)
      __syncthreads();
      FINE_MARK(7)
      PHASE_MARK(1)
      // ---- EVAL: fused forward + chi^2 of all proposals ----------------------------------------------
      ev.eval_chi(s.prop, ndim, Hs, s.chi, side);
      FINE_MARK(8)
      __syncthreads();
      FINE_MARK(9)
      PHASE_MARK(2)
      // ---- ACCEPT (threads [0,Hs)) while the other threads draw the random numbers of the next half-step (measured:
      //      running the draws as side work under the evaluation instead is 5-8 % slower for every evaluator — they
      //      land on the evaluation's critical path, here they are off it); then the shuffle keys of the next step
      //      (first half-step) or the scan + placement of its key ranking (second half-step) ---------------------------
      {
        const int nspare = NT - min(Hs, NT);
        const bool spare = tid >= Hs;
        if (spare || nspare == 0)
          draw_rows(dctx, sp == 0 ? t : t + 1u, sp ^ 1, spare ? tid - Hs : tid, spare ? nspare : NT);
      }
      for (int q = tid; q < Hs; q += NT) {
        const int k = list[off + q];
        const double lpo = s.lp[k];
        const double lpn = s.inb[q] ? -0.5 * (ev.chi_of(s.chi, q) + llc) : neg_inf();
        if (lpn != lpn) flag |= 1;
        // emcee: accept iff (ndim-1) ln zz + lp' - lp > ln u.  The logarithms were taken in FP32
        // (|error| < 1e-5): unless the margin is below the threshold the FP64 decision is already
        // determined; otherwise (about 1 proposal in 10^4) it is recomputed in FP64 as the oracle does.
        const double est = __dsub_rn(lpn, lpo) + f32_widen_int(lfb[q]);
        bool accept;
        if (!accept_filter(est, lpn, lpo, accept)) {
          const u32x4 r = philox4x32_10((uint32_t)q, t, spec, (uint32_t)(1 + sp), k0, k1);     // re-draw u2
          const double lnpdiff = __dsub_rn(__dadd_rn(__dmul_rn((double)(ndim - 1), log(zzb[q])), lpn), lpo);
          accept = lnpdiff > log(u53_int(r.w, (r.z << 16) | 0x8000u));
        }
        if (accept) {
          copy_dims(s.coords + k * ndim, s.prop + q * ndim, ndim);
          s.lp[k] = lpn;
          s.acc[k] += 1;
        }
      }
      FINE_MARK(10)
      if (sp == 0) {
        gen_keys(t + 1u, tid, NT);
        if (binned && !kLegacyRank)                  // bin counters of the ranking at the end of this step (last read: the
          for (int i = tid; i < 256; i += NT) s.hist[i] = 0;   // previous step's ranking, two barriers ago)
      }
      else if (binned && kRankInAccept && !kLegacyRank) {
        // second half-step: bin slot of this thread's key of the NEXT step's split (keys drawn and counters zeroed one
        // half-step ago) — the first of the ranking's barriers is the one that ends this accept phase
        rk_key = 0; rk_bin = 0; rk_slot = 0;
        if (tid < W) {
          rk_key = s.keys[tid];
          rk_bin = (int)(rk_key >> 24);
          rk_slot = atomicAdd(&s.hist[rk_bin], 1);
        }
      }
      FINE_MARK(11)
      __syncthreads();
      PHASE_MARK(3)
    }
    // ---- split of the next step: rank its keys (drawn during this step's first accept phase; bin slots taken in the
    //      second one): scan | barrier | placement | barrier | count.  (Spreading ALL of the binned ranking over the
    //      barriers of the second half-step, as the warp-private kernel does, measured 2-3 % slower here: the per-warp
    //      scan lands on the accept phase of all eight warps.) ---------------------------------------------------------
    if (binned && kLegacyRank) {
      rank_keys_binned<NT>(s.keys, list_next, W, s.hist, s.sorted);     // 4 barriers inside
      __syncthreads();                               // (and the doubled barrier below: see kLegacyRank)
    } else if (binned) {
      if (!kRankInAccept) {                          // bin slots in a phase of their own (one more barrier)
        rk_key = 0; rk_bin = 0; rk_slot = 0;
        if (tid < W) {
          rk_key = s.keys[tid];
          rk_bin = (int)(rk_key >> 24);
          rk_slot = atomicAdd(&s.hist[rk_bin], 1);
        }
        __syncthreads();
      }
      rank_binned_rest<NT>(list_next, W, s.hist, s.sorted, rk_key, rk_bin, rk_slot);
    } else {
      side.begin(s.keys, list_next, W, 0);
      side.finish();
    }
    PHASE_MARK(0)
    // the proposals of the next step read list_next: synchronise here (round 2c: once — this barrier was doubled)
    __syncthreads();
    // ---- backend.save_step: chain[it] = coords ; log_prob[it] = lp (reads only; the next writer of coords / lp is the
    //      next accept phase, two barriers away) -----------------------------------------------------------------------
    if (it >= first && (it - first) % P.thin == 0) {
      if (P.chain != nullptr && writer) {
        double* dst = P.chain + ((size_t)b * P.nkeep + kept) * W * ndim;
        for (int i = tid; i < W * ndim; i += NT) __stcs(dst + i, s.coords[i]);
      }
      if (P.logp != nullptr && writer) {
        double* dst = P.logp + ((size_t)b * P.nkeep + kept) * W;
        for (int i = tid; i < W; i += NT) __stcs(dst + i, s.lp[i]);
      }
      ++kept;
    }
    PHASE_MARK(4)
  }
  PHASE_PRINT
  // ---- final state ------------------------------------------------------------------------------
  if (writer) {
    double* gco = P.coords + (size_t)b * W * ndim;
    for (int i = tid; i < W * ndim; i += NT) gco[i] = s.coords[i];
    for (int i = tid; i < W; i += NT) {
      if (P.lp) P.lp[(size_t)b * W + i] = s.lp[i];
      if (P.accepted) P.accepted[(size_t)b * W + i] = s.acc[i];
    }
    if (P.flags && flag) atomicOr(P.flags + b, flag);
  }
  ev.release();
  if (Eval::kClustered && cs > 1) cg::this_cluster().sync();   // peers may still read our shared memory
}

}  // namespace bisip
