// Shared device helpers: Philox4x32-10, DMMA wrappers, small math.  sm_100a only.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/bisip_b200.h"

#ifndef __CUDA_ARCH__
#define BISIP_HOST_PASS 1
#endif

namespace bisip {

constexpr int kThreads = 256;   // CTA size of every hot-path kernel
constexpr int kWarps = kThreads / 32;

// ---------------------------------------------------------------- Philox4x32-10
// Salmon et al. 2011 (Random123).  Same stream as oracle/bisip_oracle.c (KAT-tested there).
struct u32x4 { uint32_t x, y, z, w; };

__device__ __forceinline__ u32x4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return {c0, c1, c2, c3};
}

// NumPy legacy random_sample recipe: 53-bit uniform in [0,1)
__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  return __dmul_rn(__dadd_rn(__dmul_rn((double)(a >> 5), 67108864.0), (double)(b >> 6)),
                   1.0 / 9007199254740992.0);
}

// The same number built on the INTEGER pipe: (a>>5) 2^26 + (b>>6) is a 53-bit integer m, and m 2^-53 is exact in
// binary64, so assembling sign / exponent / mantissa from clz gives the identical bits without the two int->double
// conversions, the multiply and the add — FP64-pipe instructions that, in the sampler's serial phases, queue behind
// the co-resident warps' DMMA / DFMA streams (ncu: the FP64 ops of those phases draw 5-8x the stall samples of an
// integer op).
__device__ __forceinline__ double u53_int(uint32_t a, uint32_t b) {
  const unsigned long long m = ((unsigned long long)(a >> 5) << 26) | (unsigned long long)(b >> 6);
  const int lz = __clzll((long long)m);                       // m < 2^53: lz >= 11
  const unsigned long long mant = (m << (lz + 1)) >> 12;      // drop the leading one; the 12 bits shifted out are zero
  const unsigned long long bits = ((unsigned long long)(1033 - lz) << 52) | mant;
  return m ? __longlong_as_double((long long)bits) : 0.0;
}

// float -> double widening (exact) on the integer pipe; denormal floats flush to zero (callers pass O(1) numbers)
__device__ __forceinline__ double f32_widen_int(float f) {
  const uint32_t b = __float_as_uint(f);
  const uint32_t e = (b >> 23) & 0xffu;
  const uint32_t hi = (b & 0x80000000u) | ((e + 896u) << 20) | ((b >> 3) & 0xfffffu);
  return e ? __hiloint2double((int)hi, (int)(b << 29)) : 0.0;
}

// ---------------------------------------------------------------- FP64 tensor tiles
// mma.sync .f64 lowers to DMMA.8x8x4 on sm_100a (tools/peaks.cu verifies the fragment maps):
//   A (16xK):  a[i] -> row g + 8*(i&1), col t + 4*(i>>1)
//   B (Kx8):   b[i] -> row t + 4*i,     col g
//   C (16x8):  c0,c1 -> row g, cols 2t,2t+1 ; c2,c3 -> row g+8        (g = lane>>2, t = lane&3)
__device__ __forceinline__ void dmma_16x8x8(double (&d)[4], const double (&a)[4], const double (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+d"(d[0]), "+d"(d[1]), "+d"(d[2]), "+d"(d[3])
      : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(b[0]), "d"(b[1]));
}
__device__ __forceinline__ void dmma_16x8x16(double (&d)[4], const double (&a)[8], const double (&b)[4]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, "
      "{%12,%13,%14,%15}, {%0,%1,%2,%3};"
      : "+d"(d[0]), "+d"(d[1]), "+d"(d[2]), "+d"(d[3])
      : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(a[4]), "d"(a[5]), "d"(a[6]), "d"(a[7]),
        "d"(b[0]), "d"(b[1]), "d"(b[2]), "d"(b[3]));
}

__device__ __forceinline__ double neg_inf() { return __longlong_as_double(0xfff0000000000000LL); }

__host__ __device__ __forceinline__ int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ __forceinline__ size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace bisip
