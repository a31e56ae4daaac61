// Counter-based Gaussian noise: Philox4x32-10 (Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as
// 1, 2, 3", SC 2011; the rounds and constants of Random123), the exact uniform mapping and the Box-Muller pair of
// k_row_noise (csrc/row_noise.cu).  Host and device code, so that tests/host/philox_host_check.cu can check the
// generator against the Random123 known-answer vectors without a GPU.
//
// The noise contract (DESIGN.md 4.8): for row seed s, draw index d and sample n of the row,
//   key (s & 0xffffffff, s >> 32), counter (n / 4, d, 0, 0) -> words x0..x3,
//   u(x) = (2 (x >> 9) + 1) 2^-24,
//   samples 4j, 4j+1 = r cos(theta), r sin(theta) with r = sqrt(-2 ln u(x0)), theta = 2 pi u(x1);
//   samples 4j+2, 4j+3 the same from x2, x3.
#pragma once
#include <math.h>
#include <stdint.h>

#ifndef BABE_HD
#define BABE_HD __host__ __device__ __forceinline__
#endif

namespace babe {

constexpr uint32_t kPhiloxM0 = 0xD2511F53u, kPhiloxM1 = 0xCD9E8D57u;   // round multipliers
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u, kPhiloxW1 = 0xBB67AE85u;   // key schedule (golden ratio, sqrt(3) - 1)

struct Philox4 {
  uint32_t x[4];
};

BABE_HD uint32_t philox_mulhi(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

// Philox4x32 with 10 rounds: counter (c0, c1, c2, c3), key (k0, k1).
BABE_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = philox_mulhi(kPhiloxM0, c0), lo0 = kPhiloxM0 * c0;
    const uint32_t hi1 = philox_mulhi(kPhiloxM1, c2), lo1 = kPhiloxM1 * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += kPhiloxW0;
    k1 += kPhiloxW1;
  }
  Philox4 o;
  o.x[0] = c0; o.x[1] = c1; o.x[2] = c2; o.x[3] = c3;
  return o;
}

// u(x) = (2 (x >> 9) + 1) 2^-24: an odd multiple of 2^-24 below 2^24, exact in fp32, in [2^-24, 1 - 2^-24].
BABE_HD float philox_uniform(uint32_t x) {
  return (float)(((x >> 9) << 1) | 1u) * 5.9604644775390625e-8f;
}

// Box-Muller on two words: (r cos(2 pi u1), r sin(2 pi u1)) with r = sqrt(-2 ln u0).  u0 >= 2^-24 bounds r by
// sqrt(48 ln 2) = 5.77: the tails beyond 5.77 sigma are cut.
BABE_HD void box_muller(uint32_t x0, uint32_t x1, float* n0, float* n1) {
  const float r = sqrtf(-2.0f * logf(philox_uniform(x0)));
  const float v = 2.0f * philox_uniform(x1);            // exact: theta = pi v
  float s, c;
#ifdef __CUDA_ARCH__
  sincospif(v, &s, &c);
#else
  const double th = 3.14159265358979323846 * (double)v; // host builds serve the generator checks only
  s = (float)sin(th);
  c = (float)cos(th);
#endif
  *n0 = r * c;
  *n1 = r * s;
}

// The four samples 4j .. 4j+3 of row seed s, draw d.
BABE_HD void row_noise4(uint64_t seed, uint32_t draw, uint32_t j, float out[4]) {
  const Philox4 w = philox4x32_10(j, draw, 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
  box_muller(w.x[0], w.x[1], &out[0], &out[1]);
  box_muller(w.x[2], w.x[3], &out[2], &out[3]);
}

}  // namespace babe
