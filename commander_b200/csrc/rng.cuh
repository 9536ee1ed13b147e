// rng.cuh -- the counter-based Gaussian stream of the constrained-realisation fluctuation terms (cr_computeRHS,
// commander3/src/comm_cr_mod.f90:542-769: eta_q per pixel and map of every band, eta_0 per amplitude of each component
// with a prior).  Every draw is a function of (seed, draw, global index) alone, so a sample does not depend on how many
// GPUs hold the maps or which of them owns a pixel or an m.  Plain C++ apart from the __host__ __device__ markers, so
// that g++ compiles it for the CPU tests (tests/host_emul/emul_rng.cpp) and nvcc for cr_draw.cu; oracle/rng.py restates
// it in numpy.
//
// The stream (the contract the oracle and the tests hold it to):
//   Philox4x32-10 as curand_Philox4x32_10 (curand_philox4x32_x.h): M0 = 0xD2511F53, M1 = 0xCD9E8D57, key bumped by
//     (0x9E3779B9, 0xBB67AE85) between rounds; round (hi(M1 c.z) ^ c.y ^ k.x, lo(M1 c.z), hi(M0 c.x) ^ c.w ^ k.y, lo(M0 c.x)).
//   key = (seed lo, seed hi)
//   pixel draw of band q, map j (0..2), global RING pixel p:  counter (p, q << 2 | j, draw lo, draw hi)
//   prior draw of component k, map j, a_lm (l, m_s):         counter (l^2 + l + m_s, 0x80000000 | k << 2 | j, draw lo, draw hi)
//     m_s = +m for the real-packed alm[+m] slot, -m for alm[-m], 0 for m = 0 (comm_map.alm_to_chain_order's index)
//   Gaussian of the words (r0, r1, r2, r3): x1 = r0 << 21 | r1 >> 11, x2 likewise (53 bits each),
//     u1 = (x1 + 1) 2^-53 in (0, 1], u2 = x2 2^-53 in [0, 1), eta = sqrt(-2 log u1) cospi(2 u2).
//     One Gaussian per counter: the second Box-Muller value is dropped so that every (column, index) is addressable alone.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define RNG_HD __host__ __device__
#else
#define RNG_HD
#endif

namespace cmdr {

struct RngWords {
  uint32_t x, y, z, w;
};

constexpr uint32_t PHILOX_M0 = 0xD2511F53u, PHILOX_M1 = 0xCD9E8D57u;
constexpr uint32_t PHILOX_W0 = 0x9E3779B9u, PHILOX_W1 = 0xBB67AE85u;
constexpr uint32_t RNG_PRIOR_BIT = 0x80000000u;

RNG_HD inline uint32_t rng_mulhi(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

RNG_HD inline RngWords philox4x32_10(RngWords c, uint32_t k0, uint32_t k1) {
#ifdef __CUDACC__
#pragma unroll
#endif
  for (int r = 0; r < 10; ++r) {
    if (r) { k0 += PHILOX_W0; k1 += PHILOX_W1; }
    const uint32_t hi0 = rng_mulhi(PHILOX_M0, c.x), lo0 = PHILOX_M0 * c.x;
    const uint32_t hi1 = rng_mulhi(PHILOX_M1, c.z), lo1 = PHILOX_M1 * c.z;
    c = RngWords{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
  }
  return c;
}

// One standard Gaussian from four Philox words (Box-Muller, first value)
RNG_HD inline double rng_gauss(RngWords r) {
  const uint64_t x1 = ((uint64_t)r.x << 21) | (r.y >> 11), x2 = ((uint64_t)r.z << 21) | (r.w >> 11);
  const double u1 = (double)(x1 + 1) * 0x1p-53, u2 = (double)x2 * 0x1p-53;
#ifdef __CUDA_ARCH__
  return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
#else
  return sqrt(-2.0 * log(u1)) * cos(2.0 * M_PI * u2);   // libm has no cospi: within 1e-14 of the device value
#endif
}

RNG_HD inline double rng_draw(uint64_t seed, uint64_t draw, uint32_t index, uint32_t column) {
  return rng_gauss(philox4x32_10(RngWords{index, column, (uint32_t)draw, (uint32_t)(draw >> 32)}, (uint32_t)seed,
                                 (uint32_t)(seed >> 32)));
}

// column word of a pixel draw (band q, map j) and of a prior draw (component k, map j)
RNG_HD inline uint32_t rng_pix_column(uint32_t q, uint32_t j) { return (q << 2) | j; }
RNG_HD inline uint32_t rng_prior_column(uint32_t k, uint32_t j) { return RNG_PRIOR_BIT | (k << 2) | j; }

// eta of global RING pixel p in map j of band q
RNG_HD inline double rng_eta_pix(uint64_t seed, uint64_t draw, uint32_t q, uint32_t j, uint32_t p) {
  return rng_draw(seed, draw, p, rng_pix_column(q, j));
}

// eta_0 of (l, m_s) in map j of component k (m_s: +m for alm[+m], -m for alm[-m], 0 for m = 0)
RNG_HD inline double rng_eta_alm(uint64_t seed, uint64_t draw, uint32_t k, uint32_t j, int l, int ms) {
  const uint32_t ul = (uint32_t)l;
  return rng_draw(seed, draw, ul * ul + ul + (uint32_t)ms, rng_prior_column(k, j));
}

}  // namespace cmdr
