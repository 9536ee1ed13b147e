// conviqt_interp.cuh -- the psi lookup of comm_conviqt%interp (commander3/src/comm_conviqt_mod.f90:155-205) and the
// local -> RING placement of the sampler's full-sky table.  Plain C++ apart from the __host__ __device__ markers, so
// that g++ compiles it for the CPU tests (tests/host_emul/emul_conviqt_interp.cpp) and nvcc for conviqt_interp.cu.
#pragma once
#include <math.h>

#include <algorithm>
#include <cmath>
#include <limits>
#include <string>
#include <vector>

#ifdef __CUDACC__
#define CVQ_HD __host__ __device__
#else
#define CVQ_HD
#endif

namespace cmdr {

// Single-precision operations that nvcc may not contract into an FMA: the reference (and oracle/conviqt.py) rounds
// after every multiply.  On the host (g++, built with -ffp-contract=off) plain operators round the same way.
CVQ_HD inline float cvq_mul(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
CVQ_HD inline float cvq_add(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
CVQ_HD inline float cvq_sub(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fsub_rn(a, b);
#else
  return a - b;
#endif
}
CVQ_HD inline float cvq_div(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fdiv_rn(a, b);
#else
  return a / b;
#endif
}
CVQ_HD inline float cvq_nan() {
#ifdef __CUDA_ARCH__
  return __int_as_float(0x7fffffff);
#else
  return std::numeric_limits<float>::quiet_NaN();
#endif
}

// psires = real(2 pi / psisteps, sp) and 2 pi in single precision, as the constructor sets them (:39, :91-92)
inline float cvq_psires(int psisteps) { return (float)(2.0 * 3.14159265358979323846 / psisteps); }
inline float cvq_twopi() { return (float)(2.0 * 3.14159265358979323846); }

// interp(pix, psi), :155-205, for one sample of the table tab[psisteps][npix] (global RING pixel order).  Same float
// operations in the same order as the reference: unwrap = modulo(-psi, 2 pi); optim == 2 takes the nearest of the
// psisteps bins, any other value interpolates linearly between bins psii and psii + 1 (cyclic).
// Beyond the reference, which has no answer for them:
//  * a pixel outside 0 .. npix - 1, and a psi that is not finite, give NaN;
//  * when -psi is a tiny positive number, unwrap rounds up to 2 pi and psii to psisteps, one row past the cube in the
//    reference; the row read is then row 0 (the same angle), with x0 = psisteps * psires kept in the weights.
CVQ_HD inline float conviqt_interp_sample(const float *tab, long long npix, int psisteps, float psires, float twopi,
                                          int optim, int pix, float psi) {
  if (pix < 0 || (long long)pix >= npix) return cvq_nan();
  float unwrap = fmodf(-psi, twopi);
  if (unwrap < 0.0f) unwrap = cvq_add(unwrap, twopi);      // Fortran modulo: the sign of the divisor
  if (unwrap != unwrap) return cvq_nan();
  const float q = cvq_div(unwrap, psires);
  if (optim == 2) {
    int b = (int)rintf(q);
    if (b < 0) b = 0;
    if (b >= psisteps) b = 0;
    return tab[(long long)b * npix + pix];
  }
  const int psii = (int)q;
  int psiu = psii + 1;
  if (psiu >= psisteps) psiu = 0;
  const float x0 = cvq_mul((float)psii, psires), x1 = cvq_mul((float)psiu, psires);
  const float c0 = tab[(long long)(psii >= psisteps ? 0 : psii) * npix + pix], c1 = tab[(long long)psiu * npix + pix];
  return cvq_div(cvq_add(cvq_mul(c0, cvq_sub(x1, unwrap)), cvq_mul(c1, cvq_sub(unwrap, x0))), cvq_sub(x1, x0));
}

// ---- the sampler's table, built from the ranks' local cubes (host side) ------------------------------------------

// HEALPix ring scheme (comm_map._ring_start / _in_ring_count)
inline long long cvq_ring_npix(int nside, int ring) {
  const int north = ring > 2 * nside ? 4 * nside - ring : ring;
  return north < nside ? 4LL * north : 4LL * nside;
}
inline long long cvq_ring_start(int nside, int ring) {
  const long long npix = 12LL * nside * nside;
  const int north = ring > 2 * nside ? 4 * nside - ring : ring;
  const long long ofs = north < nside ? 2LL * north * (north - 1)
                                      : 2LL * nside * (nside - 1) + (long long)(north - nside) * 4 * nside;
  return north == ring ? ofs : npix - cvq_ring_npix(nside, ring) - ofs;
}

// One contiguous stretch of a 2-D copy: for every row k, dst[dst + k * dst_pitch + j] = src[src + k * src_pitch + j],
// j < n.  Stretches are at most CVQ_RUN elements long so that a copy of few long stretches still fills the GPU.
struct CvqRun {
  long long src, dst;
  int n;
};
constexpr int CVQ_RUN = 4096;

inline void cvq_add_runs(std::vector<CvqRun> &runs, long long src, long long dst, long long n) {
  for (long long j = 0; j < n; j += CVQ_RUN) runs.push_back({src + j, dst + j, (int)std::min<long long>(CVQ_RUN, n - j)});
}

// Checks the ring lists of the ranks (1-based ring numbers, each rank's in its geometry's storage order): no ring twice
// and, with `whole`, every ring of an nside map held by some rank.  Returns the reason of a refusal, or an empty string.
inline std::string cvq_check_rings(int nside, const std::vector<std::vector<int>> &rings, bool whole) {
  if (nside < 1 || 12.0 * nside * nside > 2147483647.0)
    return "nside " + std::to_string(nside) + " unsupported (pixel numbers are 32-bit: 12 nside^2 <= 2^31 - 1)";
  std::vector<int> seen(4 * nside, 0);
  for (const auto &rr : rings)
    for (int r : rr) {
      if (r < 1 || r > 4 * nside - 1) return "ring " + std::to_string(r) + " outside 1.." + std::to_string(4 * nside - 1);
      if (seen[r]++) return "ring " + std::to_string(r) + " held twice";
    }
  if (!whole) return "";
  for (int r = 1; r < 4 * nside; ++r)
    if (!seen[r])
      return "ring " + std::to_string(r) + " held by no rank: the geometries must cover the sphere (the full-sky geometry "
             "on one GPU, comm_mapinfo's round-robin rings on several)";
  return "";
}

// The placement of every rank's local pixels in the table: rank r's cube block starts at r * rank_stride in the source
// (rows src_pitch apart) and holds its rings in geometry order, each ring's pixels following the previous ring's
// (the running sum of nph); ring `ring` lands at its RING-scheme start in a table with rows of 12 nside^2 pixels.
inline std::vector<CvqRun> cvq_scatter_runs(int nside, const std::vector<std::vector<int>> &rings, long long rank_stride) {
  std::vector<CvqRun> runs;
  for (size_t r = 0; r < rings.size(); ++r) {
    long long loc = 0;
    for (int ring : rings[r]) {
      const long long n = cvq_ring_npix(nside, ring);
      cvq_add_runs(runs, (long long)r * rank_stride + loc, cvq_ring_start(nside, ring), n);
      loc += n;
    }
  }
  return runs;
}

}  // namespace cmdr
