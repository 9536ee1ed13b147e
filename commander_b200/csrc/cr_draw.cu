// cr_draw.cu -- the fluctuation terms of cr_computeRHS (commander3/src/comm_cr_mod.f90:542-769) drawn on the device from
// the counter-based stream of rng.cuh, for both system kinds (cr.cu, cr_multi.cu):
//   * k_rhs_map_draw: m = N^-1 d + sqrt(N^-1) eta(q, j, p) for one band and map, one CTA per local ring (table of
//     cr_draw.h), threads along the ring: the global pixel index is the ring's RING start plus the thread's offset;
//   * k_eta_alm_draw: eta_0 of one component at its local real-packed slots, one CTA per (local m, map), threads over l.
// Per pixel the map pass reads 16 B (N^-1, d; 8 B without data), writes 8 B and runs one Philox4x32-10, one FP64 log, one
// sqrt and one cospi.
#include <cmath>

#include "kernels.h"
#include "rng.cuh"

namespace cmdr {

namespace {

constexpr int NTHR = 256;

// m = N^-1 d + sqrt(N^-1) eta in the expression order of k_rhs_map (cr.cu), so that cr_computeRHS fed with the
// materialised draws gives the same bits; d == nullptr: d = 0; invN == nullptr: m = eta (the draws alone)
__global__ void __launch_bounds__(NTHR) k_rhs_map_draw(double *__restrict__ m, const double *__restrict__ invN,
                                                      const double *__restrict__ d, const CrRing *__restrict__ rings,
                                                      unsigned long long seed, unsigned long long draw, unsigned column) {
  const CrRing r = rings[blockIdx.x];
  for (int t = threadIdx.x; t < r.nph; t += NTHR) {
    const long long i = r.loc + t;
    const double eta = rng_draw(seed, draw, (uint32_t)(r.glob + t), column);
    if (!invN) {
      m[i] = eta;
      continue;
    }
    double v = invN[i] * (d ? d[i] : 0.0);
    v = fma(sqrt(invN[i]), eta, v);
    m[i] = v;
  }
}

// out[j * stride + slot] = eta_0(k, j, l, m_s) at every local real-packed slot of `a`
__global__ void __launch_bounds__(NTHR) k_eta_alm_draw(double *__restrict__ out, long long stride, int lmax,
                                                      const int *__restrict__ mval, const long long *__restrict__ mvstart,
                                                      unsigned long long seed, unsigned long long draw, unsigned k) {
  const int m = mval[blockIdx.x], j = blockIdx.y;
  double *o = out + (long long)j * stride + mvstart[blockIdx.x];
  for (int l = m + threadIdx.x; l <= lmax; l += NTHR) {
    if (m == 0) {
      o[l] = rng_eta_alm(seed, draw, k, j, l, 0);
    } else {                                         // (l, +m) at 2 l, (l, -m) right after it
      o[2 * l] = rng_eta_alm(seed, draw, k, j, l, m);
      o[2 * l + 1] = rng_eta_alm(seed, draw, k, j, l, -m);
    }
  }
}

}  // namespace

CrRing *cr_ring_table_device(const sharp_geom_info *g) { return upload(cr_ring_table(g->nside, g->ring)); }

void cr_draw_pix(double *dst, const CrRing *rings, int nrings, long long np, unsigned long long seed, unsigned long long draw,
                 int q, int j, cudaStream_t st) {
  if (!np) return;
  double *out = dst;
  if (!is_device_ptr(dst)) out = static_cast<double *>(scratch_get("cr_draw_pix", sizeof(double) * np));
  k_rhs_map_draw<<<nrings, NTHR, 0, st>>>(out, nullptr, nullptr, rings, seed, draw, rng_pix_column(q, j));
  count_launch(1);
  if (out != dst) CMDR_CUDA_CHECK(cudaMemcpyAsync(dst, out, sizeof(double) * np, cudaMemcpyDeviceToHost, st));
}

void cr_draw_alm(double *out, long long stride, sharp_alm_info *a, int nmaps, unsigned long long seed, unsigned long long draw,
                 int k, cudaStream_t st) {
  if (!a->nm) return;
  ensure_alm_device(a);
  k_eta_alm_draw<<<dim3((unsigned)a->nm, (unsigned)nmaps), NTHR, 0, st>>>(out, stride, a->lmax, a->d_mval, a->d_mvstart, seed,
                                                                          draw, (unsigned)k);
  count_launch(1);
}

void cr_rhs_column(double *m, const double *invN, const double *data_col, const RhsEta &eta, int col, int q, int j, long long np,
                   const CrRing *rings, int nrings, double *tmp, cudaStream_t st) {
  if (!np) return;
  const double *d = nullptr;
  if (data_col) {
    CMDR_CUDA_CHECK(cudaMemcpyAsync(tmp, data_col, sizeof(double) * np, cudaMemcpyDefault, st));
    d = tmp;
  }
  if (!eta.draw) {
    if (eta.pix) CMDR_CUDA_CHECK(cudaMemcpyAsync(tmp + np, eta.pix[col], sizeof(double) * np, cudaMemcpyDefault, st));
    cr_rhs_map(m, invN, d, eta.pix ? tmp + np : nullptr, np, st);
  } else if (eta.terms & CMDR_CR_ETA_PIX) {
    k_rhs_map_draw<<<nrings, NTHR, 0, st>>>(m, invN, d, rings, eta.seed, eta.index, rng_pix_column(q, j));
    count_launch(1);
  } else if (d) {
    cr_rhs_map(m, invN, d, nullptr, np, st);
  } else {
    CMDR_CUDA_CHECK(cudaMemsetAsync(m, 0, sizeof(double) * np, st));
  }
}

}  // namespace cmdr
