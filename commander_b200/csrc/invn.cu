// invn.cu -- diagonal of the inverse noise covariance in harmonic space, N^-1_{lm,lm}: the input of the
// diagonal CG preconditioner.  Replaces `compute_invN_lm`, commander3/src/comm_N_mod.f90:127-197.
//
// The reference sums products of Wigner 3j symbols (SLATEC DRC3JJ, two calls per (l,m)):
//     N_lm = (-1)^m (2l+1)/sqrt(4pi) npix/(4pi) sum_{L<=min(2l,lmax)} a_L0 sqrt(2L+1) (l l L; -m m 0)(l l L; 0 0 0)
// where a_L0 are the m=0 coefficients of YtW(N^-1 map).  The summand is the Gaunt integral of
// |Y_lm|^2 Y_L0, so the whole sum is an integral over the sphere of |Y_lm|^2 times the azimuthally averaged
// inverse-noise profile nbar(x) = sum_L a_L0 lambda_L0(x):
//     N_lm = npix/(4pi) 2pi int_{-1}^{1} lambda_lm(x)^2 nbar(x) dx .
// The integrand is a polynomial in x of degree <= 2l + lmax <= 3 lmax, so Gauss-Legendre quadrature with
// K >= (3 lmax + 1)/2 nodes reproduces the 3j sum exactly (to rounding), and what remains is the loop this
// library already runs at speed: the lambda_lm recurrence over l for many colatitudes at once, here with a
// squared accumulate.  No 3j recursion, O(lmax^3) FMAs on the FP64 pipe instead of on 16 host threads.
//
// One warp per (local m, block of 32*R nodes); x -> -x symmetry folds the nodes to the positive half.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

#include "det.h"
#include "kernels.h"
#include "legendre_core.cuh"

namespace cmdr {

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr double SCALE_DOWN_D = 7.458340731200207e-155;   // 2^-512

struct InvNParams {
  int lmax, nm, nnodes, nmaps;
  const int *mval;
  const long long *mvstart, *cofs;
  const double *coef, *Kstart;
  const double *trig;      // nnodes * 4: cth, sth, sh, ch
  const double *f;         // nmaps * nnodes: folded weight * profile, see cmdr_sht_invn_diag
  double *out[3];
  long long nalm;
  // deterministic mode (det.h): partials of component c at det + c * dl.comp_stride(), one value per l (part 0), local m's
  // from dl.im0; every (node block, m, l) is stored, so no records are needed
  double *det;
  DetLayout dl;
};

// DET: lane 0 stores each l's sum of the warp (0.0 where the warp is below the threshold) instead of adding it to out
template <int R, int NM, bool DET = false>
__global__ void __launch_bounds__(32, 16) invn_kernel(InvNParams p) {
  const int im = (DET ? p.dl.im0 : 0) + blockIdx.y, m = p.mval[im];
  const int lane = threadIdx.x;
  const int node0 = blockIdx.x * (32 * R);
  double x[R], cur[R], prev[R], f[R][NM];
  int k[R];
  const double K = p.Kstart[m];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int n = node0 + lane * R + r;
    x[r] = cur[r] = prev[r] = 0.0; k[r] = 0;
#pragma unroll
    for (int c = 0; c < NM; ++c) f[r][c] = 0.0;
    if (n < p.nnodes) {
      const double4 tg = reinterpret_cast<const double4 *>(p.trig)[n];
      RingTrig g{tg.x, tg.y, tg.z, tg.w};
      x[r] = g.cth;
      start_spin0(m, K, g, cur[r], k[r]);
#pragma unroll
      for (int c = 0; c < NM; ++c) f[r][c] = p.f[(size_t)c * p.nnodes + n];
    }
  }
  const double2 *coef = reinterpret_cast<const double2 *>(p.coef + p.cofs[im]);   // {A'_l, g_l}, row l - m
  const long long mvs = p.mvstart[im];
  for (int l0 = m; l0 <= p.lmax; l0 += 8) {
    bool none_on = true;
#pragma unroll
    for (int r = 0; r < R; ++r) none_on &= (k[r] < 0);
    const bool skip = __all_sync(FULL, none_on);      // nothing above 2^-70 yet: recurrence only
    const int nl = min(8, p.lmax - l0 + 1);
    for (int j = 0; j < nl; ++j) {
      const int l = l0 + j;
      const double2 cg = coef[l - m];
      if (DET && skip && lane == 0)
#pragma unroll
        for (int c = 0; c < NM; ++c) p.det[c * p.dl.comp_stride() + p.dl.index(0, blockIdx.x, im, l, 0)] = 0.0;
      if (!skip) {
        double s[NM];
#pragma unroll
        for (int c = 0; c < NM; ++c) s[c] = 0.0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const double v = k[r] == 0 ? cur[r] : 0.0;
          const double v2 = v * v;
#pragma unroll
          for (int c = 0; c < NM; ++c) s[c] = fma(v2, f[r][c], s[c]);
        }
#pragma unroll
        for (int c = 0; c < NM; ++c) {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) s[c] += __shfl_xor_sync(FULL, s[c], o);
        }
        if (lane == 0) {
          const double g2 = cg.y * cg.y;
#pragma unroll
          for (int c = 0; c < NM; ++c) {
            const double val = g2 * s[c];
            if (DET) {
              p.det[c * p.dl.comp_stride() + p.dl.index(0, blockIdx.x, im, l, 0)] = val;
            } else if (m == 0) {
              atomicAdd(p.out[c] + mvs + l, val);
            } else {
              atomicAdd(p.out[c] + mvs + 2 * (long long)l, val);
              atomicAdd(p.out[c] + mvs + 2 * (long long)l + 1, val);
            }
          }
        }
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const double nxt = step0(cg.x, x[r], cur[r], prev[r]);
        prev[r] = cur[r]; cur[r] = nxt;
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (k[r] < 0 && needs_rescale(cur[r])) { cur[r] *= SCALE_DOWN_D; prev[r] *= SCALE_DOWN_D; ++k[r]; }
  }
}

// Ordered reduce of the deterministic mode: out = out + (sum over node blocks in ascending order), both entries of an
// m > 0 pair getting the same value as with the atomics
template <int NM>
__global__ void __launch_bounds__(256) invn_reduce_kernel(InvNParams p) {
  const int im = p.dl.im0 + blockIdx.y, m = p.mval[im];
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < m || l > p.lmax) return;
  const long long mvs = p.mvstart[im];
  const size_t bstride = (size_t)p.dl.nm * p.dl.row();
#pragma unroll
  for (int c = 0; c < NM; ++c) {
    const double *src = p.det + c * p.dl.comp_stride() + p.dl.index(0, 0, im, l, 0);
    double s = 0.0;
    for (int b = 0; b < p.dl.nb; ++b) s += src[(size_t)b * bstride];
    if (m == 0) {
      p.out[c][mvs + l] = p.out[c][mvs + l] + s;
    } else {
      p.out[c][mvs + 2 * (long long)l] = p.out[c][mvs + 2 * (long long)l] + s;
      p.out[c][mvs + 2 * (long long)l + 1] = p.out[c][mvs + 2 * (long long)l + 1] + s;
    }
  }
}

// Positive half of the K-point Gauss-Legendre rule (K even): Newton iteration on P_K in long double.
void gauss_legendre_half(int K, std::vector<long double> &x, std::vector<long double> &w) {
  const int h = K / 2;
  x.resize(h); w.resize(h);
  const long double pi = acosl(-1.0L);
  for (int i = 0; i < h; ++i) {
    long double z = cosl(pi * (i + 0.75L) / (K + 0.5L));
    long double pp = 0.0L;
    for (int it = 0; it < 100; ++it) {
      long double p1 = 1.0L, p2 = 0.0L;
      for (int j = 1; j <= K; ++j) {
        long double p3 = p2;
        p2 = p1;
        p1 = ((2.0L * j - 1.0L) * z * p2 - (j - 1.0L) * p3) / j;
      }
      pp = K * (z * p1 - p2) / (z * z - 1.0L);
      long double dz = p1 / pp;
      z -= dz;
      if (fabsl(dz) < 1e-19L) break;
    }
    // one more evaluation of the derivative at the converged node
    long double p1 = 1.0L, p2 = 0.0L;
    for (int j = 1; j <= K; ++j) {
      long double p3 = p2;
      p2 = p1;
      p1 = ((2.0L * j - 1.0L) * z * p2 - (j - 1.0L) * p3) / j;
    }
    pp = K * (z * p1 - p2) / (z * z - 1.0L);
    x[i] = z;
    w[i] = 2.0L / ((1.0L - z * z) * pp * pp);
  }
}

}  // namespace

}  // namespace cmdr

using namespace cmdr;

extern "C" {

// commander3/src/comm_N_mod.f90:127-197 (`compute_invN_lm`), after its `YtW_scalar` and `mpi_bcast`:
// a_l0[c] points at the lmax+1 m=0 coefficients of YtW(N^-1 map) for component c (host memory, the
// same on every rank); out[c] receives N_lm in the local real-packed alm order of `alm_info` (both
// entries of an m>0 pair get the same value, :176-181), host or device memory.  npix = 12 nside^2.
void cmdr_sht_invn_diag(int nmaps, const double *const *a_l0, double npix, const sharp_alm_info *alm_info,
                        double *const *out, void *stream) {
  if (nmaps < 1 || nmaps > 3) { fprintf(stderr, "cmdr_sht_invn_diag: nmaps %d unsupported (1..3)\n", nmaps); abort(); }
  sharp_alm_info *a = const_cast<sharp_alm_info *>(alm_info);
  if (!a->real_packed) { fprintf(stderr, "cmdr_sht_invn_diag: needs a real-packed alm_info\n"); abort(); }
  cudaStream_t st = (cudaStream_t)stream;
  const int lmax = a->lmax;
  const long long nalm = a->nalm;
  if (nalm == 0 || a->nm == 0) return;
  // quadrature exact for polynomials of degree 3 lmax: K >= (3 lmax + 1) / 2 nodes, K even
  int K = (3 * lmax + 1) / 2 + 1;
  K += K & 1;
  const int h = K / 2;
  std::vector<long double> gx, gw;
  gauss_legendre_half(K, gx, gw);
  // folded profile: f_c(x_k) = npix/2 * w_k * (nbar_c(x_k) + nbar_c(-x_k)) = npix * w_k * sum_{L even} a_L0 lambda_L0(x_k)
  std::vector<double> trig((size_t)h * 4), f((size_t)nmaps * h);
  const long double fourpi = 4.0L * acosl(-1.0L);
  unsigned nt = std::thread::hardware_concurrency();
  if (nt == 0) nt = 4;
  if (nt > 32) nt = 32;
  std::vector<std::thread> th;
  for (unsigned t = 0; t < nt; ++t) {
    th.emplace_back([&, t]() {
      for (int i = (int)t; i < h; i += (int)nt) {
        const long double z = gx[i];
        trig[4 * (size_t)i + 0] = (double)z;
        trig[4 * (size_t)i + 1] = (double)sqrtl((1.0L - z) * (1.0L + z));
        trig[4 * (size_t)i + 2] = (double)sqrtl(0.5L * (1.0L - z));
        trig[4 * (size_t)i + 3] = (double)sqrtl(0.5L * (1.0L + z));
        long double acc[3] = {0.0L, 0.0L, 0.0L};
        long double p0 = 1.0L, p1 = z;       // P_0, P_1
        for (int L = 0; L <= lmax; ++L) {
          long double pl;
          if (L == 0) pl = p0;
          else if (L == 1) pl = p1;
          else {
            pl = ((2.0L * L - 1.0L) * z * p1 - (L - 1.0L) * p0) / L;
            p0 = p1; p1 = pl;
          }
          if ((L & 1) == 0) {
            const long double lam = sqrtl((2.0L * L + 1.0L) / fourpi) * pl;
            for (int c = 0; c < nmaps; ++c) acc[c] += (long double)a_l0[c][L] * lam;
          }
        }
        for (int c = 0; c < nmaps; ++c) f[(size_t)c * h + i] = (double)((long double)npix * gw[i] * acc[c]);
      }
    });
  }
  for (auto &t : th) t.join();

  ensure_alm_device(a);
  LegAlm A = make_legalm(a, Job{}, nullptr, true);   // spin 0, one-step table {A', g}
  double *d_trig = static_cast<double *>(scratch_get("invn_trig", sizeof(double) * trig.size()));
  double *d_f = static_cast<double *>(scratch_get("invn_f", sizeof(double) * f.size()));
  CMDR_CUDA_CHECK(cudaMemcpyAsync(d_trig, trig.data(), sizeof(double) * trig.size(), cudaMemcpyHostToDevice, st));
  CMDR_CUDA_CHECK(cudaMemcpyAsync(d_f, f.data(), sizeof(double) * f.size(), cudaMemcpyHostToDevice, st));
  bool on_dev = true;
  for (int c = 0; c < nmaps; ++c) on_dev = on_dev && is_device_ptr(out[c]);
  InvNParams p;
  p.lmax = lmax; p.nm = a->nm; p.nnodes = h; p.nmaps = nmaps;
  p.mval = A.mval; p.mvstart = A.mvstart; p.cofs = A.cofs; p.coef = A.coef; p.Kstart = A.Kstart;
  p.trig = d_trig; p.f = d_f; p.nalm = nalm;
  double *buf = on_dev ? nullptr : static_cast<double *>(scratch_get("invn_out", sizeof(double) * (size_t)nalm * nmaps));
  for (int c = 0; c < 3; ++c) p.out[c] = nullptr;
  for (int c = 0; c < nmaps; ++c) {
    p.out[c] = on_dev ? out[c] : buf + (size_t)c * nalm;
    CMDR_CUDA_CHECK(cudaMemsetAsync(p.out[c], 0, sizeof(double) * nalm, st));
  }
  constexpr int R = 4;
  dim3 grid((h + 32 * R - 1) / (32 * R), a->nm);
  p.det = nullptr;
  if (deterministic()) {
    // partials of at most 1/16 of the device memory per launch: several launches over m ranges beyond that
    static size_t cap = 0;
    if (!cap) { size_t fr, tot; CMDR_CUDA_CHECK(cudaMemGetInfo(&fr, &tot)); cap = tot / 16; }
    p.dl.nb = (int)grid.x; p.dl.lmax = lmax;
    const size_t per_m = (size_t)grid.x * p.dl.row() * sizeof(double) * nmaps;
    const int mpl = (int)std::max<size_t>(1, std::min<size_t>(cap / per_m, a->nm));
    for (int i0 = 0; i0 < a->nm; i0 += mpl) {
      p.dl.im0 = i0; p.dl.nm = std::min(mpl, a->nm - i0);
      p.det = static_cast<double *>(scratch_get("det_part", sizeof(double) * p.dl.comp_stride() * nmaps));
      const dim3 gi(grid.x, p.dl.nm), gr((lmax + 1 + 255) / 256, p.dl.nm);
      switch (nmaps) {
        case 1: invn_kernel<R, 1, true><<<gi, 32, 0, st>>>(p); invn_reduce_kernel<1><<<gr, 256, 0, st>>>(p); break;
        case 2: invn_kernel<R, 2, true><<<gi, 32, 0, st>>>(p); invn_reduce_kernel<2><<<gr, 256, 0, st>>>(p); break;
        default: invn_kernel<R, 3, true><<<gi, 32, 0, st>>>(p); invn_reduce_kernel<3><<<gr, 256, 0, st>>>(p); break;
      }
      count_launch(2);
    }
  } else {
    switch (nmaps) {
      case 1: invn_kernel<R, 1><<<grid, 32, 0, st>>>(p); break;
      case 2: invn_kernel<R, 2><<<grid, 32, 0, st>>>(p); break;
      default: invn_kernel<R, 3><<<grid, 32, 0, st>>>(p); break;
    }
    count_launch(1);
  }
  CMDR_CUDA_CHECK(cudaGetLastError());
  if (!on_dev)
    for (int c = 0; c < nmaps; ++c)
      CMDR_CUDA_CHECK(cudaMemcpyAsync(out[c], p.out[c], sizeof(double) * nalm, cudaMemcpyDeviceToHost, st));
  // the host staging vectors (trig, f) go out of scope on return
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

}  // extern "C"
