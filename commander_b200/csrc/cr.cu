// cr.cu -- the constrained-realisation CG of Commander3 behind the C ABI, device resident.
//
// Replaces, for one diffuse signal component with a diagonal prior seen through nbands bands that share one
// comm_mapinfo (the CMB amplitude solve of BASELINE.json configs[2]):
//   cr_matmulA            commander3/src/comm_cr_mod.f90:771-1024   A = P + sqrt(S) sum_nu F B^t Y^t N^-1 Y B F sqrt(S)
//   cr_computeRHS         commander3/src/comm_cr_mod.f90:542-769    b = sqrt(S) sum_nu F B^t Y^t (N^-1 d + N^-1/2 eta_nu) + eta_0
//   cr_invM (diagonal)    commander3/src/comm_cr_mod.f90:1026-1077, comm_diffuse_comp_mod.f90:2186-2235 (npre = 1),
//                         with N^-1_{lm,lm} from compute_invN_lm, commander3/src/comm_N_mod.f90:127-197
//   solve_cr_eqn_by_CG    commander3/src/comm_cr_mod.f90:201-348    same update order and convergence test
//   mpi_dot_product       commander3/src/comm_utils.f90:599-614     device reduction + 8-byte NCCL all-reduce
//
// What the reference does with ~10 host passes over the vectors and a PCIe round trip per sharp_execute runs
// here without a single element-wise pass over a_lm or the map outside the transform kernels:
//   * sqrt(S) (comm_Cl_mod.f90:588-637), the beam b_l (comm_B_bl_mod.f90:108-127) and F_mean
//     (comm_diffuse_comp_mod.f90:2077-2080) are one factor per (band, component, l) that the Legendre kernels apply
//     when they load the a_lm (synthesis) and when they store them (analysis);
//   * N^-1 (comm_N_rms_mod.f90:264-273: siN^2 x mask per pixel) is applied by the ring-FFT epilogue as it writes
//     the map;
//   * "+ x" and the sum over bands are the accumulate mode of the analysis kernels (y starts as P x);
//   * r, d, q, x stay on the device, the scalars alpha and beta are computed on the device from the reduced
//     dot products, and with the shipped criterion `fixed_iter` (parameter_files/param_BP8.1_v1.txt:40-47) the host
//     never waits for the GPU inside the loop.
#include <cmath>
#include <cstring>
#include <vector>

#include "kernels.h"

using namespace cmdr;

extern "C" void cmdr_sht_allreduce_sum(int comm, double *dev_buf, int n, void *stream);
extern "C" void cmdr_sht_invn_diag(int nmaps, const double *const *a_l0, double npix, const sharp_alm_info *alm_info,
                                   double *const *out, void *stream);

struct cmdr_cr_system {
  int comm = -1, nbands = 0, nmaps = 0, lmax = 0;
  sharp_geom_info *gT = nullptr, *gP = nullptr;
  sharp_alm_info *a = nullptr;
  long long nalm = 0, npix = 0, n = 0;      // n = nmaps * nalm: length of a CG vector
  bool prior = false;
  double *invN = nullptr;      // [nbands][nmaps][npix]
  double *lsc = nullptr;       // [nbands][nmaps][lmax+1]: sqrt(S) b_l (F_mean, mb_eff folded into b_l by the caller)
  double *blF = nullptr;       // [nbands][nmaps][lmax+1]: b_l alone (RHS of a component without prior uses lsc too)
  double *Minv = nullptr;      // [nmaps][nalm] diagonal preconditioner, nullptr = identity
  double *map = nullptr;       // [nmaps][npix] work map
  double *vx = nullptr, *vr = nullptr, *vd = nullptr, *vq = nullptr, *vb = nullptr;   // [nmaps][nalm] each
  double *sc = nullptr;        // device scalars, see S_* below
  double *partial = nullptr;   // per-block partial sums
  double *hist = nullptr;      // delta_new per iteration (device)
  int hist_cap = 0;
  double *h_sc = nullptr;      // pinned host mirror of the scalars
  unsigned long long n_matmul = 0;
  std::vector<double> h_lsc;   // host copy of lsc (preconditioner build)
  std::vector<long long> col;  // a_lm per column of a CG vector: nmaps x nalm, or those of every component (multi)
  cmdr::CrMulti *multi = nullptr;   // several components and bands (cmdr_cr_setup_multi, cr_multi.cu)
  double *vs = nullptr;        // M^-1 r of the block or pseudo-inverse preconditioner (multi)
  CrRing *rings = nullptr;     // local -> global ring table of the drawn fluctuation terms (cr_draw.cu; one-component)
};

namespace {

constexpr int NBLK = 592;      // 148 SMs x 4: grid of the vector kernels (fixed => reproducible partial sums)
constexpr int NTHR = 256;
enum { S_DNEW = 0, S_DOLD, S_DQ, S_ALPHA, S_BETA, S_D0, S_TMP, S_COUNT = 8 };

__device__ __forceinline__ double block_sum(double v) {
  __shared__ double sh[NTHR / 32];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < NTHR / 32) t = sh[threadIdx.x];
  if (threadIdx.x < 32) for (int o = 4; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  __syncthreads();
  return t;   // valid in thread 0
}

// partial[b] = sum over this block's elements of a[i] * b[i] (* w[i] when w != nullptr)
__global__ void __launch_bounds__(NTHR) k_dot(const double *__restrict__ a, const double *__restrict__ b,
                                             const double *__restrict__ w, long long n, double *partial) {
  double acc = 0.0;
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR)
    acc += w ? a[i] * b[i] * w[i] : a[i] * b[i];
  acc = block_sum(acc);
  if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

// sum of the block partials in a fixed order -> sc[S_TMP]
__global__ void __launch_bounds__(NTHR) k_finish(const double *partial, int nblk, double *sc) {
  double acc = 0.0;
  for (int i = threadIdx.x; i < nblk; i += NTHR) acc += partial[i];
  acc = block_sum(acc);
  if (threadIdx.x == 0) sc[S_TMP] = acc;
}

// scalar bookkeeping after a reduced dot product landed in sc[S_TMP]
//   what 0: delta_new = tmp (initial r.d)           1: delta0 = tmp
//        2: dq = tmp, alpha = delta_new / dq         3: delta_old = delta_new, delta_new = tmp, beta = new / old; hist[it] = new
__global__ void k_scalar(double *sc, int what, double *hist, int it) {
  const double t = sc[S_TMP];
  if (what == 0) { sc[S_DNEW] = t; if (hist) hist[0] = t; }
  else if (what == 1) sc[S_D0] = t;
  else if (what == 2) { sc[S_DQ] = t; sc[S_ALPHA] = sc[S_DNEW] / t; }
  else { sc[S_DOLD] = sc[S_DNEW]; sc[S_DNEW] = t; sc[S_BETA] = t / sc[S_DOLD]; if (hist) hist[it] = t; }
}

// x += alpha d ; r -= alpha q ; partial = sum r (Minv r)      (solve_cr_eqn_by_CG :254-270 in one pass)
__global__ void __launch_bounds__(NTHR) k_update(double *__restrict__ x, double *__restrict__ r, const double *__restrict__ d,
                                                const double *__restrict__ q, const double *__restrict__ Minv, long long n,
                                                const double *sc, double *partial) {
  const double alpha = sc[S_ALPHA];
  double acc = 0.0;
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR) {
    x[i] = fma(alpha, d[i], x[i]);
    const double ri = fma(-alpha, q[i], r[i]);
    r[i] = ri;
    acc += Minv ? ri * ri * Minv[i] : ri * ri;
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

// d = Minv r + beta d   (first = 1: d = Minv r)
__global__ void __launch_bounds__(NTHR) k_direction(double *__restrict__ d, const double *__restrict__ r,
                                                   const double *__restrict__ Minv, long long n, const double *sc, int first) {
  const double beta = first ? 0.0 : sc[S_BETA];
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR) {
    const double s = Minv ? Minv[i] * r[i] : r[i];
    d[i] = first ? s : fma(beta, d[i], s);
  }
}

// out = a - b
__global__ void __launch_bounds__(NTHR) k_sub(double *__restrict__ out, const double *__restrict__ a, const double *__restrict__ b, long long n) {
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR) out[i] = a[i] - b[i];
}

// z = Minv r
__global__ void __launch_bounds__(NTHR) k_mul(double *__restrict__ z, const double *__restrict__ r, const double *__restrict__ w, long long n) {
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR) z[i] = w ? w[i] * r[i] : r[i];
}

// RHS map of one band: m = invN d (+ sqrt(invN) eta)
__global__ void __launch_bounds__(NTHR) k_rhs_map(double *__restrict__ m, const double *__restrict__ invN, const double *__restrict__ d,
                                                 const double *__restrict__ eta, long long n) {
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR) {
    double v = invN[i] * d[i];
    if (eta) v = fma(sqrt(invN[i]), eta[i], v);
    m[i] = v;
  }
}

// b += eta_alm
__global__ void __launch_bounds__(NTHR) k_add(double *__restrict__ b, const double *__restrict__ e, long long n) {
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR) b[i] += e[i];
}

// Minv[c][i] = 1 / (P + sum_nu lsc_nu[c][l_i]^2 N_lm,nu[c][i]) : accumulate the band terms, then invert
__global__ void __launch_bounds__(NTHR) k_precond_acc(double *__restrict__ acc, const double *__restrict__ nlm, const double *__restrict__ lsc,
                                                     const int *__restrict__ l_of, long long nalm) {
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < nalm; i += (long long)gridDim.x * NTHR) {
    const double f = lsc[l_of[i]];
    acc[i] = fma(f * f, nlm[i], acc[i]);
  }
}
__global__ void __launch_bounds__(NTHR) k_precond_inv(double *__restrict__ acc, double P, long long n) {
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR) {
    const double v = P + acc[i];
    acc[i] = v > 0.0 ? 1.0 / v : 1.0;        // an unconstrained mode without prior passes through (comp2ind == -1)
  }
}

template <typename T>
T *dalloc(size_t n) {
  T *p = nullptr;
  CMDR_CUDA_CHECK(cudaMalloc(&p, sizeof(T) * (n ? n : 1)));
  return p;
}

void cols(double *base, long long stride, int n, double **out) { for (int c = 0; c < n; ++c) out[c] = base + (size_t)c * stride; }

// dot product over ranks into sc[S_TMP], then the scalar step `what`
void reduce_and_step(cmdr_cr_system *s, int what, int it, cudaStream_t st) {
  k_finish<<<1, NTHR, 0, st>>>(s->partial, NBLK, s->sc);
  cmdr_sht_allreduce_sum(s->comm, s->sc + S_TMP, 1, st);
  k_scalar<<<1, 1, 0, st>>>(s->sc, what, s->hist, it);
  count_launch(2);
}

// y = A x on device vectors ([nmaps][nalm] contiguous)
void matmulA_dev(cmdr_cr_system *s, const double *x, double *y, cudaStream_t st) {
  if (s->multi) {
    cr_multi_matmulA(s->multi, x, y, st);
    ++s->n_matmul;
    return;
  }
  if (s->prior) CMDR_CUDA_CHECK(cudaMemcpyAsync(y, x, sizeof(double) * s->n, cudaMemcpyDeviceToDevice, st));   // P = 1
  else CMDR_CUDA_CHECK(cudaMemsetAsync(y, 0, sizeof(double) * s->n, st));
  double *xa[3], *ya[3], *mp[3];
  cols(const_cast<double *>(x), s->nalm, s->nmaps, xa);
  cols(y, s->nalm, s->nmaps, ya);
  cols(s->map, s->npix, s->nmaps, mp);
  for (int b = 0; b < s->nbands; ++b) {
    XformOpts o;
    for (int c = 0; c < s->nmaps; ++c) {
      o.lscale[c] = s->lsc + ((size_t)b * s->nmaps + c) * (s->lmax + 1);
      o.pixscale[c] = s->invN + ((size_t)b * s->nmaps + c) * s->npix;
    }
    // sqrt(S), F, B on load; Y; N^-1 as the map is written          (:797-836, 858-864, 888-892, 905)
    execute_iqu_opts(s->comm, SHARP_Y, s->nmaps, xa, mp, s->gT, s->gP, s->a, SHARP_DP, &o, st);
    // Y^t; B^t, F^t, sqrt(S) on store; accumulated into y over the bands   (:913-918, 926-934, 957-1008)
    XformOpts ot;
    for (int c = 0; c < s->nmaps; ++c) ot.lscale[c] = o.lscale[c];
    execute_iqu_opts(s->comm, SHARP_Yt, s->nmaps, ya, mp, s->gT, s->gP, s->a, SHARP_DP | SHARP_ADD, &ot, st);
  }
  ++s->n_matmul;
}

void copy_in(cmdr_cr_system *s, double *dst, const double *const *src, cudaStream_t st) {
  size_t o = 0;
  for (size_t c = 0; c < s->col.size(); o += s->col[c++])
    if (s->col[c]) CMDR_CUDA_CHECK(cudaMemcpyAsync(dst + o, src[c], sizeof(double) * s->col[c], cudaMemcpyDefault, st));
}
void copy_out(cmdr_cr_system *s, double *const *dst, const double *src, cudaStream_t st) {
  size_t o = 0;
  for (size_t c = 0; c < s->col.size(); o += s->col[c++])
    if (s->col[c]) CMDR_CUDA_CHECK(cudaMemcpyAsync(dst[c], src + o, sizeof(double) * s->col[c], cudaMemcpyDefault, st));
}

// CG vectors, device scalars and their host mirror, for a system of s->n unknowns
void alloc_work(cmdr_cr_system *s, cudaStream_t st) {
  s->vx = dalloc<double>(s->n); s->vr = dalloc<double>(s->n); s->vd = dalloc<double>(s->n);
  s->vq = dalloc<double>(s->n); s->vb = dalloc<double>(s->n);
  s->sc = dalloc<double>(S_COUNT);
  CMDR_CUDA_CHECK(cudaMemsetAsync(s->sc, 0, sizeof(double) * S_COUNT, st));
  s->partial = dalloc<double>(NBLK);
  CMDR_CUDA_CHECK(cudaHostAlloc(&s->h_sc, sizeof(double) * S_COUNT, cudaHostAllocDefault));
}

// the preconditioner step of the CG: z = M^-1 r with the block or pseudo-inverse preconditioner of a multi system
bool block_precond(const cmdr_cr_system *s) { return s->multi && cr_multi_has_precond(s->multi); }

void no_diag_precond(const cmdr_cr_system *s, const char *who) {
  if (!s->multi) return;
  fprintf(stderr, "%s: a system of several components has a block preconditioner, not a diagonal one\n", who);
  abort();
}

}  // namespace

namespace cmdr {

void cr_rhs_map(double *m, const double *invN, const double *d, const double *eta, long long n, cudaStream_t st) {
  k_rhs_map<<<NBLK, NTHR, 0, st>>>(m, invN, d, eta, n);
  count_launch(1);
}

// compute_invN_lm (comm_N_mod.f90:127-197): YtW_scalar of every N^-1 column on geom_info_T (:146), its m = 0
// coefficients to every rank, then the 3j sum (evaluated as a quadrature on the device, invn.cu)
void cr_invn_lm(int comm, int nmaps, double *invN, sharp_geom_info *gT, sharp_geom_info *gP, sharp_alm_info *a, double *nlm,
                cudaStream_t st) {
  const int nl = a->lmax + 1;
  for (int c = 0; c < nmaps; ++c) {
    double *ap[1] = {nlm + (size_t)c * a->nalm};
    double *mp[1] = {invN + (size_t)c * gT->npix};
    execute_iqu_opts(comm, SHARP_YtW, 1, ap, mp, gT, gP, a, SHARP_DP, nullptr, st);
  }
  double *al0_d = dalloc<double>((size_t)nmaps * nl);
  std::vector<double> al0((size_t)nmaps * nl);
  int im0 = -1;
  for (int im = 0; im < a->nm; ++im) if (a->mval[im] == 0) im0 = im;
  CMDR_CUDA_CHECK(cudaMemsetAsync(al0_d, 0, sizeof(double) * nmaps * nl, st));
  if (im0 >= 0)
    for (int c = 0; c < nmaps; ++c)
      CMDR_CUDA_CHECK(cudaMemcpyAsync(al0_d + (size_t)c * nl, nlm + (size_t)c * a->nalm + a->mvstart[im0], sizeof(double) * nl,
                                      cudaMemcpyDeviceToDevice, st));
  cmdr_sht_allreduce_sum(comm, al0_d, nmaps * nl, st);   // the mpi_bcast from the owner of m = 0 (:147-152): zero elsewhere
  CMDR_CUDA_CHECK(cudaMemcpyAsync(al0.data(), al0_d, sizeof(double) * nmaps * nl, cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  const double *ap[3];
  double *op[3];
  for (int c = 0; c < nmaps; ++c) { ap[c] = al0.data() + (size_t)c * nl; op[c] = nlm + (size_t)c * a->nalm; }
  cmdr_sht_invn_diag(nmaps, ap, 12.0 * (double)gT->nside * (double)gT->nside, a, op, st);
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  cudaFree(al0_d);
}

}  // namespace cmdr

extern "C" {

cmdr_cr_system *cmdr_cr_setup(int comm, int nbands, int nmaps, const sharp_geom_info *geom_T, const sharp_geom_info *geom_P,
                              const sharp_alm_info *alm_info, const double *const *invN, const double *const *b_l,
                              const double *const *sqrtS, int precond) {
  if (nmaps != 1 && nmaps != 3) { fprintf(stderr, "cmdr_cr_setup: nmaps %d unsupported (1 or 3)\n", nmaps); abort(); }
  if (nbands < 1) { fprintf(stderr, "cmdr_cr_setup: nbands %d\n", nbands); abort(); }
  cmdr_cr_system *s = new cmdr_cr_system;
  s->nbands = nbands; s->nmaps = nmaps;
  s->gT = const_cast<sharp_geom_info *>(geom_T); s->gP = const_cast<sharp_geom_info *>(geom_P);
  s->a = const_cast<sharp_alm_info *>(alm_info);
  comm = effective_comm(comm, s->gT, s->a, "cmdr_cr_setup");
  s->comm = comm;
  if (!s->a->real_packed) { fprintf(stderr, "cmdr_cr_setup: needs the real-packed a_lm layout of comm_mapinfo\n"); abort(); }
  s->lmax = s->a->lmax; s->nalm = s->a->nalm; s->npix = s->gT->npix; s->n = (long long)nmaps * s->nalm;
  s->prior = sqrtS != nullptr;
  const int nl = s->lmax + 1;
  cudaStream_t st = 0;
  // N^-1 per band / component / pixel
  s->invN = dalloc<double>((size_t)nbands * nmaps * s->npix);
  for (int i = 0; i < nbands * nmaps; ++i)
    if (s->npix) CMDR_CUDA_CHECK(cudaMemcpyAsync(s->invN + (size_t)i * s->npix, invN[i], sizeof(double) * s->npix, cudaMemcpyDefault, st));
  // one factor per (band, component, l): sqrt(S) b_l, zero for the l < 2 polarisation modes
  s->h_lsc.assign((size_t)nbands * nmaps * nl, 0.0);
  for (int b = 0; b < nbands; ++b)
    for (int c = 0; c < nmaps; ++c)
      for (int l = 0; l < nl; ++l) {
        double v = b_l[b * nmaps + c][l] * (sqrtS ? sqrtS[c][l] : 1.0);
        if (c > 0 && l < 2) v = 0.0;
        s->h_lsc[((size_t)b * nmaps + c) * nl + l] = v;
      }
  s->lsc = dalloc<double>(s->h_lsc.size());
  CMDR_CUDA_CHECK(cudaMemcpyAsync(s->lsc, s->h_lsc.data(), sizeof(double) * s->h_lsc.size(), cudaMemcpyHostToDevice, st));
  s->map = dalloc<double>((size_t)nmaps * s->npix);
  s->rings = cr_ring_table_device(s->gT);
  s->col.assign(nmaps, s->nalm);
  alloc_work(s, st);
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  if (precond == 1) {
    // diagonal preconditioner (initDiffPrecond_diagonal / updateDiffPrecond_diagonal for npre = 1,
    // commander3/src/comm_diffuse_comp_mod.f90:1167-1252, 1313-1557): N^-1_{lm,lm} of every band from
    // compute_invN_lm (comm_N_mod.f90:127-197): YtW_scalar of the N^-1 map, its m = 0 coefficients to every rank,
    // then the 3j sum (evaluated as a quadrature on the device, invn.cu)
    s->Minv = dalloc<double>(s->n);
    CMDR_CUDA_CHECK(cudaMemsetAsync(s->Minv, 0, sizeof(double) * s->n, st));
    std::vector<int> l_of(s->nalm);
    {
      long long i = 0;
      for (int im = 0; im < s->a->nm; ++im) {
        const int m = s->a->mval[im];
        for (int l = m; l <= s->lmax; ++l) { l_of[i++] = l; if (m > 0) l_of[i++] = l; }
      }
    }
    int *d_lof = dalloc<int>(s->nalm);
    if (s->nalm) CMDR_CUDA_CHECK(cudaMemcpyAsync(d_lof, l_of.data(), sizeof(int) * s->nalm, cudaMemcpyHostToDevice, st));
    double *nlm = s->vq;                               // [nmaps][nalm] scratch
    for (int b = 0; b < nbands; ++b) {
      cr_invn_lm(comm, nmaps, s->invN + (size_t)b * nmaps * s->npix, s->gT, s->gP, s->a, nlm, st);
      for (int c = 0; c < nmaps; ++c)
        k_precond_acc<<<NBLK, NTHR, 0, st>>>(s->Minv + (size_t)c * s->nalm, nlm + (size_t)c * s->nalm,
                                            s->lsc + ((size_t)b * nmaps + c) * nl, d_lof, s->nalm);
      count_launch(nmaps);
    }
    k_precond_inv<<<NBLK, NTHR, 0, st>>>(s->Minv, s->prior ? 1.0 : 0.0, s->n);
    count_launch(1);
    CMDR_CUDA_CHECK(cudaGetLastError());
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
    cudaFree(d_lof);
  }
  return s;
}

cmdr_cr_system *cmdr_cr_setup_multi(int comm, int ncomp, const sharp_alm_info *const *comp_alm, const int *comp_nmaps,
                                    const double *const *sqrtS, int nbands, const sharp_geom_info *const *band_geom_T,
                                    const sharp_geom_info *const *band_geom_P, const sharp_alm_info *const *band_alm,
                                    const int *band_nmaps, const double *const *invN, const double *const *b_l,
                                    const double *F_mean, int precond) {
  size_t free_b = 0, total_b = 0;
  CMDR_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  const CrPlan plan = plan_cr_multi(ncomp, comp_alm, comp_nmaps, sqrtS, nbands, band_geom_T, band_geom_P, band_alm, band_nmaps,
                                    invN, b_l, F_mean, precond, free_b);
  if (!plan.error.empty()) { fprintf(stderr, "cmdr_sht: cmdr_cr_setup_multi: %s\n", plan.error.c_str()); abort(); }
  int c = comm;
  for (int q = 0; q < nbands; ++q) c = effective_comm(comm, band_geom_T[q], band_alm[q], "cmdr_cr_setup_multi");
  cudaStream_t st = 0;
  cmdr_cr_system *s = new cmdr_cr_system;
  s->comm = c;
  s->nbands = nbands;
  s->multi = cr_multi_create(c, plan, comp_alm, comp_nmaps, sqrtS, band_geom_T, band_geom_P, band_alm, band_nmaps, invN, b_l, F_mean,
                             precond, st);
  cr_multi_columns(s->multi, s->col);
  s->n = cr_multi_length(s->multi);
  alloc_work(s, st);
  if (block_precond(s)) s->vs = dalloc<double>(s->n);
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  return s;
}

// Per-pixel mixing of one (band, component) pair of a cmdr_cr_setup_multi handle, or F_mean again with F = NULL.
void cmdr_cr_set_mixing_map(cmdr_cr_system *s, int band, int comp, const double *const *F, void *stream) {
  if (!s->multi) {
    fprintf(stderr, "cmdr_sht: cmdr_cr_set_mixing_map: %s\n", check_cr_mixing(false, 0, 0, nullptr, nullptr, band, comp, F).c_str());
    abort();
  }
  cr_multi_set_mixing(s->multi, band, comp, F, (cudaStream_t)stream);
}

// Selects (on != 0) the pseudo-inverse preconditioner of a cmdr_cr_setup_multi handle, or the one chosen at setup.
void cmdr_cr_set_pseudoinv(cmdr_cr_system *s, int on, void *stream) {
  if (!s->multi) {
    fprintf(stderr, "cmdr_sht: cmdr_cr_set_pseudoinv: %s\n", check_cr_pseudoinv(false, 0, 0, 0).c_str());
    abort();
  }
  cr_multi_set_pseudoinv(s->multi, on, (cudaStream_t)stream);
  if (block_precond(s) && !s->vs) s->vs = dalloc<double>(s->n);   // a handle built with precond 0
}

void cmdr_cr_destroy(cmdr_cr_system *s) {
  if (!s) return;
  cudaDeviceSynchronize();
  cudaFree(s->invN); cudaFree(s->lsc); cudaFree(s->blF); cudaFree(s->Minv); cudaFree(s->map);
  cudaFree(s->vx); cudaFree(s->vr); cudaFree(s->vd); cudaFree(s->vq); cudaFree(s->vb);
  cudaFree(s->sc); cudaFree(s->partial); cudaFree(s->hist); cudaFree(s->vs); cudaFree(s->rings);
  if (s->h_sc) cudaFreeHost(s->h_sc);
  if (s->multi) cr_multi_destroy(s->multi);
  delete s;
}

// Replaces the caller-visible preconditioner: Minv[c] -> nalm doubles (host or device), or nullptr for the identity.
void cmdr_cr_set_precond_diag(cmdr_cr_system *s, const double *const *Minv) {
  no_diag_precond(s, "cmdr_cr_set_precond_diag");
  if (!Minv) { cudaFree(s->Minv); s->Minv = nullptr; return; }
  if (!s->Minv) s->Minv = dalloc<double>(s->n);
  for (int c = 0; c < s->nmaps; ++c)
    if (s->nalm) CMDR_CUDA_CHECK(cudaMemcpy(s->Minv + (size_t)c * s->nalm, Minv[c], sizeof(double) * s->nalm, cudaMemcpyDefault));
}

// Copies the diagonal preconditioner out (1 / (P + sum_nu S b_l^2 N^-1_lm)); out[c] -> nalm doubles, host or device.
void cmdr_cr_get_precond_diag(const cmdr_cr_system *s, double *const *out) {
  no_diag_precond(s, "cmdr_cr_get_precond_diag");
  for (int c = 0; c < s->nmaps; ++c)
    if (s->nalm) {
      if (s->Minv) CMDR_CUDA_CHECK(cudaMemcpy(out[c], s->Minv + (size_t)c * s->nalm, sizeof(double) * s->nalm, cudaMemcpyDefault));
    }
}

void cmdr_cr_matmulA(cmdr_cr_system *s, const double *const *x, double *const *y, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  copy_in(s, s->vd, x, st);
  matmulA_dev(s, s->vd, s->vq, st);
  copy_out(s, y, s->vq, st);
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

void cmdr_cr_invM(cmdr_cr_system *s, const double *const *r, double *const *z, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  copy_in(s, s->vd, r, st);
  if (block_precond(s)) {
    cr_multi_precond(s->multi, s->vd, s->vq, st);
  } else {
    k_mul<<<NBLK, NTHR, 0, st>>>(s->vq, s->vd, s->Minv, s->n);
    count_launch(1);
  }
  copy_out(s, z, s->vq, st);
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

}  // extern "C"

namespace {

// The drawn eta_0 of every component with a prior into the device CG vector out (zeros elsewhere)
void draw_alm(cmdr_cr_system *s, unsigned long long seed, unsigned long long draw, double *out, cudaStream_t st) {
  if (s->multi) {
    cr_multi_draw_eta(s->multi, seed, draw, nullptr, out, st);
  } else if (s->prior) {
    cr_draw_alm(out, s->nalm, s->a, s->nmaps, seed, draw, 0, st);
  } else {
    CMDR_CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double) * s->n, st));
  }
}

// cr_computeRHS into the caller's b.  data: nbands * nmaps column pointers (nullptr: d = 0, drawn terms only); the pixel
// term from `eta`, the prior term from the caller's eta_alm columns or, with eta.draw, from the stream
void compute_rhs(cmdr_cr_system *s, const double *const *data, const RhsEta &eta, const double *const *eta_alm, double *const *b,
                 cudaStream_t st) {
  const double *alm = nullptr;   // eta_0 as a device CG vector (s->vq), or none
  if (eta.draw) {
    const bool prior = s->multi ? true : s->prior;   // cr_multi_rhs adds it on the components with a prior only
    if ((eta.terms & CMDR_CR_ETA_ALM) && prior) { draw_alm(s, eta.seed, eta.index, s->vq, st); alm = s->vq; }
  } else if (eta_alm) {
    copy_in(s, s->vq, eta_alm, st);
    alm = s->vq;
  }
  if (s->multi) {
    cr_multi_rhs(s->multi, data, eta, alm, s->vb, st);
    copy_out(s, b, s->vb, st);
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
    return;
  }
  CMDR_CUDA_CHECK(cudaMemsetAsync(s->vb, 0, sizeof(double) * s->n, st));
  double *ba[3], *mp[3];
  cols(s->vb, s->nalm, s->nmaps, ba);
  cols(s->map, s->npix, s->nmaps, mp);
  double *tmp = static_cast<double *>(scratch_get("cr_rhs_in", sizeof(double) * (size_t)2 * (s->npix ? s->npix : 1)));
  for (int bnd = 0; bnd < s->nbands; ++bnd) {
    XformOpts o;
    for (int c = 0; c < s->nmaps; ++c) {
      const int i = bnd * s->nmaps + c;
      o.lscale[c] = s->lsc + (size_t)i * (s->lmax + 1);
      cr_rhs_column(mp[c], s->invN + (size_t)i * s->npix, data ? data[i] : nullptr, eta, i, bnd, c, s->npix, s->rings,
                    s->gT->nrings, tmp, st);
    }
    execute_iqu_opts(s->comm, SHARP_Yt, s->nmaps, ba, mp, s->gT, s->gP, s->a, SHARP_DP | SHARP_ADD, &o, st);
  }
  if (alm) {
    k_add<<<NBLK, NTHR, 0, st>>>(s->vb, alm, s->n);
    count_launch(1);
  }
  copy_out(s, b, s->vb, st);
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

// cmdr_cr_compute_rhs_draw's arguments, checked on every rank and compared between them before any of them aborts
void check_draw_call(const cmdr_cr_system *s, unsigned long long seed, unsigned long long draw, int terms, cudaStream_t st) {
  const std::string err = check_cr_draw(terms);
  int w[CR_DRAW_WORDS];
  cr_draw_words(seed, draw, terms, err.empty(), w);
  bool same = true;
  for (int i = 0; i < CR_DRAW_WORDS; ++i) same = comm_all_equal(s->comm, w[i], st) && same;
  if (!err.empty()) { fprintf(stderr, "cmdr_sht: cmdr_cr_compute_rhs_draw: %s\n", err.c_str()); abort(); }
  if (!same) {
    fprintf(stderr, "cmdr_sht: cmdr_cr_compute_rhs_draw: the ranks passed different (seed, draw, terms) or one of them an "
                    "invalid argument; every rank of the communicator must make the same call\n");
    abort();
  }
}

}  // namespace

extern "C" {

// data / eta_pix: nbands * nmaps column pointers (n_pix each; eta_pix may be NULL), eta_alm: nmaps pointers or NULL
void cmdr_cr_compute_rhs(cmdr_cr_system *s, const double *const *data, const double *const *eta_pix,
                         const double *const *eta_alm, double *const *b, void *stream) {
  RhsEta eta;
  eta.pix = eta_pix;
  compute_rhs(s, data, eta, eta_alm, b, (cudaStream_t)stream);
}

void cmdr_cr_compute_rhs_draw(cmdr_cr_system *s, const double *const *data, unsigned long long seed, unsigned long long draw,
                              int terms, double *const *b, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  check_draw_call(s, seed, draw, terms, st);
  RhsEta eta;
  eta.draw = true;
  eta.seed = seed;
  eta.index = draw;
  eta.terms = terms;
  compute_rhs(s, data, eta, nullptr, b, st);
}

void cmdr_cr_draw_eta(cmdr_cr_system *s, unsigned long long seed, unsigned long long draw, double *const *eta_pix,
                      double *const *eta_alm, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (s->multi) {
    cr_multi_draw_eta(s->multi, seed, draw, eta_pix, nullptr, st);
  } else if (eta_pix) {
    for (int bnd = 0; bnd < s->nbands; ++bnd)
      for (int c = 0; c < s->nmaps; ++c)
        cr_draw_pix(eta_pix[bnd * s->nmaps + c], s->rings, s->gT->nrings, s->npix, seed, draw, bnd, c, st);
  }
  if (eta_alm) {
    draw_alm(s, seed, draw, s->vq, st);
    copy_out(s, eta_alm, s->vq, st);
  }
  CMDR_CUDA_CHECK(cudaGetLastError());
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

// solve_cr_eqn_by_CG.  b, x: nmaps column pointers (host or device); x holds the initial guess when x0_given != 0
// and receives the solution.  conv_crit: 0 = 'residual', 1 = 'fixed_iter'.  hist (optional, host, maxiter + 1 doubles):
// r^t M^-1 r before the first iteration and after every iteration.  Returns the number of iterations done.
int cmdr_cr_solve(cmdr_cr_system *s, const double *const *b, double *const *x, int x0_given, int maxiter, double cg_tol,
                  int conv_crit, int cg_miniter, int cg_check_conv_freq, double *hist, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (conv_crit != 0 && conv_crit != 1) { fprintf(stderr, "cmdr_cr_solve: Unsupported convergence criterion = %d\n", conv_crit); abort(); }
  if (cg_check_conv_freq < 1) cg_check_conv_freq = 1;
  if (s->hist_cap < maxiter + 1) { cudaFree(s->hist); s->hist = dalloc<double>(maxiter + 1); s->hist_cap = maxiter + 1; }
  CMDR_CUDA_CHECK(cudaMemsetAsync(s->hist, 0, sizeof(double) * (maxiter + 1), st));
  copy_in(s, s->vb, b, st);
  if (x0_given) {
    copy_in(s, s->vx, x, st);
    matmulA_dev(s, s->vx, s->vq, st);                                          // r = b - A x            (:200)
    k_sub<<<NBLK, NTHR, 0, st>>>(s->vr, s->vb, s->vq, s->n);
  } else {
    CMDR_CUDA_CHECK(cudaMemsetAsync(s->vx, 0, sizeof(double) * s->n, st));     // "x is zero": A x = 0, r = b
    CMDR_CUDA_CHECK(cudaMemcpyAsync(s->vr, s->vb, sizeof(double) * s->n, cudaMemcpyDeviceToDevice, st));
    ++s->n_matmul;
  }
  // the block and pseudo-inverse preconditioners are one more step (z = M^-1 r into s->vs) before the dot products that
  // the diagonal one fuses into k_update / k_direction / k_dot
  const bool block = block_precond(s);
  if (block) cr_multi_precond(s->multi, s->vr, s->vd, st);                     // d = invM r           (:202)
  else k_direction<<<NBLK, NTHR, 0, st>>>(s->vd, s->vr, s->Minv, s->n, s->sc, 1);
  k_dot<<<NBLK, NTHR, 0, st>>>(s->vr, s->vd, nullptr, s->n, s->partial);       // delta_new = r.d      (:205)
  reduce_and_step(s, 0, 0, st);
  if (block) {                                                                 // delta0 = b.invM b    (:207)
    cr_multi_precond(s->multi, s->vb, s->vs, st);
    k_dot<<<NBLK, NTHR, 0, st>>>(s->vb, s->vs, nullptr, s->n, s->partial);
  } else {
    k_dot<<<NBLK, NTHR, 0, st>>>(s->vb, s->vb, s->Minv, s->n, s->partial);
  }
  reduce_and_step(s, 1, 0, st);
  count_launch(4);
  CMDR_CUDA_CHECK(cudaMemcpyAsync(s->h_sc, s->sc, sizeof(double) * S_COUNT, cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  const double delta0 = s->h_sc[S_D0];
  double delta_new = s->h_sc[S_DNEW];
  if (delta0 > 1e30) fprintf(stderr, "CR warning: Large initial residual = %g\n", delta0);
  const double lim_convergence = cg_tol * delta0;                              // :219-221
  double val_convergence = 1e2 * lim_convergence;
  int it = 0;
  for (int i = 1; i <= maxiter; ++i) {
    if (i % cg_check_conv_freq == 0) {                                         // :234-246
      if (conv_crit == 0 && i > 1) {       // 'residual' needs delta_new on the host; 'fixed_iter' never exits early
        CMDR_CUDA_CHECK(cudaMemcpyAsync(s->h_sc, s->sc, sizeof(double) * S_COUNT, cudaMemcpyDeviceToHost, st));
        CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
        delta_new = s->h_sc[S_DNEW];
      }
      val_convergence = delta_new;
      if (conv_crit == 0 && val_convergence < lim_convergence && (i >= cg_miniter || delta_new <= 1e-30 * delta0)) break;
    }
    matmulA_dev(s, s->vd, s->vq, st);                                          // q = A d              (:252)
    k_dot<<<NBLK, NTHR, 0, st>>>(s->vd, s->vq, nullptr, s->n, s->partial);     // alpha = delta_new / d.q  (:253)
    reduce_and_step(s, 2, i, st);
    k_update<<<NBLK, NTHR, 0, st>>>(s->vx, s->vr, s->vd, s->vq, s->Minv, s->n, s->sc, s->partial);   // :254-270
    if (block) {
      cr_multi_precond(s->multi, s->vr, s->vs, st);
      k_dot<<<NBLK, NTHR, 0, st>>>(s->vr, s->vs, nullptr, s->n, s->partial);
      count_launch(1);
    }
    reduce_and_step(s, 3, i, st);
    k_direction<<<NBLK, NTHR, 0, st>>>(s->vd, block ? s->vs : s->vr, s->Minv, s->n, s->sc, 0);   // d = s + beta d (:272)
    count_launch(3);
    it = i;
  }
  (void)val_convergence;
  copy_out(s, x, s->vx, st);
  if (hist) CMDR_CUDA_CHECK(cudaMemcpyAsync(hist, s->hist, sizeof(double) * (maxiter + 1), cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaGetLastError());
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  return it;
}

unsigned long long cmdr_cr_matmul_count(const cmdr_cr_system *s) { return s->n_matmul; }

}  // extern "C"
