// cr_multi.cu -- the constrained-realisation operator of several diffuse components seen through bands of their own
// nside, lmax, beam and noise (cr_matmulA and cr_computeRHS of commander3/src/comm_cr_mod.f90:542-1024 as written), and
// its block-diagonal preconditioner (comm_diffuse_comp_mod.f90:1167-1557, 2186-2235).  The entry point and the CG loop
// are those of cr.cu; this file holds what differs from the one-component system:
//   * band gather: a_q = sum_k F_mean[q][k] b_q sqrt(S_k) x_k on the band's transform layout at
//     L_q = min(lmax_q, max_k lmax_k) -- evalDiffuseBand(alm_out) over the components, then alm_equal (:858-882);
//   * Y with N^-1 fused into the ring-FFT epilogue, then Y^t into the band buffer (:888-918);
//   * component gather: y_k = sum_q (the same factor) a'_q + P x_k, one pass per component over every band buffer
//     (projectDiffuseBand(alm_in), :926-1008), written as a gather per component slot: no atomics, deterministic;
//   * block preconditioner: npre x npre per (map, l, m) slot of info_pre, built from N_lm of every band and applied
//     once per CG iteration;
//   * spatially varying mixing of a (band, component) pair (cmdr_cr_set_mixing_map): evalDiffuseBand's Y, x F, YtW
//     (comm_diffuse_comp_mod.f90:2070-2083) before the band gather, and projectDiffuseBand's (:2142-2151) after the
//     band transform, F fused into the ring-FFT epilogue of the Y, b_l and sqrt(S) into the Legendre load and store;
//   * pseudo-inverse preconditioner (cmdr_cr_set_pseudoinv, applyDiffPrecond_pseudoinv :2237-2380): the band gather
//     with U+ instead of g, WY with N = 1 / N^-1 fused into the ring-FFT epilogue, YtW, the component gather with
//     alpha^2 U+, plus P P^t r on every preconditioner slot (tables from cr_pinv.h).
// Every re-pack is rank-local because all handles list the same m's (cr_plan.h).
#include <cmath>
#include <vector>

#include "cr_block.cuh"
#include "cr_pinv.h"
#include "kernels.h"

extern "C" void cmdr_sht_allreduce_sum(int comm, double *dev_buf, int n, void *stream);

namespace cmdr {

namespace {

constexpr int NTHR = 256;

// What the kernels read of the system: layouts (cr_plan.h), component and band descriptors, per-l factors.
struct CrDev {
  int nm = 0, ncomp = 0, nbands = 0, nl = 0;   // nl = lmax_all + 1: stride of the per-l tables
  const int *mval = nullptr;
  const long long *bstart = nullptr;           // [layout][im]
  const long long *off = nullptr, *cnalm = nullptr;   // per component: offset in a CG vector, a_lm per map
  const int *cnm = nullptr, *clmax = nullptr;
  double *const *buf = nullptr;                // per band: a_lm at L_q, [nmaps_q][nalm]
  const long long *bnalm = nullptr;
  const int *bnm = nullptr, *L = nullptr;
  const double *g = nullptr;                   // [k][q][j][l]: F_mean b_l sqrt(S), 0 where the pair has no such slot
  int xform0 = 0, pre = 0;                     // layout index of band 0 at L_0, of the preconditioner slots
  double *const *mix = nullptr;                // per pair q * ncomp + k: its mixing buffer, nullptr for F_mean mixing
  const int *mlay = nullptr;                   // per pair: layout of the buffer after the backward mix
  __device__ long long start(int layout, int im) const { return bstart[(size_t)layout * nm + im]; }
  __device__ double fac(const double *tab, int k, int q, int j, int l) const {
    return tab[(((size_t)k * nbands + q) * 3 + j) * nl + l];
  }
};

// The slot of this thread in an m-block launch over a layout of lmax `L`: grid.y = common m index, t = offset in the
// m block, the map index is grid.z.  False outside the layout.
__device__ __forceinline__ bool mslot(const CrDev &D, int L, int &l, int &t) {
  const int m = D.mval[blockIdx.y];
  t = blockIdx.x * NTHR + threadIdx.x;
  if (m > L) return false;
  if (t >= (m == 0 ? L + 1 : 2 * (L + 1 - m))) return false;
  l = m == 0 ? t : m + (t >> 1);
  return true;
}

// a_q[j, slot] = sum_k tab[k][q][j][l] x_k[j, slot_k] (tab: g, or U+ of the pseudo-inverse); with MIX, the mixed pairs
// add their buffer (b_l Y^t W F Y sqrt(S) x_k on the band's transform layout) instead
template <bool MIX>
__global__ void __launch_bounds__(NTHR) k_cr_band_gather(CrDev D, int q, const double *__restrict__ tab, const double *__restrict__ x) {
  int l, t;
  if (!mslot(D, D.L[q], l, t)) return;
  const int j = blockIdx.z, im = blockIdx.y;
  double acc = 0.0;
  for (int k = 0; k < D.ncomp; ++k) {
    if (MIX && D.mix[q * D.ncomp + k]) {          // every l <= L_q: F spreads the component beyond its lmax
      if (j < D.cnm[k]) acc += D.mix[q * D.ncomp + k][(long long)j * D.bnalm[q] + D.start(D.xform0 + q, im) + t];
      continue;
    }
    if (j >= D.cnm[k] || l > D.clmax[k]) continue;
    acc = fma(D.fac(tab, k, q, j, l), x[D.off[k] + (long long)j * D.cnalm[k] + D.start(k, im) + t], acc);
  }
  D.buf[q][(long long)j * D.bnalm[q] + D.start(D.xform0 + q, im) + t] = acc;
}

// y_k[j, slot] = sum_q tab[k][q][j][l] a'_q[j, slot_q] (+ add[slot] when add != nullptr; tab: g, or alpha^2 U+ of the
// pseudo-inverse); with MIX, the mixed pairs add their buffer (sqrt(S) Y^t W F Y b_l a'_q, on layout mlay,
// l <= min(lmax_k, L_q)) instead
template <bool MIX>
__global__ void __launch_bounds__(NTHR) k_cr_comp_gather(CrDev D, int k, const double *__restrict__ tab, const double *__restrict__ add,
                                                        double *__restrict__ y) {
  int l, t;
  if (!mslot(D, D.clmax[k], l, t)) return;
  const int j = blockIdx.z, im = blockIdx.y;
  double acc = 0.0;
  for (int q = 0; q < D.nbands; ++q) {
    if (j >= D.bnm[q] || l > D.L[q]) continue;
    const int ip = q * D.ncomp + k;
    if (MIX && D.mix[ip]) acc += D.mix[ip][(long long)j * D.bnalm[q] + D.start(D.mlay[ip], im) + t];
    else acc = fma(D.fac(tab, k, q, j, l), D.buf[q][(long long)j * D.bnalm[q] + D.start(D.xform0 + q, im) + t], acc);
  }
  const long long i = D.off[k] + (long long)j * D.cnalm[k] + D.start(k, im) + t;
  y[i] = add ? acc + add[i] : acc;
}

// the component-side input of a mixed pair whose component has the larger lmax: x_k truncated at L_q = lmax_q on the
// band's transform layout (the buffer of the pair)
__global__ void __launch_bounds__(NTHR) k_cr_mix_pack(CrDev D, int q, int k, const double *__restrict__ x, double *__restrict__ out) {
  int l, t;
  if (!mslot(D, D.L[q], l, t)) return;
  const int j = blockIdx.z, im = blockIdx.y;
  out[(long long)j * D.bnalm[q] + D.start(D.xform0 + q, im) + t] = x[D.off[k] + (long long)j * D.cnalm[k] + D.start(k, im) + t];
}

// M[j, slot, k1 <= k2] += N_lm b_l^2 F_k1 F_k2 of band q (f = F_mean b_l, zero beyond either lmax)
__global__ void __launch_bounds__(NTHR) k_cr_pre_acc(CrDev D, int q, const double *__restrict__ nlm, long long nalm_band,
                                                    int band_layout, const double *__restrict__ f, double *__restrict__ M,
                                                    long long ntot, long long nalm_pre) {
  int l, t;
  if (!mslot(D, D.L[q], l, t)) return;
  const int j = blockIdx.z, im = blockIdx.y;
  const double w = nlm[(long long)j * nalm_band + D.start(band_layout, im) + t];
  double r[CR_MAX_NPRE];
#pragma unroll
  for (int k = 0; k < CR_MAX_NPRE; ++k) r[k] = k < D.ncomp ? D.fac(f, k, q, j, l) : 0.0;
  double *m = M + (long long)j * nalm_pre + D.start(D.pre, im) + t;
#pragma unroll
  for (int k1 = 0; k1 < CR_MAX_NPRE; ++k1)
#pragma unroll
    for (int k2 = k1; k2 < CR_MAX_NPRE; ++k2)
      if (k2 < D.ncomp && r[k1] != 0.0 && r[k2] != 0.0) m[(long long)cr_tri(k1, k2, D.ncomp) * ntot] += w * r[k1] * r[k2];
}

// sqrt(S) on both sides, the prior, the inversion: one thread per (map, preconditioner slot)
__global__ void __launch_bounds__(NTHR) k_cr_pre_finish(CrDev D, int lmax_pre, const double *__restrict__ sS, unsigned prior,
                                                       double *M, long long ntot, long long nalm_pre) {
  int l, t;
  if (!mslot(D, lmax_pre, l, t)) return;
  const int j = blockIdx.z, im = blockIdx.y;
  double s[CR_MAX_NPRE];
  bool pr[CR_MAX_NPRE];
  for (int k = 0; k < D.ncomp; ++k) {
    pr[k] = (prior >> k) & 1u;
    s[k] = sS[((size_t)k * 3 + j) * D.nl + l];
  }
  cr_block_finish_invert<CR_MAX_NPRE>(M + (long long)j * nalm_pre + D.start(D.pre, im) + t, ntot, D.ncomp, s, pr);
}

// z = M r on every preconditioner slot: gather r from each component (zero where it has no such slot), one block
// product, z back to each component's slot.  A preconditioner slot maps to at most one slot per component, so the
// writes do not conflict.
template <int NMAX>
__global__ void __launch_bounds__(NTHR) k_cr_pre_apply(CrDev D, int lmax_pre, const double *__restrict__ M, long long ntot,
                                                      long long nalm_pre, const double *__restrict__ r, double *__restrict__ z) {
  int l, t;
  if (!mslot(D, lmax_pre, l, t)) return;
  const int j = blockIdx.z, im = blockIdx.y;
  double rv[NMAX], zv[NMAX];
  long long idx[NMAX];
#pragma unroll
  for (int k = 0; k < NMAX; ++k) {
    idx[k] = -1;
    rv[k] = 0.0;
    if (k < D.ncomp && j < D.cnm[k] && l <= D.clmax[k]) {
      idx[k] = D.off[k] + (long long)j * D.cnalm[k] + D.start(k, im) + t;
      rv[k] = r[idx[k]];
    }
  }
  cr_block_apply<NMAX>(M + (long long)j * nalm_pre + D.start(D.pre, im) + t, ntot, D.ncomp, rv, zv);
#pragma unroll
  for (int k = 0; k < NMAX; ++k)
    if (idx[k] >= 0) z[idx[k]] = zv[k];
}

// N = 1 / N^-1 where N^-1 > 0, else 0: the noise covariance N%N of the pseudo-inverse (masked pixels carry no information)
__global__ void __launch_bounds__(NTHR) k_cr_noise_cov(double *__restrict__ N, const double *__restrict__ invN, long long n) {
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR)
    N[i] = invN[i] > 0.0 ? 1.0 / invN[i] : 0.0;
}

// partial[2 b], partial[2 b + 1] = sum of v, sum of v^2 over block b's elements (compute_alpha_nu's sums, first stage)
__global__ void __launch_bounds__(NTHR) k_cr_sum2_partial(const double *__restrict__ v, long long n, double *__restrict__ partial) {
  __shared__ double sh[2][NTHR];
  double s1 = 0.0, s2 = 0.0;
  for (long long i = (long long)blockIdx.x * NTHR + threadIdx.x; i < n; i += (long long)gridDim.x * NTHR) {
    const double t = v[i];
    s1 += t;
    s2 = fma(t, t, s2);
  }
  sh[0][threadIdx.x] = s1; sh[1][threadIdx.x] = s2;
  __syncthreads();
  for (int o = NTHR / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) { sh[0][threadIdx.x] += sh[0][threadIdx.x + o]; sh[1][threadIdx.x] += sh[1][threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { partial[2 * blockIdx.x] = sh[0][0]; partial[2 * blockIdx.x + 1] = sh[1][0]; }
}

// out[0..1] = the block partials summed in a fixed order (second stage)
__global__ void __launch_bounds__(NTHR) k_cr_sum2_finish(const double *__restrict__ partial, int nblk, double *__restrict__ out) {
  __shared__ double sh[2][NTHR];
  double s1 = 0.0, s2 = 0.0;
  for (int b = threadIdx.x; b < nblk; b += NTHR) { s1 += partial[2 * b]; s2 += partial[2 * b + 1]; }
  sh[0][threadIdx.x] = s1; sh[1][threadIdx.x] = s2;
  __syncthreads();
  for (int o = NTHR / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) { sh[0][threadIdx.x] += sh[0][threadIdx.x + o]; sh[1][threadIdx.x] += sh[1][threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { out[0] = sh[0][0]; out[1] = sh[1][0]; }
}

// The prior term of the pseudo-inverse (:2322-2346) on every preconditioner slot: out_k = sum_k2 (P P^t)[k][k2] r_k2
// with P P^t of this slot's (map, l) from PP ([j][l][cr_tri], cr_pinv_tables).  One thread per (map, slot); each
// component slot is written by exactly one thread, and every one of them is written.
template <int NMAX>
__global__ void __launch_bounds__(NTHR) k_cr_pinv_prior(CrDev D, int lmax_pre, const double *__restrict__ PP,
                                                       const double *__restrict__ r, double *__restrict__ out) {
  int l, t;
  if (!mslot(D, lmax_pre, l, t)) return;
  const int j = blockIdx.z, im = blockIdx.y;
  double rv[NMAX], zv[NMAX];
  long long idx[NMAX];
#pragma unroll
  for (int k = 0; k < NMAX; ++k) {
    idx[k] = -1;
    rv[k] = 0.0;
    if (k < D.ncomp && j < D.cnm[k] && l <= D.clmax[k]) {
      idx[k] = D.off[k] + (long long)j * D.cnalm[k] + D.start(k, im) + t;
      rv[k] = r[idx[k]];
    }
  }
  const int ntri = D.ncomp * (D.ncomp + 1) / 2;
  cr_block_apply<NMAX>(PP + ((long long)j * (lmax_pre + 1) + l) * ntri, 1, D.ncomp, rv, zv);
#pragma unroll
  for (int k = 0; k < NMAX; ++k)
    if (idx[k] >= 0) out[idx[k]] = zv[k];
}

template <typename T>
T *dalloc(size_t n) {
  T *p = nullptr;
  CMDR_CUDA_CHECK(cudaMalloc(&p, sizeof(T) * (n ? n : 1)));
  return p;
}

// grid of an m-block launch over a layout of lmax L
dim3 mgrid(int L, int nm, int nmaps) { return dim3((unsigned)((2 * (L + 1) + NTHR - 1) / NTHR), (unsigned)nm, (unsigned)nmaps); }

}  // namespace

struct CrMulti {
  CrPlan p;
  int comm = -1;
  std::vector<int> cnm, bnm;
  std::vector<long long> off;            // per component: offset in a CG vector (ncomp + 1 entries)
  unsigned prior = 0;                    // bit k: component k has a prior
  std::vector<sharp_geom_info *> gT, gP;
  std::vector<sharp_alm_info *> ca;      // per component: its amplitude handle
  std::vector<sharp_alm_info *> xa;      // per band: the transform handle at L_q
  std::vector<bool> own_xa;              // built here (L_q < lmax_q)
  std::vector<long long> npix;
  std::vector<double *> invN, buf;       // per band: [nmaps_q][npix_q], [nmaps_q][nalm at L_q]
  std::vector<CrRing *> rings;           // per band: local -> global ring table of the drawn fluctuation terms (cr_draw.cu)
  double *map = nullptr;                 // [3][max npix]
  CrDev D;
  int *d_mval = nullptr, *d_cnm = nullptr, *d_clmax = nullptr, *d_bnm = nullptr, *d_L = nullptr;
  long long *d_bstart = nullptr, *d_off = nullptr, *d_cnalm = nullptr, *d_bnalm = nullptr;
  double **d_buf = nullptr;
  double *d_g = nullptr;
  double *Mtri = nullptr;                // block table, nullptr without preconditioner
  long long ntot = 0;                    // nmaps_pre * nalm_pre: stride of the triangle elements
  // spatially varying mixing, per pair q * ncomp + k (cmdr_cr_set_mixing_map)
  std::vector<double *> F;               // [nmin][npix_q] on the device, nullptr: F_mean mixing
  std::vector<double *> mix;             // [nmin][nalm at L_q]: the pair's forward, then backward, mix
  int nmixed = 0;
  std::vector<double> h_sS, h_bl;        // [k][j][l] sqrt(S), [q][j][l] b_l: the lscale of the mixing transforms
  std::vector<double> h_g;               // [k][q][j][l] F_mean b_l sqrt(S): what the pseudo-inverse's V is made of
  double *d_sS = nullptr, *d_bl = nullptr;
  double **d_mix = nullptr;
  int *d_mlay = nullptr;
  // pseudo-inverse preconditioner (cmdr_cr_set_pseudoinv), built on first use
  std::vector<sharp_alm_info *> ba;      // per band: its own handle (alpha_nu runs at lmax_q)
  bool pinv = false;                     // selected for invM / solve
  std::vector<double *> Ncov;            // per band: [nmaps_q][npix_q] N = 1 / N^-1 (0 where N^-1 <= 0), empty until built
  double *d_U = nullptr, *d_UA = nullptr;   // [k][q][j][l] U+ and alpha^2 U+
  double *d_PP = nullptr;                // [nmaps_pre][lmax_pre + 1][ncomp (ncomp + 1) / 2] P P^t
  double *pt = nullptr;                  // prior term P P^t r: a CG vector
  int nmin(int q, int k) const { return std::min(bnm[q], cnm[k]); }
  // lmax_k <= lmax_q: the component side of the mix runs on the component's own handle (reads x_k, writes its layout);
  // else on the band's transform handle at L_q = lmax_q, through k_cr_mix_pack
  bool direct(int q, int k) const { return p.lmax[p.comp(k)] <= p.lmax[p.band(q)]; }
};

long long cr_multi_length(const CrMulti *S) { return S->off.back(); }
bool cr_multi_has_precond(const CrMulti *S) { return S->pinv || S->Mtri != nullptr; }
void cr_multi_columns(const CrMulti *S, std::vector<long long> &len) {
  len.clear();
  for (int k = 0; k < S->p.ncomp; ++k) len.insert(len.end(), S->cnm[k], S->p.nalm[S->p.comp(k)]);
}

CrMulti *cr_multi_create(int comm, const CrPlan &plan, const sharp_alm_info *const *comp_alm, const int *comp_nmaps,
                         const double *const *sqrtS,
                         const sharp_geom_info *const *band_geom_T, const sharp_geom_info *const *band_geom_P,
                         const sharp_alm_info *const *band_alm, const int *band_nmaps, const double *const *invN,
                         const double *const *b_l, const double *F_mean, int precond, cudaStream_t st) {
  CrMulti *S = new CrMulti;
  S->p = plan;
  S->comm = comm;
  const CrPlan &p = S->p;
  const int nc = p.ncomp, nb = p.nbands, nl = p.lmax_all + 1, nm = p.nm();
  S->cnm.assign(comp_nmaps, comp_nmaps + nc);
  S->bnm.assign(band_nmaps, band_nmaps + nb);
  S->off.assign(nc + 1, 0);
  for (int k = 0; k < nc; ++k) S->ca.push_back(const_cast<sharp_alm_info *>(comp_alm[k]));
  S->F.assign((size_t)nc * nb, nullptr);
  S->mix.assign((size_t)nc * nb, nullptr);
  std::vector<int> clmax(nc), cofs(nc + 1, 0), bofs(nb + 1, 0);   // first sqrtS / b_l / invN column of each
  std::vector<long long> cnalm(nc);
  for (int k = 0; k < nc; ++k) {
    clmax[k] = p.lmax[p.comp(k)];
    cnalm[k] = p.nalm[p.comp(k)];
    S->off[k + 1] = S->off[k] + S->cnm[k] * cnalm[k];
    cofs[k + 1] = cofs[k] + S->cnm[k];
    if (sqrtS && sqrtS[cofs[k]]) S->prior |= 1u << k;
  }
  for (int q = 0; q < nb; ++q) bofs[q + 1] = bofs[q] + S->bnm[q];
  // per-l factors sqrt(S), F_mean b_l and their product g (cr_pinv.h)
  std::vector<double> sS, f, g;
  cr_factor_tables(nc, nb, nl, S->cnm.data(), clmax.data(), S->bnm.data(), p.L.data(), S->prior, sqrtS, b_l, F_mean, sS, f, g);
  S->h_sS = sS;
  S->h_g = g;
  S->h_bl.assign((size_t)nb * 3 * nl, 0.0);
  for (int q = 0; q < nb; ++q)
    for (int j = 0; j < S->bnm[q]; ++j)
      for (int l = 0; l <= p.L[q]; ++l) S->h_bl[((size_t)q * 3 + j) * nl + l] = b_l[bofs[q] + j][l];
  // bands: handles, N^-1, buffers
  long long maxpix = 0;
  for (int q = 0; q < nb; ++q) {
    S->gT.push_back(const_cast<sharp_geom_info *>(band_geom_T[q]));
    S->gP.push_back(const_cast<sharp_geom_info *>(band_geom_P[q]));
    sharp_alm_info *a = const_cast<sharp_alm_info *>(band_alm[q]);
    S->ba.push_back(a);
    const bool own = p.L[q] < a->lmax;
    if (own) {
      std::vector<int> ms;
      for (int m : a->mval) if (m <= p.L[q]) ms.push_back(m);
      sharp_make_mmajor_real_packed_alm_info(p.L[q], 1, (int)ms.size(), ms.data(), &a);
    }
    S->xa.push_back(a);
    S->own_xa.push_back(own);
    const long long np = S->gT[q]->npix;
    S->npix.push_back(np);
    maxpix = std::max(maxpix, np);
    double *d = dalloc<double>((size_t)S->bnm[q] * np);
    for (int j = 0; j < S->bnm[q]; ++j)
      if (np) CMDR_CUDA_CHECK(cudaMemcpyAsync(d + (size_t)j * np, invN[bofs[q] + j], sizeof(double) * np, cudaMemcpyDefault, st));
    S->invN.push_back(d);
    S->rings.push_back(cr_ring_table_device(S->gT[q]));
    S->buf.push_back(dalloc<double>((size_t)S->bnm[q] * p.nalm[p.xform(q)]));
  }
  S->map = dalloc<double>((size_t)3 * maxpix);
  std::vector<int> bnm(S->bnm), L(p.L);
  std::vector<long long> bnalm(nb);
  for (int q = 0; q < nb; ++q) bnalm[q] = p.nalm[p.xform(q)];
  S->d_mval = upload(p.mval); S->d_bstart = upload(p.bstart);
  S->d_off = upload(S->off); S->d_cnalm = upload(cnalm); S->d_cnm = upload(S->cnm); S->d_clmax = upload(clmax);
  S->d_buf = upload(S->buf); S->d_bnalm = upload(bnalm); S->d_bnm = upload(bnm); S->d_L = upload(L);
  S->d_g = upload(g);
  CrDev &D = S->D;
  D.nm = nm; D.ncomp = nc; D.nbands = nb; D.nl = nl;
  D.mval = S->d_mval; D.bstart = S->d_bstart; D.off = S->d_off; D.cnalm = S->d_cnalm; D.cnm = S->d_cnm; D.clmax = S->d_clmax;
  D.buf = S->d_buf; D.bnalm = S->d_bnalm; D.bnm = S->d_bnm; D.L = S->d_L; D.g = S->d_g;
  D.xform0 = p.xform(0); D.pre = p.pre();
  if (precond == 1) {
    // initDiffPrecond_diagonal / updateDiffPrecond_diagonal (comm_diffuse_comp_mod.f90:1167-1557) for npre = ncomp:
    // N^-1_{lm,lm} of every band on its own layout, accumulated into the blocks, then finished and inverted per slot
    const long long nalm_pre = p.nalm[p.pre()];
    S->ntot = (long long)p.nmaps_pre * nalm_pre;
    S->Mtri = dalloc<double>(p.precond_bytes / sizeof(double));
    CMDR_CUDA_CHECK(cudaMemsetAsync(S->Mtri, 0, p.precond_bytes, st));
    double *d_f = upload(f), *d_sS = upload(sS);
    for (int q = 0; q < nb; ++q) {
      const long long na = p.nalm[p.band(q)];
      double *nlm = dalloc<double>((size_t)S->bnm[q] * na);
      cr_invn_lm(comm, S->bnm[q], S->invN[q], S->gT[q], S->gP[q], const_cast<sharp_alm_info *>(band_alm[q]), nlm, st);
      if (nm) {
        k_cr_pre_acc<<<mgrid(p.L[q], nm, std::min(S->bnm[q], p.nmaps_pre)), NTHR, 0, st>>>(D, q, nlm, na, p.band(q), d_f, S->Mtri,
                                                                                             S->ntot, nalm_pre);
        count_launch(1);
      }
      CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
      cudaFree(nlm);
    }
    if (nm) {
      k_cr_pre_finish<<<mgrid(p.lmax_pre, nm, p.nmaps_pre), NTHR, 0, st>>>(D, p.lmax_pre, d_sS, S->prior, S->Mtri, S->ntot, nalm_pre);
      count_launch(1);
    }
    CMDR_CUDA_CHECK(cudaGetLastError());
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
    cudaFree(d_f); cudaFree(d_sS);
  }
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  return S;
}

void cr_multi_destroy(CrMulti *S) {
  for (size_t q = 0; q < S->xa.size(); ++q) {
    if (S->own_xa[q]) sharp_destroy_alm_info(S->xa[q]);
    cudaFree(S->invN[q]); cudaFree(S->buf[q]); cudaFree(S->rings[q]);
  }
  for (size_t i = 0; i < S->F.size(); ++i) { cudaFree(S->F[i]); cudaFree(S->mix[i]); }
  for (double *n : S->Ncov) cudaFree(n);
  cudaFree(S->d_U); cudaFree(S->d_UA); cudaFree(S->d_PP); cudaFree(S->pt);
  cudaFree(S->d_sS); cudaFree(S->d_bl); cudaFree(S->d_mix); cudaFree(S->d_mlay);
  cudaFree(S->map); cudaFree(S->Mtri);
  cudaFree(S->d_mval); cudaFree(S->d_bstart); cudaFree(S->d_off); cudaFree(S->d_cnalm); cudaFree(S->d_cnm); cudaFree(S->d_clmax);
  cudaFree(S->d_buf); cudaFree(S->d_bnalm); cudaFree(S->d_bnm); cudaFree(S->d_L); cudaFree(S->d_g);
  delete S;
}

namespace {
void band_cols(CrMulti *S, int q, double **alm, double **map) {
  for (int j = 0; j < S->bnm[q]; ++j) {
    alm[j] = S->buf[q] + (size_t)j * S->p.nalm[S->p.xform(q)];
    map[j] = S->map + (size_t)j * S->npix[q];
  }
}

// y_k = sum_q g a'_q (+ add on the components with a prior), every component; with `pinv`, y_k = sum_q alpha^2 U+ a'_q
// + add on every component, F_mean mixing on every pair
void comp_gather(CrMulti *S, const double *add, double *y, cudaStream_t st, bool pinv = false) {
  if (!S->p.nm()) return;
  for (int k = 0; k < S->p.ncomp; ++k) {
    const dim3 grid = mgrid(S->p.lmax[S->p.comp(k)], S->p.nm(), S->cnm[k]);
    const double *a = (pinv || ((S->prior >> k) & 1u)) ? add : nullptr;
    if (pinv) k_cr_comp_gather<false><<<grid, NTHR, 0, st>>>(S->D, k, S->d_UA, a, y);
    else if (S->nmixed) k_cr_comp_gather<true><<<grid, NTHR, 0, st>>>(S->D, k, S->d_g, a, y);
    else k_cr_comp_gather<false><<<grid, NTHR, 0, st>>>(S->D, k, S->d_g, a, y);
    count_launch(1);
  }
}

// The map columns of a mixing transform of band q and its fused factors: F as the map is written, `ls` per l
void mix_opts(CrMulti *S, int q, int k, const double *ls, int nl, double **map, XformOpts &o) {
  const int ip = q * S->p.ncomp + k;
  for (int j = 0; j < S->nmin(q, k); ++j) {
    map[j] = S->map + (size_t)j * S->npix[q];
    o.pixscale[j] = S->F[ip] + (size_t)j * S->npix[q];
    o.lscale[j] = ls + (size_t)j * nl;
  }
}

// evalDiffuseBand's mixing of pair (q, k) (:2070-2083, 2086): mix = b_l Y^t W (F Y (sqrt(S) x_k)) at L_q.  The Y runs at
// min(lmax_k, L_q): its input holds no more.
void mix_forward(CrMulti *S, int q, int k, const double *x, cudaStream_t st) {
  const CrPlan &p = S->p;
  const int ip = q * p.ncomp + k, n = S->nmin(q, k), nl = p.lmax_all + 1;
  const long long na = p.nalm[p.xform(q)];
  double *alm[3], *map[3];
  XformOpts o;
  mix_opts(S, q, k, S->d_sS + (size_t)k * 3 * nl, nl, map, o);
  sharp_alm_info *ac = S->xa[q];
  if (S->direct(q, k)) {
    ac = S->ca[k];
    for (int j = 0; j < n; ++j) alm[j] = const_cast<double *>(x) + S->off[k] + (size_t)j * p.nalm[p.comp(k)];
  } else {
    if (p.nm()) {
      k_cr_mix_pack<<<mgrid(p.L[q], p.nm(), n), NTHR, 0, st>>>(S->D, q, k, x, S->mix[ip]);
      count_launch(1);
    }
    for (int j = 0; j < n; ++j) alm[j] = S->mix[ip] + (size_t)j * na;
  }
  execute_iqu_opts(S->comm, SHARP_Y, n, alm, map, S->gT[q], S->gP[q], ac, SHARP_DP, &o, st);
  XformOpts ob;
  for (int j = 0; j < n; ++j) {
    alm[j] = S->mix[ip] + (size_t)j * na;
    ob.lscale[j] = S->d_bl + ((size_t)q * 3 + j) * nl;
  }
  execute_iqu_opts(S->comm, SHARP_YtW, n, alm, map, S->gT[q], S->gP[q], S->xa[q], SHARP_DP, &ob, st);
}

// Y^t of band q's map into its buffer (:913-918), then projectDiffuseBand's mixing of every mixed pair (:2142-2152):
// mix = sqrt(S) Y^t W (F Y (b_l a'_q)), its Y^t W at min(lmax_k, L_q) on the layout the component gather reads
void band_back(CrMulti *S, int q, double **alm, double **map, cudaStream_t st) {
  execute_iqu_opts(S->comm, SHARP_Yt, S->bnm[q], alm, map, S->gT[q], S->gP[q], S->xa[q], SHARP_DP, nullptr, st);
  if (!S->nmixed) return;
  const CrPlan &p = S->p;
  const int nl = p.lmax_all + 1;
  const long long na = p.nalm[p.xform(q)];
  for (int k = 0; k < p.ncomp; ++k) {
    const int ip = q * p.ncomp + k, n = S->nmin(q, k);
    if (!S->F[ip]) continue;
    double *a[3], *mp[3];
    XformOpts o;
    mix_opts(S, q, k, S->d_bl + (size_t)q * 3 * nl, nl, mp, o);
    for (int j = 0; j < n; ++j) a[j] = S->buf[q] + (size_t)j * na;
    execute_iqu_opts(S->comm, SHARP_Y, n, a, mp, S->gT[q], S->gP[q], S->xa[q], SHARP_DP, &o, st);
    XformOpts os;
    for (int j = 0; j < n; ++j) {
      a[j] = S->mix[ip] + (size_t)j * na;
      os.lscale[j] = S->d_sS + ((size_t)k * 3 + j) * nl;
    }
    execute_iqu_opts(S->comm, SHARP_YtW, n, a, mp, S->gT[q], S->gP[q], S->direct(q, k) ? S->ca[k] : S->xa[q], SHARP_DP, &os, st);
  }
}
}  // namespace

// y = A x on device vectors in the layout of cr_system.extract_comp
void cr_multi_matmulA(CrMulti *S, const double *x, double *y, cudaStream_t st) {
  double *alm[3], *map[3];
  for (int q = 0; q < S->p.nbands; ++q) {
    if (S->nmixed)
      for (int k = 0; k < S->p.ncomp; ++k)
        if (S->F[q * S->p.ncomp + k]) mix_forward(S, q, k, x, st);
    if (S->p.nm()) {
      const dim3 grid = mgrid(S->p.L[q], S->p.nm(), S->bnm[q]);
      if (S->nmixed) k_cr_band_gather<true><<<grid, NTHR, 0, st>>>(S->D, q, S->d_g, x);
      else k_cr_band_gather<false><<<grid, NTHR, 0, st>>>(S->D, q, S->d_g, x);
      count_launch(1);
    }
    band_cols(S, q, alm, map);
    XformOpts o;                                                   // N^-1 as the map is written   (:888-905)
    for (int j = 0; j < S->bnm[q]; ++j) o.pixscale[j] = S->invN[q] + (size_t)j * S->npix[q];
    execute_iqu_opts(S->comm, SHARP_Y, S->bnm[q], alm, map, S->gT[q], S->gP[q], S->xa[q], SHARP_DP, &o, st);
    band_back(S, q, alm, map, st);                                 // :913-918, 2142-2151
  }
  comp_gather(S, x, y, st);                                        // :926-1008, + P x
}

// b = sum_q g Y^t (N^-1 d_q + N^-1/2 eta_q) (+ eta_alm on the components with a prior); eta_q from the caller or drawn
// (RhsEta), data nullptr: d = 0; eta_alm: device vector or nullptr
void cr_multi_rhs(CrMulti *S, const double *const *data, const RhsEta &eta, const double *eta_alm, double *b, cudaStream_t st) {
  double *alm[3], *map[3];
  long long maxpix = 1;
  for (long long np : S->npix) maxpix = std::max(maxpix, np);
  double *tmp = static_cast<double *>(scratch_get("cr_rhs_in", sizeof(double) * (size_t)2 * maxpix));
  int col = 0;
  for (int q = 0; q < S->p.nbands; ++q) {
    band_cols(S, q, alm, map);
    const long long np = S->npix[q];
    for (int j = 0; j < S->bnm[q]; ++j, ++col)
      cr_rhs_column(map[j], S->invN[q] + (size_t)j * np, data ? data[col] : nullptr, eta, col, q, j, np, S->rings[q],
                    S->gT[q]->nrings, tmp, st);
    band_back(S, q, alm, map, st);
  }
  comp_gather(S, eta_alm, b, st);
}

void cr_multi_draw_eta(CrMulti *S, unsigned long long seed, unsigned long long draw, double *const *eta_pix, double *eta_alm,
                       cudaStream_t st) {
  if (eta_pix)
    for (int q = 0, col = 0; q < S->p.nbands; ++q)
      for (int j = 0; j < S->bnm[q]; ++j, ++col)
        cr_draw_pix(eta_pix[col], S->rings[q], S->gT[q]->nrings, S->npix[q], seed, draw, q, j, st);
  if (!eta_alm) return;
  for (int k = 0; k < S->p.ncomp; ++k) {
    double *out = eta_alm + S->off[k];
    const long long na = S->p.nalm[S->p.comp(k)];
    if ((S->prior >> k) & 1u) cr_draw_alm(out, na, S->ca[k], S->cnm[k], seed, draw, k, st);
    else if (na) CMDR_CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double) * S->cnm[k] * na, st));
  }
}

// Installs (F != nullptr) or removes the per-pixel mixing map of pair (band, comp); the arguments are checked
void cr_multi_set_mixing(CrMulti *S, int band, int comp, const double *const *F, cudaStream_t st) {
  const CrPlan &p = S->p;
  const std::string err = check_cr_mixing(true, p.ncomp, p.nbands, S->cnm.data(), S->bnm.data(), band, comp, F);
  // every rank learns whether all passed the same (band, comp, NULL-ness) and all were valid before any of them aborts
  const int code = err.empty() ? (band * p.ncomp + comp) * 2 + (F != nullptr) : -1;
  const bool same = comm_all_equal(S->comm, code, st);
  if (!err.empty()) { fprintf(stderr, "cmdr_sht: cmdr_cr_set_mixing_map: %s\n", err.c_str()); abort(); }
  if (!same) {
    fprintf(stderr, "cmdr_sht: cmdr_cr_set_mixing_map: the ranks passed different (band, comp, F == NULL) or one of them an "
                    "invalid argument; every rank of the communicator must make the same call\n");
    abort();
  }
  const int ip = band * p.ncomp + comp, n = S->nmin(band, comp);
  const long long np = S->npix[band];
  if (!F) {
    if (S->F[ip]) {
      CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
      cudaFree(S->F[ip]); cudaFree(S->mix[ip]);
      S->F[ip] = S->mix[ip] = nullptr;
      --S->nmixed;
    }
  } else {
    if (!S->F[ip]) {
      S->F[ip] = dalloc<double>((size_t)n * np);
      S->mix[ip] = dalloc<double>((size_t)n * p.nalm[p.xform(band)]);
      ++S->nmixed;
    }
    for (int j = 0; j < n; ++j)
      if (np) CMDR_CUDA_CHECK(cudaMemcpyAsync(S->F[ip] + (size_t)j * np, F[j], sizeof(double) * np, cudaMemcpyDefault, st));
  }
  if (!S->d_mix) {
    S->d_sS = upload(S->h_sS);
    S->d_bl = upload(S->h_bl);
    std::vector<int> mlay((size_t)p.ncomp * p.nbands);
    for (int q = 0; q < p.nbands; ++q)
      for (int k = 0; k < p.ncomp; ++k) mlay[(size_t)q * p.ncomp + k] = S->direct(q, k) ? p.comp(k) : p.xform(q);
    S->d_mlay = upload(mlay);
    S->d_mix = dalloc<double *>(S->mix.size());
    S->D.mlay = S->d_mlay;
    S->D.mix = S->d_mix;
  }
  CMDR_CUDA_CHECK(cudaMemcpyAsync(S->d_mix, S->mix.data(), sizeof(double *) * S->mix.size(), cudaMemcpyHostToDevice, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

namespace {
// Builds what the pseudo-inverse needs (initDiffPrecond_pseudoinv, comm_diffuse_comp_mod.f90:1255-1294, 1560-1658):
// N per band, alpha_nu per band and map group, the U+ / alpha^2 U+ / P P^t tables.  Collective (transforms and one
// all-reduce); synchronises the stream.
void pinv_build(CrMulti *S, cudaStream_t st) {
  const CrPlan &p = S->p;
  const int nc = p.ncomp, nb = p.nbands, nl = p.lmax_all + 1;
  constexpr int NBLK = 592;
  double *partial = dalloc<double>(2 * NBLK);
  double *sums = dalloc<double>((size_t)4 * nb);   // [q][T, QU][sum tau, sum tau^2]
  CMDR_CUDA_CHECK(cudaMemsetAsync(sums, 0, sizeof(double) * 4 * nb, st));
  for (int q = 0; q < nb; ++q) {
    const long long np = S->npix[q];
    double *N = dalloc<double>((size_t)S->bnm[q] * np);
    if (np) {
      k_cr_noise_cov<<<NBLK, NTHR, 0, st>>>(N, S->invN[q], (long long)S->bnm[q] * np);
      count_launch(1);
    }
    S->Ncov.push_back(N);
    // compute_alpha_nu (comm_N_rms_mod.f90:218-247): tau = Y Yt (N^-1) on the band's own handle, into the work map
    const long long na = p.nalm[p.band(q)];
    double *alm_d = dalloc<double>((size_t)S->bnm[q] * na);
    double *alm[3], *in[3], *map[3];
    for (int j = 0; j < S->bnm[q]; ++j) {
      alm[j] = alm_d + (size_t)j * na;
      in[j] = S->invN[q] + (size_t)j * np;
      map[j] = S->map + (size_t)j * np;
    }
    execute_iqu_opts(S->comm, SHARP_Yt, S->bnm[q], alm, in, S->gT[q], S->gP[q], S->ba[q], SHARP_DP, nullptr, st);
    execute_iqu_opts(S->comm, SHARP_Y, S->bnm[q], alm, map, S->gT[q], S->gP[q], S->ba[q], SHARP_DP, nullptr, st);
    for (int grp = 0; grp < (S->bnm[q] == 3 ? 2 : 1); ++grp) {   // T alone, Q and U together
      if (!np) continue;
      k_cr_sum2_partial<<<NBLK, NTHR, 0, st>>>(S->map + (size_t)grp * np, (grp ? 2 : 1) * np, partial);
      k_cr_sum2_finish<<<1, NTHR, 0, st>>>(partial, NBLK, sums + 4 * q + 2 * grp);
      count_launch(2);
    }
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
    cudaFree(alm_d);
  }
  cmdr_sht_allreduce_sum(S->comm, sums, 4 * nb, st);
  std::vector<double> h(4 * nb), alpha((size_t)3 * nb, 0.0);
  CMDR_CUDA_CHECK(cudaMemcpyAsync(h.data(), sums, sizeof(double) * 4 * nb, cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  cudaFree(partial); cudaFree(sums);
  for (int q = 0; q < nb; ++q)
    for (int j = 0; j < S->bnm[q]; ++j) {
      const double s1 = h[4 * q + 2 * (j > 0)], s2 = h[4 * q + 2 * (j > 0) + 1];
      alpha[(size_t)q * 3 + j] = s1 > 0.0 ? std::sqrt(s2 / s1) : 0.0;
    }
  std::vector<int> clmax(nc);
  for (int k = 0; k < nc; ++k) clmax[k] = p.lmax[p.comp(k)];
  std::vector<double> U, UA, PP;
  cr_pinv_tables(nc, nb, nl, p.nmaps_pre, p.lmax_pre, S->cnm.data(), clmax.data(), S->prior, S->h_g, alpha.data(), U, UA, PP);
  S->d_U = upload(U);
  S->d_UA = upload(UA);
  S->d_PP = upload(PP);
  S->pt = dalloc<double>(S->off.back());
}

// z = M^-1 r with the pseudo-inverse (applyDiffPrecond_pseudoinv, :2237-2380).  buf[q] and map are scratch here:
// cr_multi_matmulA and cr_multi_rhs rewrite both before they read them.
void pinv_apply(CrMulti *S, const double *r, double *z, cudaStream_t st) {
  const CrPlan &p = S->p;
  if (p.nm()) {                                                    // P P^t r, :2322-2346
    const dim3 grid = mgrid(p.lmax_pre, p.nm(), p.nmaps_pre);
    if (p.ncomp <= 4) k_cr_pinv_prior<4><<<grid, NTHR, 0, st>>>(S->D, p.lmax_pre, S->d_PP, r, S->pt);
    else if (p.ncomp <= 8) k_cr_pinv_prior<8><<<grid, NTHR, 0, st>>>(S->D, p.lmax_pre, S->d_PP, r, S->pt);
    else k_cr_pinv_prior<CR_MAX_NPRE><<<grid, NTHR, 0, st>>>(S->D, p.lmax_pre, S->d_PP, r, S->pt);
    count_launch(1);
  }
  double *alm[3], *map[3];
  for (int q = 0; q < p.nbands; ++q) {
    if (p.nm()) {                                                  // sum over (U+)^t, :2270-2285
      k_cr_band_gather<false><<<mgrid(p.L[q], p.nm(), S->bnm[q]), NTHR, 0, st>>>(S->D, q, S->d_U, r);
      count_launch(1);
    }
    band_cols(S, q, alm, map);
    XformOpts o;                                                   // N%N as the map is written, :2288-2290
    for (int j = 0; j < S->bnm[q]; ++j) o.pixscale[j] = S->Ncov[q] + (size_t)j * S->npix[q];
    execute_iqu_opts(S->comm, SHARP_WY, S->bnm[q], alm, map, S->gT[q], S->gP[q], S->xa[q], SHARP_DP, &o, st);
    execute_iqu_opts(S->comm, SHARP_YtW, S->bnm[q], alm, map, S->gT[q], S->gP[q], S->xa[q], SHARP_DP, nullptr, st);   // :2292
  }
  comp_gather(S, S->pt, z, st, true);                              // alpha^2, sum over U+, :2293-2315
}
}  // namespace

// Selects (on) or deselects the pseudo-inverse preconditioner; the tables are built on the first selection
void cr_multi_set_pseudoinv(CrMulti *S, int on, cudaStream_t st) {
  const CrPlan &p = S->p;
  size_t need = 0;
  if (on && S->Ncov.empty() && p.ncomp <= CR_MAX_NPRE) {
    const size_t ntab = (size_t)p.ncomp * p.nbands * 3 * (p.lmax_all + 1);
    size_t pix = 0, alm = 0;
    for (int q = 0; q < p.nbands; ++q) {
      pix += (size_t)S->bnm[q] * S->npix[q];
      alm = std::max(alm, (size_t)S->bnm[q] * (size_t)p.nalm[p.band(q)]);
    }
    need = sizeof(double) * (2 * ntab + (size_t)p.nmaps_pre * (p.lmax_pre + 1) * (p.ncomp * (p.ncomp + 1) / 2) + pix + alm +
                             (size_t)S->off.back());
  }
  size_t free_b = 0, total_b = 0;
  CMDR_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  const std::string err = check_cr_pseudoinv(true, p.ncomp, need, free_b);
  // every rank learns whether all passed the same `on` and all were valid before any of them aborts
  const bool same = comm_all_equal(S->comm, err.empty() ? (on != 0) : -1, st);
  if (!err.empty()) { fprintf(stderr, "cmdr_sht: cmdr_cr_set_pseudoinv: %s\n", err.c_str()); abort(); }
  if (!same) {
    fprintf(stderr, "cmdr_sht: cmdr_cr_set_pseudoinv: the ranks passed different `on` or one of them was refused; every rank "
                    "of the communicator must make the same call\n");
    abort();
  }
  if (on && S->Ncov.empty()) pinv_build(S, st);
  S->pinv = on != 0;
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

// z = M^-1 r with the selected preconditioner: the pseudo-inverse, or the block diagonal
void cr_multi_precond(CrMulti *S, const double *r, double *z, cudaStream_t st) {
  const CrPlan &p = S->p;
  if (S->pinv) { pinv_apply(S, r, z, st); return; }
  if (!p.nm()) return;
  const dim3 grid = mgrid(p.lmax_pre, p.nm(), p.nmaps_pre);
  const long long nalm_pre = p.nalm[p.pre()];
  if (p.ncomp <= 4) k_cr_pre_apply<4><<<grid, NTHR, 0, st>>>(S->D, p.lmax_pre, S->Mtri, S->ntot, nalm_pre, r, z);
  else if (p.ncomp <= 8) k_cr_pre_apply<8><<<grid, NTHR, 0, st>>>(S->D, p.lmax_pre, S->Mtri, S->ntot, nalm_pre, r, z);
  else k_cr_pre_apply<CR_MAX_NPRE><<<grid, NTHR, 0, st>>>(S->D, p.lmax_pre, S->Mtri, S->ntot, nalm_pre, r, z);
  count_launch(1);
}

}  // namespace cmdr
