// abi.cu -- the C ABI of libcmdr_sht: handle construction, device residency of the
// geometry / alm descriptors, host<->device staging and the single-GPU execute paths.
//
// Drop-in for the libsharp2 entry points bound by commander3/src/sharp.f90:32-105
// (SURVEY.md 8b).  Multi-GPU entry points live in dist.cu.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "kernels.h"
#include "legendre_core.cuh"

namespace cmdr {

void destroy_plans(sharp_geom_info *g);
void forget_layout(const sharp_alm_info *a);
void dist_forget_handle(const void *h);   // dist.cu: drops every cached distributed plan built for this handle

bool phase_ring_major() {
  static const bool ring = !(getenv("CMDR_SHT_PH_LAYOUT") && getenv("CMDR_SHT_PH_LAYOUT")[0] == 'm');
  return ring;
}

static std::atomic<unsigned long long> g_launches{0};
void count_launch(int n) { g_launches += (unsigned long long)n; }

// ---------------------------------------------------------------- scratch arena
struct ScratchBuf { void *ptr = nullptr; size_t bytes = 0; };
static std::map<std::string, ScratchBuf> g_scratch;
static std::mutex g_mu;

void *scratch_get(const char *name, size_t bytes) {
  int dev = 0;
  CMDR_CUDA_CHECK(cudaGetDevice(&dev));
  std::string key = std::string(name) + "@" + std::to_string(dev);
  std::lock_guard<std::mutex> lk(g_mu);
  ScratchBuf &b = g_scratch[key];
  if (b.bytes < bytes) {
    if (b.ptr) { CMDR_CUDA_CHECK(cudaDeviceSynchronize()); CMDR_CUDA_CHECK(cudaFree(b.ptr)); }
    size_t want = bytes + bytes / 16 + 256;
    CMDR_CUDA_CHECK(cudaMalloc(&b.ptr, want));
    b.bytes = want;
  }
  return b.ptr;
}

static void scratch_release() {
  std::lock_guard<std::mutex> lk(g_mu);
  for (auto &kv : g_scratch) if (kv.second.ptr) cudaFree(kv.second.ptr);
  g_scratch.clear();
}

// ---------------------------------------------------------------- device residency
void ensure_alm_device(sharp_alm_info *a) {
  int dev = 0;
  CMDR_CUDA_CHECK(cudaGetDevice(&dev));
  if (a->device == dev) return;
  if (a->device >= 0) { fprintf(stderr, "cmdr_sht: alm_info used on two devices\n"); abort(); }
  a->device = dev;
  a->d_mval = upload(a->mval);
  a->d_mvstart = upload(a->mvstart);
  std::vector<int> m2im(a->mmax + 2, -1);
  for (int i = 0; i < a->nm; ++i) m2im[a->mval[i]] = i;
  a->d_m2im = upload(m2im);
}

static const double *ensure_start_norms(sharp_alm_info *a, int spin) {
  auto it = a->d_K.find(spin);
  if (it != a->d_K.end()) return it->second;
  const int mmax = a->mmax < 0 ? 0 : a->mmax;
  std::vector<double> K0, K2, Ks;
  if (spin == 0 || spin == 2) build_start_norms(mmax, K0, K2);
  else build_start_norms_spin(mmax, spin, Ks);
  double *d = upload(spin == 0 ? K0 : (spin == 2 ? K2 : Ks));
  a->d_K[spin] = d;
  return d;
}

void ensure_coef(sharp_alm_info *a, int spin) {
  CoefDev &c = a->coef[spin];
  if (c.ready) return;
  std::vector<double> tab; std::vector<long long> ofs;
  std::vector<long long> tofs(a->nm + 1, 0);
  if (spin == COEF_KEY_S0X2 || spin == COEF_KEY_S0X2P2) {   // spin 0 in steps of two l: one tile row per step
    const int lmax = spin == COEF_KEY_S0X2 ? a->lmax : a->lmax + 2;
    std::vector<double> mix;
    build_coef_table_x2(lmax, a->mval, tab, mix, ofs);
    c.tab2 = upload(mix);
    for (int i = 0; i < a->nm; ++i) {
      long long n = lmax >= a->mval[i] ? (lmax - a->mval[i]) / 2 + 1 : 0;
      tofs[i + 1] = tofs[i] + ((n + 7) & ~7LL);
    }
  } else {
    build_coef_table(a->lmax, spin, a->mval, tab, ofs);
    for (int i = 0; i < a->nm; ++i) {
      int l0 = a->mval[i] > spin ? a->mval[i] : spin;
      long long n = a->lmax >= l0 ? a->lmax - l0 + 1 : 0;
      tofs[i + 1] = tofs[i] + ((n + 7) & ~7LL);
    }
  }
  c.tab = upload(tab);
  c.ofs = upload(ofs);
  c.tofs = upload(tofs);
  c.trows = tofs[a->nm];
  c.nofs = ofs[a->nm];
  c.ready = true;
}

void ensure_geom_device(sharp_geom_info *g) {
  int dev = 0;
  CMDR_CUDA_CHECK(cudaGetDevice(&dev));
  if (g->device == dev) return;
  if (g->device >= 0) { fprintf(stderr, "cmdr_sht: geom_info used on two devices\n"); abort(); }
  g->device = dev;
  std::vector<double> trig(4 * (size_t)g->npairs);
  for (int p = 0; p < g->npairs; ++p) {
    trig[4 * p] = g->cth[p]; trig[4 * p + 1] = g->sth[p]; trig[4 * p + 2] = g->sh[p]; trig[4 * p + 3] = g->ch[p];
  }
  g->d_trig = upload(trig);
  g->d_wgt = upload(g->wgt);
  g->d_nph = upload(g->nph);
  g->d_shifted = upload(g->shifted);
  g->d_ofsN = upload(g->ofsN);
  g->d_ofsS = upload(g->ofsS);
  std::vector<long long> zbase(g->npairs);
  std::vector<int> zidx(g->npairs), znp(g->npairs), zlen(g->npairs), zblue(g->npairs);
  for (const FftRegion &R : g->regions)
    for (int i = 0; i < R.np; ++i) {
      int p = R.first + i;
      zbase[p] = R.base; zidx[p] = i; znp[p] = R.np; zlen[p] = R.len; zblue[p] = R.bluestein ? 1 : 0;
    }
  g->d_zbase = upload(zbase); g->d_zidx = upload(zidx); g->d_znp = upload(znp);
  g->d_zlen = upload(zlen); g->d_zblue = upload(zblue);
}

// per-ring-pair m cut-off for (lmax, spin)
const int *ensure_mlim(sharp_geom_info *g, int lmax, int spin) {
  long long key = ((long long)lmax << 8) | spin;
  auto it = g->mlim.find(key);
  if (it != g->mlim.end()) return it->second;
  std::vector<int> ml(g->npairs);
  for (int p = 0; p < g->npairs; ++p) ml[p] = mlim_for_ring(lmax, spin, g->sth[p], g->cth[p]);
  int *d = upload(ml);
  g->mlim[key] = d;
  return d;
}

// ---------------------------------------------------------------- geometry construction
void ring_trig_ld(int nside, int north, long double &cth, long double &sth, long double &sh, long double &ch) {
  long double ns = nside;
  long double omc;   // 1 - cos(theta)
  if (north < nside) omc = (long double)north * north / (3.0L * ns * ns);
  else omc = 1.0L - (2.0L * ns - north) * 2.0L / (3.0L * ns);
  cth = 1.0L - omc;
  sth = sqrtl(omc * (2.0L - omc));
  sh = sqrtl(0.5L * omc);
  ch = sqrtl(1.0L - 0.5L * omc);
}

// Bluestein work length of a polar-cap ring with nph points: a power of two >= 2 nph - 1, at
// least 1024 so that the shortest rings share one batched plan instead of a dozen tiny launches
static int blue_len(int nph) { int m = 1024; while (m < 2 * nph - 1) m <<= 1; return m; }


// FFT regions: polar-cap pairs grouped by Bluestein work length, then the belt
static void build_regions(sharp_geom_info *g) {
  const int nside = g->nside;
  g->regions.clear();
  long long base = 0;
  int p = 0;
  while (p < g->npairs && g->north[p] < nside) {
    int M = blue_len(g->nph[p]);
    FftRegion R; R.first = p; R.len = M; R.bluestein = true; R.base = base;
    while (p < g->npairs && g->north[p] < nside && blue_len(g->nph[p]) == M) ++p;
    R.np = p - R.first;
    base += (long long)R.np * R.len;
    g->regions.push_back(R);
  }
  g->vlen_total = base;
  if (p < g->npairs) {
    FftRegion R; R.first = p; R.np = g->npairs - p; R.len = 4 * nside; R.bluestein = false; R.base = base;
    base += (long long)R.np * R.len;
    g->regions.push_back(R);
  }
  g->zlen_total = base;
}

// Sub-geometry over parent pairs [a, b): same pixel offsets, own FFT regions / plans.
sharp_geom_info *make_subgeom(const sharp_geom_info *g, int a, int b) {
  sharp_geom_info *s = new sharp_geom_info;
  s->nside = g->nside; s->nrings = 0; s->npix = g->npix; s->pair0 = a; s->npairs = b - a;
  auto cut = [&](auto &dst, const auto &src) { dst.assign(src.begin() + a, src.begin() + b); };
  cut(s->north, g->north); cut(s->cth, g->cth); cut(s->sth, g->sth); cut(s->sh, g->sh); cut(s->ch, g->ch);
  cut(s->wgt, g->wgt); cut(s->nph, g->nph); cut(s->shifted, g->shifted); cut(s->ofsN, g->ofsN); cut(s->ofsS, g->ofsS);
  build_regions(s);
  return s;
}

// True when the north rows (ascending) and the south rows (descending) of consecutive ring pairs are adjacent in the
// map, so that any range of pairs is two plain memory ranges per component.
bool pairs_contiguous(const sharp_geom_info *g) {
  const int np = g->npairs;
  for (int p = 0; p < np; ++p) {
    if (g->ofsN[p] < 0) return false;
    if (g->ofsS[p] < 0 && p != np - 1) return false;
    if (p + 1 < np && g->ofsN[p + 1] != g->ofsN[p] + g->nph[p]) return false;
    if (p + 1 < np && g->ofsS[p + 1] >= 0 && g->ofsS[p] != g->ofsS[p + 1] + g->nph[p + 1]) return false;
  }
  return np > 0;
}

// Splits the pairs into chunks of roughly equal pixel count whose north rings (ascending) and
// south rings (descending) are each contiguous in the map, so that a chunk is two plain
// memory ranges per component.  Leaves g->subs empty when the ring list does not allow that.
void ensure_subgeoms(sharp_geom_info *g, int nchunks) {
  if (g->subs_built) return;
  g->subs_built = true;
  const int np = g->npairs;
  if (np < 1024 || !pairs_contiguous(g)) return;
  // chunk = a multiple of 512 ring pairs: the Legendre CTAs cover 256 or 512 pair slots, so
  // any other boundary would leave lanes idle in every CTA row of the chunk
  const int unit = nchunks > 8 ? 256 : 512;
  int per = ((np + nchunks - 1) / nchunks + unit - 1) / unit * unit;
  if (per >= np) return;
  for (int a = 0; a < np; a += per) g->subs.push_back(make_subgeom(g, a, std::min(np, a + per)));
}

}  // namespace cmdr

using namespace cmdr;

// =================================================================== ABI part 1
extern "C" {

void sharp_make_general_alm_info(int lmax, int nm, int stride, const int *mval, const ptrdiff_t *mvstart,
                                 int flags, sharp_alm_info **out) {
  if (stride != 1) { fprintf(stderr, "cmdr_sht: alm stride %d unsupported (only 1)\n", stride); abort(); }
  sharp_alm_info *a = new sharp_alm_info;
  a->lmax = lmax; a->nm = nm; a->stride = stride; a->flags = flags;
  a->real_packed = (flags & SHARP_REAL_HARMONICS) != 0;
  a->mval.assign(mval, mval + nm);
  a->mvstart.resize(nm);
  long long cnt = 0;
  for (int i = 0; i < nm; ++i) {
    a->mvstart[i] = (long long)mvstart[i];
    int m = mval[i];
    if (m < 0 || m > lmax) { fprintf(stderr, "cmdr_sht: bad m=%d\n", m); abort(); }
    cnt += (long long)(lmax + 1 - m) * ((a->real_packed && m > 0) ? 2 : 1);
    if (m > a->mmax) a->mmax = m;
  }
  a->nalm = cnt;
  *out = a;
}

void sharp_make_mmajor_real_packed_alm_info(int lmax, int stride, int nm, const int *ms, sharp_alm_info **out) {
  if (stride != 1) { fprintf(stderr, "cmdr_sht: alm stride %d unsupported (only 1)\n", stride); abort(); }
  std::vector<int> mval(nm);
  std::vector<ptrdiff_t> mvstart(nm);
  long long idx = 0;
  for (int i = 0; i < nm; ++i) {
    int m = ms ? ms[i] : i;
    int f = m == 0 ? 1 : 2;
    mval[i] = m;
    mvstart[i] = (ptrdiff_t)(idx - (long long)f * m);
    idx += (long long)f * (lmax + 1 - m);
  }
  sharp_make_general_alm_info(lmax, nm, 1, mval.data(), mvstart.data(), SHARP_PACKED | SHARP_REAL_HARMONICS, out);
}

ptrdiff_t sharp_alm_count(const sharp_alm_info *self) { return (ptrdiff_t)self->nalm; }

void sharp_destroy_alm_info(sharp_alm_info *a) {
  if (!a) return;
  dist_forget_handle(a);
  seed_forget(a);
  if (a->device >= 0) {
    forget_layout(a);
    cudaFree(a->d_mval); cudaFree(a->d_mvstart); cudaFree(a->d_m2im);
    for (auto &kv : a->d_K) cudaFree(kv.second);
    for (auto &kv : a->coef) if (kv.second.ready) { cudaFree(kv.second.tab); cudaFree(kv.second.tab2); cudaFree(kv.second.ofs); cudaFree(kv.second.tofs); }
  }
  delete a;
}

void sharp_make_subset_healpix_geom_info(int nside, int stride, int nrings, const int *rings,
                                         const double *weight, sharp_geom_info **out) {
  if (stride != 1) { fprintf(stderr, "cmdr_sht: map stride %d unsupported (only 1)\n", stride); abort(); }
  sharp_geom_info *g = new sharp_geom_info;
  g->nside = nside; g->nrings = nrings;
  const int nn = 2 * nside;
  std::vector<long long> oN(nn + 1, -1), oS(nn + 1, -1);
  long long ofs = 0;
  g->ring.resize(nrings);
  for (int i = 0; i < nrings; ++i) {
    int ring = rings ? rings[i] : i + 1;
    if (ring < 1 || ring > 4 * nside - 1) { fprintf(stderr, "cmdr_sht: bad ring %d\n", ring); abort(); }
    g->ring[i] = ring;
    int north = ring > nn ? 4 * nside - ring : ring;
    int nph = north < nside ? 4 * north : 4 * nside;
    if (ring == north) oN[north] = ofs; else oS[north] = ofs;
    ofs += nph;
  }
  g->npix = ofs;
  const double pixarea_w = 4.0 * M_PI / (12.0 * (double)nside * (double)nside);
  for (int i = 1; i <= nn; ++i) {
    if (oN[i] < 0 && oS[i] < 0) continue;
    long double c, s, sh, ch;
    ring_trig_ld(nside, i, c, s, sh, ch);
    g->north.push_back(i);
    g->cth.push_back((double)c); g->sth.push_back((double)s); g->sh.push_back((double)sh); g->ch.push_back((double)ch);
    g->nph.push_back(i < nside ? 4 * i : 4 * nside);
    g->shifted.push_back(i < nside ? 1 : (((i - nside) & 1) ? 0 : 1));
    g->wgt.push_back(pixarea_w * (weight ? weight[i - 1] : 1.0));
    g->ofsN.push_back(oN[i]); g->ofsS.push_back(oS[i]);
  }
  g->npairs = (int)g->north.size();
  build_regions(g);
  *out = g;
}

void sharp_destroy_geom_info(sharp_geom_info *g) {
  if (!g) return;
  dist_forget_handle(g);
  seed_forget(g);
  for (sharp_geom_info *sub : g->subs) sharp_destroy_geom_info(sub);
  g->subs.clear();
  if (g->device >= 0) {
    destroy_plans(g);
    cudaFree(g->d_trig); cudaFree(g->d_wgt); cudaFree(g->d_nph); cudaFree(g->d_shifted);
    cudaFree(g->d_ofsN); cudaFree(g->d_ofsS); cudaFree(g->d_zbase); cudaFree(g->d_zidx);
    cudaFree(g->d_znp); cudaFree(g->d_zlen); cudaFree(g->d_zblue);
    if (g->d_vtab) cudaFree(g->d_vtab);
    if (g->d_vtab_br) cudaFree(g->d_vtab_br);
    for (auto &kv : g->d_vsub) cudaFree(kv.second);
    for (auto &kv : g->mlim) cudaFree(kv.second);
  }
  delete g;
}

ptrdiff_t sharp_map_size(const sharp_geom_info *g) { return (ptrdiff_t)g->npix; }

}  // extern "C"

// =================================================================== execution
namespace cmdr {

thread_local int g_profiling = 0;
static thread_local std::vector<double> g_prof;   // triples {spin, dir, ms}
struct ProfEv { cudaEvent_t a, b; int spin, dir; };
static thread_local std::vector<ProfEv> g_prof_pending;

void prof_begin(int spin, int dir, cudaStream_t st) {
  if (!g_profiling) return;
  ProfEv e; e.spin = spin; e.dir = dir;
  CMDR_CUDA_CHECK(cudaEventCreate(&e.a)); CMDR_CUDA_CHECK(cudaEventCreate(&e.b));
  CMDR_CUDA_CHECK(cudaEventRecord(e.a, st));
  g_prof_pending.push_back(e);
}
void prof_end(cudaStream_t st) {
  if (!g_profiling) return;
  CMDR_CUDA_CHECK(cudaEventRecord(g_prof_pending.back().b, st));
}
void prof_collect() {
  for (auto &e : g_prof_pending) {
    CMDR_CUDA_CHECK(cudaEventSynchronize(e.b));
    float ms = 0;
    CMDR_CUDA_CHECK(cudaEventElapsedTime(&ms, e.a, e.b));
    g_prof.push_back(e.spin); g_prof.push_back(e.dir); g_prof.push_back(ms);
    cudaEventDestroy(e.a); cudaEventDestroy(e.b);
  }
  g_prof_pending.clear();
}

bool is_device_ptr(const void *p) {
  if (!p) return true;
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// Identity (single-rank) phase layout tables, cached per alm_info on the device.
struct IdLayout { int *m2src = nullptr; int *zeros = nullptr; int *iota = nullptr; };
static std::map<const sharp_alm_info *, IdLayout> g_idlayout;

PhaseLayout single_layout(sharp_alm_info *a, int npairs, int ncomp_tot, int comp0) {
  IdLayout &I = g_idlayout[a];
  if (!I.zeros) {
    std::vector<int> m2src(a->mmax + 2, -1), z(a->nm + 1, 0), io(a->nm + 1);
    for (int i = 0; i < a->nm; ++i) m2src[a->mval[i]] = 0;
    for (int i = 0; i <= a->nm; ++i) io[i] = i;
    I.m2src = upload(m2src); I.zeros = upload(z); I.iota = upload(io);
  }
  PhaseLayout L;
  L.NPL = npairs; L.NML = a->nm; L.ncomp_tot = ncomp_tot; L.comp0 = comp0;
  L.mmax = a->mmax; L.m2src = I.m2src; L.m2im = a->d_m2im;
  L.nm_total = a->nm; L.mlist = a->d_mval; L.mlist_src = I.zeros; L.mlist_im = I.iota;
  return L;
}

void forget_layout(const sharp_alm_info *a) {
  auto it = g_idlayout.find(a);
  if (it == g_idlayout.end()) return;
  cudaFree(it->second.m2src); cudaFree(it->second.zeros); cudaFree(it->second.iota);
  g_idlayout.erase(it);
}

LegAlm make_legalm(sharp_alm_info *a, const Job &job, const double *const *lscale, bool classic) {
  const int spin = job.spin;
  ensure_alm_device(a);
  const int key = (spin == 0 && !classic) ? COEF_KEY_S0X2 : spin;
  ensure_coef(a, key);
  LegAlm A;
  A.lmax = a->lmax; A.nm = a->nm; A.real_packed = a->real_packed ? 1 : 0;
  A.mval = a->d_mval; A.mvstart = a->d_mvstart;
  A.spin = spin;
  A.coef = a->coef[key].tab; A.coef2 = a->coef[key].tab2; A.cofs = a->coef[key].ofs;
  A.Kstart = ensure_start_norms(a, spin);
  A.tofs = a->coef[key].tofs; A.trows = a->coef[key].trows;
  static const bool front_on = !(getenv("CMDR_SHT_FRONT") && atoi(getenv("CMDR_SHT_FRONT")) == 0);
  if (spin == 2 && front_on) {   // scalar front phase of the spin-2 kernels (legendre.cu, spin2_front_phase)
    ensure_coef(a, COEF_KEY_S0X2);
    A.front_coef = a->coef[COEF_KEY_S0X2].tab; A.front_mix = a->coef[COEF_KEY_S0X2].tab2; A.front_cofs = a->coef[COEF_KEY_S0X2].ofs;
    A.front_K0 = ensure_start_norms(a, 0);
  }
  A.deriv1 = job.deriv1;
  if (lscale)
    for (int c = 0; c < job.alm_cols; ++c) A.lscale[c] = lscale[c];
  return A;
}

__global__ void __launch_bounds__(256) add_into_kernel(double *__restrict__ a, const double *__restrict__ r, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) a[i] = a[i] + r[i];
}

double *const *det_add_begin(bool add, double *const *alm, int ncols, size_t nd, cudaStream_t st) {
  if (!add || !deterministic() || nd == 0) return alm;
  static thread_local double *cols[4];
  double *buf = static_cast<double *>(scratch_get("det_add", sizeof(double) * nd * ncols));
  CMDR_CUDA_CHECK(cudaMemsetAsync(buf, 0, sizeof(double) * nd * ncols, st));
  for (int c = 0; c < ncols; ++c) cols[c] = buf + (size_t)c * nd;
  return cols;
}
void det_add_end(double *const *out, double *const *alm, int ncols, size_t nd, cudaStream_t st) {
  if (out == alm) return;
  for (int c = 0; c < ncols; ++c) {
    add_into_kernel<<<(unsigned)std::min<size_t>((nd + 255) / 256, 148 * 8), 256, 0, st>>>(alm[c], out[c], (long long)nd);
    count_launch();
  }
  CMDR_CUDA_CHECK(cudaGetLastError());
}

// Single-GPU transform with device pointers.  `ph` holds ncomp_tot components; this call
// handles components [comp0, comp0+ncomp) of it.
void run_single(const Job &job, double *const *alm, double *const *map, sharp_geom_info *g, sharp_alm_info *a,
                cudaStream_t st, const XformOpts *opts, int comp_off) {
  const int spin = job.spin;
  const int ncomp = job.map_cols;   // map columns and phase components (the a_lm side of a synthesis reads what it needs)
  const bool synth = job.synth;
  ensure_geom_device(g);
  LegAlm A = make_legalm(a, job, opts ? opts->lscale + comp_off : nullptr);
  const double *pixscale[2] = {nullptr, nullptr};
  if (opts)
    for (int c = 0; c < ncomp; ++c) pixscale[c] = opts->pixscale[comp_off + c];
  if (g->npairs == 0 || a->nm == 0) {
    if (!job.add) {
      if (synth) { for (int c = 0; c < ncomp; ++c) if (g->npix) CMDR_CUDA_CHECK(cudaMemsetAsync(map[c], 0, sizeof(double) * g->npix, st)); }
      else { for (int c = 0; c < ncomp; ++c) if (a->nalm) CMDR_CUDA_CHECK(cudaMemsetAsync(alm[c], 0, sizeof(double) * a->nalm * (a->real_packed ? 1 : 2), st)); }
    }
    return;
  }
  LegGeom G;
  G.nslots = g->npairs; G.NPL = g->npairs; G.nowners = 1; G.NML = a->nm; G.ncomp_tot = ncomp; G.comp0 = 0;
  G.trig = g->d_trig; G.mlim = ensure_mlim(g, a->lmax, spin);
  G.seed_geom = g; G.seed_alm = a;
  if (spin == 2 && !job.deriv1 && spin2_scalar_on()) {   // spin 2 as scalar sums (legendre.cu, launch_s2s_*)
    ensure_coef(a, COEF_KEY_S0X2P2);
    const CoefDev &c = a->coef[COEF_KEY_S0X2P2];
    A.s2s_coef = c.tab; A.s2s_mix = c.tab2; A.s2s_cofs = c.ofs; A.s2s_tofs = c.tofs; A.s2s_trows = c.trows; A.s2s_nl = c.nofs;
    A.s2s_K0 = ensure_start_norms(a, 0);
    int np = 0;   // pairs are sorted by colatitude: the polar ones come first
    while (np < g->npairs && g->sth[np] < S2S_MIN_STH) ++np;
    G.s2s_npolar = np;
  }
  PhaseLayout L = single_layout(a, g->npairs, ncomp, 0);
  double4 *ph = static_cast<double4 *>(scratch_get("phase", sizeof(double4) * (size_t)ncomp * a->nm * g->npairs));
  if (synth) {
    prof_begin(spin, 0, st);
    launch_legendre_synth(G, A, alm, ph, st);
    prof_end(st);
    prof_begin(100 + spin, 0, st);
    ringfft_synth(g, ncomp, L, ph, map, job.weighted, job.add, st, opts ? pixscale : nullptr);
    prof_end(st);
  } else {
    prof_begin(100 + spin, 1, st);
    ringfft_anal(g, ncomp, L, ph, map, job.weighted, st);
    prof_end(st);
    const size_t nd = (size_t)a->nalm * (a->real_packed ? 1 : 2);
    double *const *out = det_add_begin(job.add, alm, ncomp, nd, st);
    if (!job.add)
      for (int c = 0; c < ncomp; ++c)
        CMDR_CUDA_CHECK(cudaMemsetAsync(alm[c], 0, sizeof(double) * nd, st));
    prof_begin(spin, 1, st);
    launch_legendre_anal(G, A, out, ph, st);
    prof_end(st);
    det_add_end(out, alm, ncomp, nd, st);
  }
}

// Host/device pointer marshalling shared by sharp_execute and the IQU entry point.
Staged stage_in(const char *tag, double *const *ptrs, int n, long long count, bool copy_in, cudaStream_t st) {
  Staged s;
  s.dev.resize(n); s.host.resize(n);
  bool dev = true;
  for (int c = 0; c < n; ++c) dev = dev && is_device_ptr(ptrs[c]);
  if (dev || count == 0) { for (int c = 0; c < n; ++c) s.dev[c] = ptrs[c]; return s; }
  s.staged = true;
  double *buf = static_cast<double *>(scratch_get(tag, sizeof(double) * (size_t)count * n));
  for (int c = 0; c < n; ++c) {
    s.host[c] = ptrs[c]; s.dev[c] = buf + (size_t)c * count;
    if (copy_in) CMDR_CUDA_CHECK(cudaMemcpyAsync(s.dev[c], s.host[c], sizeof(double) * count, cudaMemcpyHostToDevice, st));
  }
  return s;
}
void stage_out(Staged &s, long long count, cudaStream_t st) {
  if (!s.staged) return;
  for (size_t c = 0; c < s.dev.size(); ++c)
    CMDR_CUDA_CHECK(cudaMemcpyAsync(s.host[c], s.dev[c], sizeof(double) * count, cudaMemcpyDeviceToHost, st));
}

// ---------------------------------------------------------------- pipelined host path
// With pinned host buffers the transform is cut into ring-pair chunks so that PCIe copies of
// one chunk overlap the kernels of the next (synthesis: Legendre+FFT of chunk c+1 while the
// map rows of chunk c go D2H; analysis: H2D of chunk c+1 while chunk c is transformed and
// accumulated into the a_lm).  Pageable buffers (the plain Fortran case) take the simple
// staged path above; registering the arrays once with cudaHostRegister enables this one.
bool is_pinned_host(const void *p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}

cudaStream_t copy_stream() {
  static std::map<int, cudaStream_t> cs;
  int dev = 0;
  CMDR_CUDA_CHECK(cudaGetDevice(&dev));
  auto it = cs.find(dev);
  if (it != cs.end()) return it->second;
  cudaStream_t s;
  CMDR_CUDA_CHECK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  cs[dev] = s;
  return s;
}

// second compute stream: consecutive m-chunk launches of the pipelined path alternate between the caller's
// stream and this one, so that the next launch fills the SMs the previous one leaves idle while it drains
// (an m-chunk launch is only ~2 waves of CTAs of similar length)
static cudaStream_t aux_stream() {
  static std::map<int, cudaStream_t> as;
  int dev = 0;
  CMDR_CUDA_CHECK(cudaGetDevice(&dev));
  auto it = as.find(dev);
  if (it != as.end()) return it->second;
  cudaStream_t s;
  CMDR_CUDA_CHECK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  as[dev] = s;
  return s;
}

cudaEvent_t pooled_event(size_t i) {
  static std::vector<cudaEvent_t> pool;
  while (pool.size() <= i) {
    cudaEvent_t e;
    CMDR_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    pool.push_back(e);
  }
  return pool[i];
}

// pixel ranges [begin, end) of a sub-geometry's northern and southern rows
void sub_ranges(const sharp_geom_info *s, long long &nb, long long &ne, long long &sb, long long &se) {
  const int n = s->npairs;
  nb = s->ofsN[0]; ne = s->ofsN[n - 1] + s->nph[n - 1];
  int last = n - 1;
  while (last >= 0 && s->ofsS[last] < 0) --last;
  if (last < 0) { sb = se = 0; return; }
  sb = s->ofsS[last]; se = s->ofsS[0] + s->nph[0];
}

// Columns of consecutive local m's are contiguous in the packed a_lm array for the layouts Commander
// builds (sharp_make_mmajor_real_packed_alm_info): returns their start offsets (doubles) and cuts the
// m range into `nch` pieces of about equal size.  False for layouts that are not dense.
bool alm_m_chunks(const sharp_alm_info *a, long long nalm_d, int nch, std::vector<long long> &mstart,
                         std::vector<int> &mcut) {
  mstart.assign(a->nm + 1, 0);
  const long long f2 = a->real_packed ? 1 : 2;
  long long pos = 0;
  for (int i = 0; i < a->nm; ++i) {
    const int m = a->mval[i];
    const long long f = (a->real_packed && m > 0) ? 2 : 1;
    const long long b = (a->mvstart[i] + f * m) * f2, e = (a->mvstart[i] + f * (a->lmax + 1)) * f2;
    if (b != pos) return false;
    mstart[i] = b; pos = e;
  }
  mstart[a->nm] = pos;
  if (pos != nalm_d || a->nm < 64) return false;
  mcut.assign(nch + 1, a->nm);
  mcut[0] = 0;
  for (int j = 1; j < nch; ++j) {
    int i = mcut[j - 1];
    while (i < a->nm && mstart[i] < nalm_d * j / nch) ++i;
    mcut[j] = i;
  }
  return true;
}

static bool try_pipelined(const Job &job, double *const *alm, double *const *map, sharp_geom_info *g,
                          sharp_alm_info *a, cudaStream_t st) {
  static const bool disabled = getenv("CMDR_SHT_NO_PIPELINE") != nullptr;
  const int spin = job.spin, nca = job.alm_cols, ncomp = job.map_cols;
  if (disabled || job.add || g->npix < (1 << 21) || a->nm == 0) return false;
  // Deterministic analysis takes the staged path: the chunks below run spin 2 on the spin-2 kernels without seed tables,
  // while a transform of device arrays runs the scalar-sum route, so only the staged path gives the device path's bits.
  if (!job.synth && deterministic()) return false;
  // host arrays of either kind: pinned ones are copied in place, pageable ones (what sharp.f90:219-224 passes)
  // go through the library's pinned arena and the copy threads (hostio.cu)
  for (int c = 0; c < nca; ++c)
    if (host_kind(alm[c]) == HostKind::Device) return false;
  for (int c = 0; c < ncomp; ++c)
    if (host_kind(map[c]) == HostKind::Device) return false;
  HostIO ioA, ioM;
  // tuning aid: CMDR_SHT_PIPE_TRACE=1 prints a timeline (ms since the call started) of the stream markers below
  static const bool trace = getenv("CMDR_SHT_PIPE_TRACE") != nullptr;
  std::vector<std::pair<std::string, cudaEvent_t>> marks;
  auto mark = [&](const char *what, int i, cudaStream_t s) {
    if (!trace) return;
    cudaEvent_t e;
    CMDR_CUDA_CHECK(cudaEventCreate(&e));
    CMDR_CUDA_CHECK(cudaEventRecord(e, s));
    marks.emplace_back(std::string(what) + " " + std::to_string(i), e);
  };
  auto dump_marks = [&]() {
    if (!trace) return;
    fprintf(stderr, "[cmdr_sht pipe] type %d spin %d:", job.type, spin);
    for (size_t k = 1; k < marks.size(); ++k) {
      float ms = 0;
      cudaEventElapsedTime(&ms, marks[0].second, marks[k].second);
      fprintf(stderr, " %s@%.2f", marks[k].first.c_str(), ms);
    }
    fprintf(stderr, "\n");
    for (auto &m : marks) cudaEventDestroy(m.second);
  };
  static const bool two_streams = !(getenv("CMDR_SHT_TWO_STREAMS") && atoi(getenv("CMDR_SHT_TWO_STREAMS")) == 0);
  static const int njoint = getenv("CMDR_SHT_JOINT") ? std::max(1, atoi(getenv("CMDR_SHT_JOINT"))) : 2;
  static const int nchunks = getenv("CMDR_SHT_CHUNKS") ? atoi(getenv("CMDR_SHT_CHUNKS")) : 8;
  ensure_subgeoms(g, nchunks);
  if (g->subs.empty()) return false;
  ensure_geom_device(g);
  LegAlm A = make_legalm(a, job);
  const long long nalm_d = a->nalm * (a->real_packed ? 1 : 2);
  double *alm_buf = static_cast<double *>(scratch_get("stage_alm", sizeof(double) * (size_t)nalm_d * nca));
  double *map_buf = static_cast<double *>(scratch_get("stage_map", sizeof(double) * (size_t)g->npix * ncomp));
  double4 *ph = static_cast<double4 *>(scratch_get("phase", sizeof(double4) * (size_t)ncomp * a->nm * g->npairs));
  ioA.init("hstage_alm", alm, nca, nalm_d, true);
  ioM.init("hstage_map", map, ncomp, g->npix, true);
  size_t maxz = 0;
  for (sharp_geom_info *sub : g->subs) { ensure_geom_device(sub); maxz = std::max(maxz, ringfft_scratch_elems(sub)); }
  if (maxz) scratch_get("fftbuf", sizeof(double2) * maxz * ncomp);
  double *alm_dev[2], *map_dev[2];
  for (int c = 0; c < nca; ++c) alm_dev[c] = alm_buf + (size_t)c * nalm_d;
  for (int c = 0; c < ncomp; ++c) map_dev[c] = map_buf + (size_t)c * g->npix;
  LegGeom G;
  G.nslots = g->npairs; G.NPL = g->npairs; G.nowners = 1; G.NML = a->nm; G.ncomp_tot = ncomp; G.comp0 = 0;
  G.trig = g->d_trig; G.mlim = ensure_mlim(g, a->lmax, spin);
  PhaseLayout L = single_layout(a, g->npairs, ncomp, 0);
  cudaStream_t cs = copy_stream();
  const int ns = (int)g->subs.size();
  mark("start", 0, st);
  if (job.synth) {
    // a_lm upload in NMCH chunks of local m's (the packed columns of consecutive m's are contiguous): the
    // first ring-pair chunk runs its Legendre kernel m-chunk by m-chunk as the data lands, so only the
    // first quarter of the upload is exposed.  Falls back to one copy for layouts that are not dense.
    static const int NMCH = getenv("CMDR_SHT_MCHUNKS") ? std::max(1, std::min(16, atoi(getenv("CMDR_SHT_MCHUNKS")))) : 16;
    std::vector<long long> mstart;
    std::vector<int> mcut;
    const int nmch = alm_m_chunks(a, nalm_d, NMCH, mstart, mcut) ? NMCH : 1;
    if (nmch == 1) {
      for (int c = 0; c < nca; ++c) ioA.h2d(alm_dev[c], c, 0, nalm_d, st);
    } else {
      cudaEvent_t e0 = pooled_event(ns + 1);               // earlier work on `st` may still read the staging buffer
      CMDR_CUDA_CHECK(cudaEventRecord(e0, st));
      CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, e0, 0));
    }
    // m-chunk j: upload on the copy stream (for pageable caller arrays the copy threads stage it first, which blocks
    // this thread -- hence the kernels of chunk j are queued right behind its upload, not after all uploads)
    auto upload_mchunk = [&](int j) {
      const long long b = mstart[mcut[j]], e = mstart[mcut[j + 1]];
      for (int c = 0; c < nca; ++c) ioA.h2d(alm_dev[c] + b, c, b, e - b, cs);
      CMDR_CUDA_CHECK(cudaEventRecord(pooled_event(ns + 2 + j), cs));
      mark("up", j, cs);
    };
    // The first `nj` ring-pair chunks share the m-chunked start: per m-chunk the Legendre kernels of all of
    // them run before the next m-chunk is needed, so the a_lm upload (4.7 ms for spin 2 at lmax 4000) hides
    // behind nj chunks of compute instead of one.
    const int nj = nmch > 1 ? std::min(njoint, ns) : 1;
    auto finish_chunk = [&](int i) {
      sharp_geom_info *sub = g->subs[i];
      L.pair0 = sub->pair0;
      mark("leg", i, st);
      ringfft_synth(sub, ncomp, L, ph, map_dev, job.weighted, false, st);
      mark("fft", i, st);
      cudaEvent_t e = pooled_event(i);
      CMDR_CUDA_CHECK(cudaEventRecord(e, st));
      CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, e, 0));
      long long nb, ne, sb, se;
      sub_ranges(sub, nb, ne, sb, se);
      for (int c = 0; c < ncomp; ++c) {
        ioM.d2h(map_dev[c] + nb, c, nb, ne - nb, cs);
        ioM.d2h(map_dev[c] + sb, c, sb, se - sb, cs);
      }
      ioM.commit(cs);
      mark("down", i, cs);
    };
    if (nmch > 1) {
      cudaStream_t as = two_streams ? aux_stream() : st;
      if (as != st) CMDR_CUDA_CHECK(cudaStreamWaitEvent(as, pooled_event(ns + 1), 0));   // e0: earlier work on st
      for (int j = 0; j < nmch; ++j) {
        cudaStream_t sj = (j & 1) ? as : st;
        upload_mchunk(j);
        CMDR_CUDA_CHECK(cudaStreamWaitEvent(sj, pooled_event(ns + 2 + j), 0));
        LegAlm Aj = A;
        Aj.im_begin = mcut[j]; Aj.im_end = mcut[j + 1];
        // one launch over the merged slot range of the first nj chunks (consecutive ring pairs; belt first)
        G.slot_begin = g->subs[ns - nj]->pair0; G.slot_end = g->subs[ns - 1]->pair0 + g->subs[ns - 1]->npairs;
        launch_legendre_synth(G, Aj, alm_dev, ph, sj, true);
        mark("legm", j, sj);
      }
      if (as != st) {
        cudaEvent_t ea = pooled_event(ns + 20);
        CMDR_CUDA_CHECK(cudaEventRecord(ea, as));
        CMDR_CUDA_CHECK(cudaStreamWaitEvent(st, ea, 0));
      }
      for (int i = ns - 1; i >= ns - nj; --i) finish_chunk(i);
    }
    for (int i = (nmch > 1 ? ns - nj : ns) - 1; i >= 0; --i) {
      sharp_geom_info *sub = g->subs[i];
      G.slot_begin = sub->pair0; G.slot_end = sub->pair0 + sub->npairs;
      launch_legendre_synth(G, A, alm_dev, ph, st, nmch == 1 && i == ns - 1);
      finish_chunk(i);
    }
    ioM.drain();                                   // pageable caller map: rows leave the arena as their chunks land
    CMDR_CUDA_CHECK(cudaStreamSynchronize(cs));
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  } else {
    static const int NMCH = getenv("CMDR_SHT_MCHUNKS") ? std::max(1, std::min(16, atoi(getenv("CMDR_SHT_MCHUNKS")))) : 16;
    std::vector<long long> mstart;
    std::vector<int> mcut;
    const int nmch = alm_m_chunks(a, nalm_d, NMCH, mstart, mcut) ? NMCH : 1;
    // the copy stream must not overwrite staging rows an earlier call on `st` still reads
    cudaEvent_t e0 = pooled_event(ns);
    CMDR_CUDA_CHECK(cudaEventRecord(e0, st));
    CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, e0, 0));
    for (int c = 0; c < ncomp; ++c) CMDR_CUDA_CHECK(cudaMemsetAsync(alm_dev[c], 0, sizeof(double) * nalm_d, st));
    const int nj = nmch > 1 ? std::min(njoint, ns) : 1;
    for (int i = 0; i < ns; ++i) {               // small polar chunks first so compute starts early
      sharp_geom_info *sub = g->subs[i];
      long long nb, ne, sb, se;
      sub_ranges(sub, nb, ne, sb, se);
      for (int c = 0; c < ncomp; ++c) {
        ioM.h2d(map_dev[c] + nb, c, nb, ne - nb, cs);
        ioM.h2d(map_dev[c] + sb, c, sb, se - sb, cs);
      }
      cudaEvent_t e = pooled_event(i);
      CMDR_CUDA_CHECK(cudaEventRecord(e, cs));
      mark("up", i, cs);
      CMDR_CUDA_CHECK(cudaStreamWaitEvent(st, e, 0));
      L.pair0 = sub->pair0;
      ringfft_anal(sub, ncomp, L, ph, map_dev, job.weighted, st);
      mark("fft", i, st);
      G.slot_begin = sub->pair0; G.slot_end = sub->pair0 + sub->npairs;
      if (i < ns - nj) { launch_legendre_anal(G, A, alm_dev, ph, st); mark("leg", i, st); }
    }
    // last `nj` ring-pair chunks: m-chunk by m-chunk over all of them, so that the finished a_lm columns go
    // back to the host while the next m-chunk is still being accumulated (nj chunks of compute per slice of
    // the download; only the last slice is exposed)
    cudaStream_t as = (two_streams && nmch > 1) ? aux_stream() : st;
    if (as != st) {
      cudaEvent_t ef = pooled_event(ns + 20);              // ring FFTs and earlier chunks done
      CMDR_CUDA_CHECK(cudaEventRecord(ef, st));
      CMDR_CUDA_CHECK(cudaStreamWaitEvent(as, ef, 0));
    }
    for (int j = 0; j < nmch && nj > 0; ++j) {
      cudaStream_t sj = (j & 1) ? as : st;
      LegAlm Aj = A;
      if (nmch > 1) { Aj.im_begin = mcut[j]; Aj.im_end = mcut[j + 1]; }    // (mcut is empty when the m's are not chunkable)
      G.slot_begin = g->subs[ns - nj]->pair0; G.slot_end = g->subs[ns - 1]->pair0 + g->subs[ns - 1]->npairs;
      launch_legendre_anal(G, Aj, alm_dev, ph, sj);   // merged slot range of the last nj chunks
      if (nmch > 1) {
        cudaEvent_t e = pooled_event(ns + 2 + j);
        CMDR_CUDA_CHECK(cudaEventRecord(e, sj));
        mark("legm", j, sj);
        CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, e, 0));
        const long long b = mstart[mcut[j]], e2 = mstart[mcut[j + 1]];
        for (int c = 0; c < ncomp; ++c) ioA.d2h(alm_dev[c] + b, c, b, e2 - b, cs);
        ioA.commit(cs);
        mark("down", j, cs);
      }
    }
    if (nmch == 1) {
      for (int c = 0; c < ncomp; ++c) ioA.d2h(alm_dev[c], c, 0, nalm_d, st);
      ioA.commit(st);
    }
    ioA.drain();
    CMDR_CUDA_CHECK(cudaStreamSynchronize(cs));
    if (as != st) CMDR_CUDA_CHECK(cudaStreamSynchronize(as));
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  dump_marks();
  return true;
}

// (l,m) count over the local m's times ring pairs (an unpaired ring counts half), times `per` nominal flops
static unsigned long long lm_pair_flops(const sharp_geom_info *g, const sharp_alm_info *a, double per) {
  double nlm = 0;
  for (int m : a->mval) nlm += a->lmax + 1 - m;
  double pairs = 0;
  for (int p = 0; p < g->npairs; ++p) pairs += (g->ofsN[p] >= 0 && g->ofsS[p] >= 0) ? 1.0 : 0.5;
  return (unsigned long long)(nlm * pairs * per);
}
unsigned long long nominal_flops(const sharp_geom_info *g, const sharp_alm_info *a, int spin) {
  return lm_pair_flops(g, a, spin == 0 ? 8.0 : 28.0);
}
// `opcnt` of a job: DERIV1 counts 20 per (l, m, ring pair) -- 12 for the spin-1 recurrence, 4 accumulate FMAs (FMA = 2)
unsigned long long job_opcnt(const sharp_geom_info *g, const sharp_alm_info *a, const Job &job) {
  return job.deriv1 ? lm_pair_flops(g, a, 20.0) : nominal_flops(g, a, job.spin);
}

void execute_any(const Job &job, void *alm_v, void *map_v, sharp_geom_info *g, sharp_alm_info *a, double *time,
                 unsigned long long *opcnt, cudaStream_t st) {
  auto t0 = std::chrono::steady_clock::now();
  const bool synth = job.synth, add = job.add;
  double *const *alm = static_cast<double *const *>(alm_v);
  double *const *map = static_cast<double *const *>(map_v);
  const long long nalm_d = a->nalm * (a->real_packed ? 1 : 2);
  if (!try_pipelined(job, alm, map, g, a, st)) {
    Staged sa = stage_in("stage_alm", alm, job.alm_cols, nalm_d, synth || add, st);
    Staged sm = stage_in("stage_map", map, job.map_cols, g->npix, !synth || add, st);
    run_single(job, sa.dev.data(), sm.dev.data(), g, a, st);
    if (synth) stage_out(sm, g->npix, st); else stage_out(sa, nalm_d, st);
    if (sa.staged || sm.staged || time) CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  if (time) *time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  if (opcnt) *opcnt = job_opcnt(g, a, job);
}

}  // namespace cmdr

extern "C" {

void sharp_execute(int type, int spin, void *alm, void *map, const sharp_geom_info *geom_info,
                   const sharp_alm_info *alm_info, int flags, double *time, unsigned long long *opcnt) {
  const Job job = job_or_abort("sharp_execute", type, spin, flags);
  execute_any(job, alm, map, const_cast<sharp_geom_info *>(geom_info), const_cast<sharp_alm_info *>(alm_info), time,
              opcnt, (cudaStream_t)0);
}

int cmdr_sht_version(void) { return 100; }

void cmdr_sht_execute_dev(int type, int spin, double *const *alm, double *const *map,
                          const sharp_geom_info *geom_info, const sharp_alm_info *alm_info, int flags,
                          void *stream) {
  const Job job = job_or_abort("cmdr_sht_execute_dev", type, spin, flags);
  run_single(job, alm, map, const_cast<sharp_geom_info *>(geom_info), const_cast<sharp_alm_info *>(alm_info),
             (cudaStream_t)stream);
}

void cmdr_sht_execute_iqu(int type, double *const *alm3, double *const *map3, const sharp_geom_info *geom_T,
                          const sharp_geom_info *geom_P, const sharp_alm_info *alm_info, int flags,
                          void *stream) {
  const Job jT = job_or_abort("cmdr_sht_execute_iqu", type, 0, flags, true);
  const Job jP = job_or_abort("cmdr_sht_execute_iqu", type, 2, flags, true);
  cudaStream_t st = (cudaStream_t)stream;
  sharp_geom_info *gT = const_cast<sharp_geom_info *>(geom_T), *gP = const_cast<sharp_geom_info *>(geom_P);
  sharp_alm_info *a = const_cast<sharp_alm_info *>(alm_info);
  const bool synth = jT.synth, add = jT.add;
  const long long nalm_d = a->nalm * (a->real_packed ? 1 : 2);
  Staged sa = stage_in("stage_alm", alm3, 3, nalm_d, synth || add, st);
  Staged sm = stage_in("stage_map", map3, 3, gT->npix, !synth || add, st);
  run_single(jT, sa.dev.data(), sm.dev.data(), gT, a, st);
  run_single(jP, sa.dev.data() + 1, sm.dev.data() + 1, gP, a, st);
  if (synth) stage_out(sm, gT->npix, st); else stage_out(sa, nalm_d, st);
  if (sa.staged || sm.staged) CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

// Batch of independent IQU transforms that share the handles (the 30 frequency bands of one Gibbs step,
// BASELINE config 5; `comm_map%Y` / `%YtW` in a loop over bands, commander3/src/comm_cr_mod.f90:880-918).
// With host buffers the bands are software-pipelined over three streams and two sets of staging buffers:
// the upload of band b+1 and the download of band b-1 run beside the kernels of band b (both DMA
// engines busy), instead of copy-compute-copy per band.  Pinned host buffers give the full overlap.
void cmdr_sht_execute_iqu_batch(int type, int nbatch, double *const *alm3, double *const *map3,
                                const sharp_geom_info *geom_T, const sharp_geom_info *geom_P,
                                const sharp_alm_info *alm_info, int flags, void *stream) {
  const Job jT = job_or_abort("cmdr_sht_execute_iqu_batch", type, 0, flags, true);
  const Job jP = job_or_abort("cmdr_sht_execute_iqu_batch", type, 2, flags, true);
  cudaStream_t st = (cudaStream_t)stream;
  sharp_geom_info *gT = const_cast<sharp_geom_info *>(geom_T), *gP = const_cast<sharp_geom_info *>(geom_P);
  sharp_alm_info *a = const_cast<sharp_alm_info *>(alm_info);
  const bool synth = jT.synth, add = jT.add;
  const long long nalm_d = a->nalm * (a->real_packed ? 1 : 2);
  const long long npix = gT->npix;
  if (nbatch <= 0) return;
  bool dev = true;
  for (int i = 0; i < 3 * nbatch; ++i) dev = dev && is_device_ptr(alm3[i]) && is_device_ptr(map3[i]);
  if (dev || nalm_d == 0 || npix == 0) {
    for (int b = 0; b < nbatch; ++b)
      cmdr_sht_execute_iqu(type, alm3 + 3 * b, map3 + 3 * b, geom_T, geom_P, alm_info, flags, stream);
    return;
  }
  static std::map<int, std::pair<cudaStream_t, cudaStream_t>> cstreams;   // per device: copy-in, copy-out
  int device = 0;
  CMDR_CUDA_CHECK(cudaGetDevice(&device));
  if (!cstreams.count(device)) {
    cudaStream_t s1, s2;
    CMDR_CUDA_CHECK(cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking));
    CMDR_CUDA_CHECK(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
    cstreams[device] = {s1, s2};
  }
  cudaStream_t cin = cstreams[device].first, cout = cstreams[device].second;
  double *abuf[2], *mbuf[2];
  abuf[0] = static_cast<double *>(scratch_get("batch_alm0", sizeof(double) * (size_t)nalm_d * 3));
  abuf[1] = static_cast<double *>(scratch_get("batch_alm1", sizeof(double) * (size_t)nalm_d * 3));
  mbuf[0] = static_cast<double *>(scratch_get("batch_map0", sizeof(double) * (size_t)npix * 3));
  mbuf[1] = static_cast<double *>(scratch_get("batch_map1", sizeof(double) * (size_t)npix * 3));
  std::vector<cudaEvent_t> up(nbatch), done(nbatch), down(nbatch);
  for (int b = 0; b < nbatch; ++b) {
    CMDR_CUDA_CHECK(cudaEventCreateWithFlags(&up[b], cudaEventDisableTiming));
    CMDR_CUDA_CHECK(cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming));
    CMDR_CUDA_CHECK(cudaEventCreateWithFlags(&down[b], cudaEventDisableTiming));
  }
  cudaEvent_t start;
  CMDR_CUDA_CHECK(cudaEventCreateWithFlags(&start, cudaEventDisableTiming));
  CMDR_CUDA_CHECK(cudaEventRecord(start, st));            // earlier work on `st` may still use the buffers
  CMDR_CUDA_CHECK(cudaStreamWaitEvent(cin, start, 0));
  CMDR_CUDA_CHECK(cudaStreamWaitEvent(cout, start, 0));
  // inputs / outputs of one band
  double **in_host = const_cast<double **>(synth ? alm3 : map3), **out_host = const_cast<double **>(synth ? map3 : alm3);
  const long long nin = synth ? nalm_d : npix, nout = synth ? npix : nalm_d;
  for (int b = 0; b < nbatch; ++b) {
    const int s = b & 1;
    double *in_dev = synth ? abuf[s] : mbuf[s], *out_dev = synth ? mbuf[s] : abuf[s];
    // upload band b once the kernels of band b-2 no longer read this staging set
    if (b >= 2) CMDR_CUDA_CHECK(cudaStreamWaitEvent(cin, done[b - 2], 0));
    for (int c = 0; c < 3; ++c)
      CMDR_CUDA_CHECK(cudaMemcpyAsync(in_dev + (size_t)c * nin, in_host[3 * b + c], sizeof(double) * nin, cudaMemcpyHostToDevice, cin));
    // accumulate into the caller's output: it has to come up too -- into the staging set whose previous content
    // (the result of band b-2) may still be on its way down on `cout`
    if (add && b >= 2) CMDR_CUDA_CHECK(cudaStreamWaitEvent(cin, down[b - 2], 0));
    if (add)
      for (int c = 0; c < 3; ++c)
        CMDR_CUDA_CHECK(cudaMemcpyAsync(out_dev + (size_t)c * nout, out_host[3 * b + c], sizeof(double) * nout, cudaMemcpyHostToDevice, cin));
    CMDR_CUDA_CHECK(cudaEventRecord(up[b], cin));
    // kernels of band b: after its upload, and after the download of band b-2 released the output set
    CMDR_CUDA_CHECK(cudaStreamWaitEvent(st, up[b], 0));
    if (b >= 2) CMDR_CUDA_CHECK(cudaStreamWaitEvent(st, down[b - 2], 0));
    double *ap[3], *mp[3];
    for (int c = 0; c < 3; ++c) { ap[c] = abuf[s] + (size_t)c * nalm_d; mp[c] = mbuf[s] + (size_t)c * npix; }
    run_single(jT, ap, mp, gT, a, st);
    run_single(jP, ap + 1, mp + 1, gP, a, st);
    CMDR_CUDA_CHECK(cudaEventRecord(done[b], st));
    // download band b
    CMDR_CUDA_CHECK(cudaStreamWaitEvent(cout, done[b], 0));
    for (int c = 0; c < 3; ++c)
      CMDR_CUDA_CHECK(cudaMemcpyAsync(out_host[3 * b + c], out_dev + (size_t)c * nout, sizeof(double) * nout, cudaMemcpyDeviceToHost, cout));
    CMDR_CUDA_CHECK(cudaEventRecord(down[b], cout));
  }
  CMDR_CUDA_CHECK(cudaStreamSynchronize(cout));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  for (int b = 0; b < nbatch; ++b) { cudaEventDestroy(up[b]); cudaEventDestroy(done[b]); cudaEventDestroy(down[b]); }
  cudaEventDestroy(start);
}

unsigned long long cmdr_sht_launch_count(void) { return g_launches.load(); }
void cmdr_sht_set_profiling(int on) { g_profiling = on; }
int cmdr_sht_last_legendre_ms(double *entries3, int max) {
  prof_collect();   // waits for the recorded events; call after synchronising the stream
  int n = (int)g_prof.size() / 3;
  if (n > max) n = max;
  for (int i = 0; i < 3 * n; ++i) entries3[i] = g_prof[i];
  g_prof.clear();
  return n;
}
unsigned long long cmdr_sht_nominal_flops(const sharp_geom_info *g, const sharp_alm_info *a, int spin) {
  return nominal_flops(g, a, spin);
}
void cmdr_sht_release_caches(void) { scratch_release(); pinned_release(); seed_release(); }

}  // extern "C"
