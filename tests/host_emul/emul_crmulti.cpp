// The input checks and slot maps of cmdr_cr_setup_multi (commander_b200/csrc/cr_plan.h) and the per-slot arithmetic of
// its block preconditioner (cr_block.cuh), compiled with g++ for the CPU test-suite.  TEST ONLY.
#include <cstring>
#include <vector>

#include "../../commander_b200/csrc/cr_block.cuh"
#include "../../commander_b200/csrc/cr_plan.h"
using namespace cmdr;

namespace {
// a real-packed m-major handle (what sharp_make_mmajor_real_packed_alm_info builds) over the m's `ms`
sharp_alm_info make_alm(int lmax, int rp, int nm, const int *ms) {
  sharp_alm_info a;
  a.lmax = lmax; a.nm = nm; a.real_packed = rp != 0;
  a.mval.assign(ms, ms + nm);
  long long idx = 0;
  for (int i = 0; i < nm; ++i) {
    const int f = ms[i] == 0 ? 1 : 2;
    a.mvstart.push_back(idx - (long long)f * ms[i]);
    idx += (long long)f * (lmax + 1 - ms[i]);
  }
  a.nalm = idx;
  return a;
}
}  // namespace

// Handles: lmax < 0 stands for a NULL handle; ms holds the m lists one after the other (nm entries each).
// prior[k]: 0 = no sqrtS columns, 1 = all given, 2 = only the first.  Out: bstart [layout][nm], nalm and lmax per
// layout, L per band, misc = {nm, lmax_pre, nmaps_pre, lmax_all}, the block table bytes.  Returns 1 when valid, 0 with
// the reason in err.
extern "C" int emul_cr_plan(int ncomp, const int *comp_lmax, const int *comp_nmaps, const int *comp_rp, const int *comp_nm,
                            const int *comp_ms, const int *prior, int nbands, const int *band_lmax, const int *band_nmaps,
                            const int *band_rp, const int *band_nm, const int *band_ms, const int *band_hasP, int precond,
                            double device_bytes, long long *bstart, long long *nalm, int *lmax, int *L, int *misc,
                            double *bytes, char *err, int errlen) {
  std::vector<sharp_alm_info> ca, ba;
  ca.reserve(ncomp > 0 ? ncomp : 0); ba.reserve(nbands > 0 ? nbands : 0);
  std::vector<const sharp_alm_info *> cp, bp;
  std::vector<const sharp_geom_info *> gT, gP;
  static sharp_geom_info geom;
  static const double one = 1.0;
  std::vector<const double *> sS, cols;
  int o = 0;
  for (int k = 0; k < ncomp; ++k) {
    ca.push_back(make_alm(comp_lmax[k], comp_rp[k], comp_nm[k], comp_ms + o));
    o += comp_nm[k];
    cp.push_back(comp_lmax[k] < 0 ? nullptr : &ca.back());
    for (int j = 0; j < comp_nmaps[k]; ++j) sS.push_back(prior[k] == 1 || (prior[k] == 2 && j == 0) ? &one : nullptr);
  }
  o = 0;
  for (int q = 0; q < nbands; ++q) {
    ba.push_back(make_alm(band_lmax[q], band_rp[q], band_nm[q], band_ms + o));
    o += band_nm[q];
    bp.push_back(band_lmax[q] < 0 ? nullptr : &ba.back());
    gT.push_back(&geom);
    gP.push_back(band_hasP[q] ? &geom : nullptr);
    for (int j = 0; j < band_nmaps[q]; ++j) cols.push_back(&one);
  }
  const double F = 1.0;
  const CrPlan p = plan_cr_multi(ncomp, cp.data(), comp_nmaps, sS.data(), nbands, gT.data(), gP.data(), bp.data(), band_nmaps,
                                 cols.data(), cols.data(), &F, precond, (size_t)device_bytes);
  snprintf(err, errlen, "%s", p.error.c_str());
  if (!p.error.empty()) return 0;
  memcpy(bstart, p.bstart.data(), sizeof(long long) * p.bstart.size());
  memcpy(nalm, p.nalm.data(), sizeof(long long) * p.nalm.size());
  memcpy(lmax, p.lmax.data(), sizeof(int) * p.lmax.size());
  memcpy(L, p.L.data(), sizeof(int) * p.L.size());
  misc[0] = p.nm(); misc[1] = p.lmax_pre; misc[2] = p.nmaps_pre; misc[3] = p.lmax_all;
  *bytes = (double)p.precond_bytes;
  return 1;
}

// One block: t (n (n + 1) / 2 doubles, upper triangle, row-major) is finished and inverted in place, then z = M r.
extern "C" void emul_cr_block(int n, double *t, const double *sS, const int *prior, const double *r, double *z) {
  bool pr[CR_MAX_NPRE] = {};
  for (int k = 0; k < n; ++k) pr[k] = prior[k] != 0;
  cr_block_finish_invert<CR_MAX_NPRE>(t, 1, n, sS, pr);
  cr_block_apply<CR_MAX_NPRE>(t, 1, n, r, z);
}

extern "C" int emul_cr_tri(int k1, int k2, int n) { return cr_tri(k1, k2, n); }
