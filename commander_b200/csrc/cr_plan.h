// cr_plan.h -- the layout arithmetic of the multi-component constrained-realisation system (cr_multi.cu): the input
// checks of cmdr_cr_setup_multi and the maps between the a_lm slots of components, bands and the block preconditioner.
// Plain C++ (no CUDA) so that the CPU tests compile it with g++.
//
// Every handle of a system lists this rank's m's as comm_mapinfo builds them (round-robin m, commander3/src/
// comm_map_mod.f90:228-261): the same m's in the same order, each handle truncated at its own lmax.  In a real-packed
// layout the element (l, +-m) then sits at offset t = f (l - m) + [sign < 0] (f = 1 for m = 0, else 2) from the start of
// its m block whatever the lmax, so moving a slot between two layouts is "block start of m in the other layout + t":
// rank-local and without a search.
#pragma once
#include <algorithm>
#include <string>
#include <vector>

#include "sht_internal.h"

namespace cmdr {

constexpr int CR_MAX_NPRE = 16;   // components per block of the preconditioner (one block lives in a thread's registers)

struct CrPlan {
  std::string error;              // empty: the input is valid
  int ncomp = 0, nbands = 0;
  int lmax_pre = 0, nmaps_pre = 0;   // preconditioner layout: max lmax_k, max nmaps_k
  int lmax_all = 0;                  // largest lmax of any handle (length of the per-l tables - 1)
  std::vector<int> mval;             // the m's of the handle with the largest lmax: the common m index im
  std::vector<int> L;                // per band: the transform lmax min(lmax_q, lmax_pre)
  // Layouts: component k, band q as given, band q at L[q] (the given one when L[q] = lmax_q, else dense m-major with
  // the same m's), and the preconditioner slots (dense m-major at lmax_pre).  bstart[layout * nm + im]: element index
  // of (l = m, +m) of mval[im] in that layout, -1 when m is above its lmax.
  std::vector<long long> bstart;
  std::vector<long long> nalm;       // per layout
  std::vector<int> lmax;             // per layout
  size_t precond_bytes = 0;          // block table: npre (npre + 1) / 2 doubles per preconditioner slot and map
  int comp(int k) const { return k; }
  int band(int q) const { return ncomp + q; }
  int xform(int q) const { return ncomp + nbands + q; }
  int pre() const { return ncomp + 2 * nbands; }
  int nm() const { return (int)mval.size(); }
};

// Checks the arguments of cmdr_cr_setup_multi (same names and meaning) and derives the slot maps.  `device_bytes`:
// device memory the block preconditioner table may take.
inline CrPlan plan_cr_multi(int ncomp, const sharp_alm_info *const *comp_alm, const int *comp_nmaps,
                            const double *const *sqrtS, int nbands, const sharp_geom_info *const *band_geom_T,
                            const sharp_geom_info *const *band_geom_P, const sharp_alm_info *const *band_alm,
                            const int *band_nmaps, const double *const *invN, const double *const *b_l,
                            const double *F_mean, int precond, size_t device_bytes) {
  CrPlan p;
  auto fail = [&p](const std::string &e) { p.error = e; return p; };
  if (ncomp < 1) return fail("ncomp " + std::to_string(ncomp) + " (at least 1)");
  if (nbands < 1) return fail("nbands " + std::to_string(nbands) + " (at least 1)");
  if (!comp_alm || !comp_nmaps) return fail("comp_alm and comp_nmaps must not be NULL");
  if (!band_geom_T || !band_geom_P || !band_alm || !band_nmaps)
    return fail("band_geom_T, band_geom_P, band_alm and band_nmaps must not be NULL");
  if (!invN || !b_l || !F_mean) return fail("invN, b_l and F_mean must not be NULL");
  if (precond != 0 && precond != 1) return fail("precond " + std::to_string(precond) + " unsupported (0 = none, 1 = block diagonal)");
  if (precond == 1 && ncomp > CR_MAX_NPRE)
    return fail("ncomp " + std::to_string(ncomp) + " above the block preconditioner's limit of " + std::to_string(CR_MAX_NPRE));
  p.ncomp = ncomp; p.nbands = nbands;
  std::vector<const sharp_alm_info *> h;   // components, then bands
  int ncol = 0;
  for (int k = 0; k < ncomp; ++k) {
    const std::string who = "component " + std::to_string(k);
    if (!comp_alm[k]) return fail(who + ": alm_info is NULL");
    if (comp_nmaps[k] != 1 && comp_nmaps[k] != 3) return fail(who + ": nmaps " + std::to_string(comp_nmaps[k]) + " unsupported (1 or 3)");
    if (!comp_alm[k]->real_packed) return fail(who + ": needs the real-packed a_lm layout of comm_mapinfo");
    if (sqrtS) {
      int given = 0;
      for (int j = 0; j < comp_nmaps[k]; ++j) given += sqrtS[ncol + j] != nullptr;
      if (given != 0 && given != comp_nmaps[k]) return fail(who + ": sqrtS columns must be all NULL (no prior) or all given");
    }
    ncol += comp_nmaps[k];
    h.push_back(comp_alm[k]);
    p.lmax_pre = std::max(p.lmax_pre, comp_alm[k]->lmax);
    p.nmaps_pre = std::max(p.nmaps_pre, comp_nmaps[k]);
  }
  int bcol = 0;
  for (int q = 0; q < nbands; ++q) {
    const std::string who = "band " + std::to_string(q);
    if (!band_alm[q] || !band_geom_T[q]) return fail(who + ": alm_info or geom_T is NULL");
    if (band_nmaps[q] != 1 && band_nmaps[q] != 3) return fail(who + ": nmaps " + std::to_string(band_nmaps[q]) + " unsupported (1 or 3)");
    if (band_nmaps[q] == 3 && !band_geom_P[q]) return fail(who + ": geom_P is NULL with nmaps 3");
    if (!band_alm[q]->real_packed) return fail(who + ": needs the real-packed a_lm layout of comm_mapinfo");
    for (int j = 0; j < band_nmaps[q]; ++j, ++bcol)
      if (!invN[bcol] || !b_l[bcol]) return fail(who + ": invN and b_l columns must not be NULL");
    h.push_back(band_alm[q]);
  }
  // the common m list: that of the handle with the largest lmax; every other one is it truncated at its own lmax
  int ref = 0;
  for (size_t i = 0; i < h.size(); ++i) if (h[i]->lmax > h[ref]->lmax) ref = (int)i;
  p.lmax_all = h[ref]->lmax;
  p.mval = h[ref]->mval;
  auto name = [ncomp](int i) { return i < ncomp ? "component " + std::to_string(i) : "band " + std::to_string(i - ncomp); };
  for (size_t i = 0; i < h.size(); ++i) {
    std::vector<int> want;
    for (int m : p.mval) if (m <= h[i]->lmax) want.push_back(m);
    if (h[i]->mval != want)
      return fail(name((int)i) + ": its local m's differ from those of " + name(ref) + " truncated at lmax " +
                  std::to_string(h[i]->lmax) + " (every handle must list this rank's m's in comm_mapinfo's order)");
  }
  const int nm = p.nm();
  const int nl = 2 * nbands + ncomp + 1;
  p.bstart.assign((size_t)nl * nm, -1);
  p.nalm.assign(nl, 0);
  p.lmax.assign(nl, 0);
  auto given = [&](int layout, const sharp_alm_info *a) {
    for (int im = 0; im < a->nm; ++im) {   // a's im-th m is mval[im]: the lists agree up to a->nm
      const int m = a->mval[im];
      p.bstart[(size_t)layout * nm + im] = a->mvstart[im] + (long long)(m == 0 ? 1 : 2) * m;
    }
    p.nalm[layout] = a->nalm;
    p.lmax[layout] = a->lmax;
  };
  auto dense = [&](int layout, int lmax) {
    long long idx = 0;
    for (int im = 0; im < nm; ++im) {
      const int m = p.mval[im];
      if (m > lmax) continue;
      p.bstart[(size_t)layout * nm + im] = idx;
      idx += (long long)(m == 0 ? 1 : 2) * (lmax + 1 - m);
    }
    p.nalm[layout] = idx;
    p.lmax[layout] = lmax;
  };
  for (int k = 0; k < ncomp; ++k) given(p.comp(k), comp_alm[k]);
  p.L.resize(nbands);
  for (int q = 0; q < nbands; ++q) {
    given(p.band(q), band_alm[q]);
    p.L[q] = std::min(band_alm[q]->lmax, p.lmax_pre);
    if (p.L[q] == band_alm[q]->lmax) given(p.xform(q), band_alm[q]);
    else dense(p.xform(q), p.L[q]);
  }
  dense(p.pre(), p.lmax_pre);
  if (precond == 1) {
    p.precond_bytes = sizeof(double) * (size_t)(ncomp * (ncomp + 1) / 2) * p.nmaps_pre * (size_t)p.nalm[p.pre()];
    if (p.precond_bytes > device_bytes)
      return fail("the block preconditioner needs " + std::to_string(p.precond_bytes) + " bytes of device memory, " +
                  std::to_string(device_bytes) + " are free");
  }
  return p;
}

// Checks the arguments of cmdr_cr_set_mixing_map (same names and meaning) on one rank.  `multi`: the handle comes from
// cmdr_cr_setup_multi (the other arguments are read only then); comp_nmaps / band_nmaps as given to it.  Returns the
// reason of a refusal, or an empty string.
inline std::string check_cr_mixing(bool multi, int ncomp, int nbands, const int *comp_nmaps, const int *band_nmaps, int band,
                                   int comp, const double *const *F) {
  if (!multi) return "needs a handle of cmdr_cr_setup_multi (a cmdr_cr_setup handle has one component and no mixing)";
  if (band < 0 || band >= nbands) return "band " + std::to_string(band) + " out of range (nbands " + std::to_string(nbands) + ")";
  if (comp < 0 || comp >= ncomp) return "comp " + std::to_string(comp) + " out of range (ncomp " + std::to_string(ncomp) + ")";
  if (!F) return "";
  const int n = std::min(band_nmaps[band], comp_nmaps[comp]);
  for (int j = 0; j < n; ++j)
    if (!F[j])
      return "F[" + std::to_string(j) + "] is NULL: give all " + std::to_string(n) +
             " columns (min(nmaps_band, nmaps_comp)), or F = NULL for F_mean mixing";
  return "";
}

// Checks a cmdr_cr_set_pseudoinv call on one rank.  `multi`: the handle comes from cmdr_cr_setup_multi; `need_bytes`:
// device memory the tables still need (0 once they are built), `free_bytes`: what the device has free.  Returns the
// reason of a refusal, or an empty string.
inline std::string check_cr_pseudoinv(bool multi, int ncomp, size_t need_bytes, size_t free_bytes) {
  if (!multi)
    return "needs a handle of cmdr_cr_setup_multi (give a one-component system to cmdr_cr_setup_multi with ncomp = 1)";
  if (ncomp > CR_MAX_NPRE)
    return "ncomp " + std::to_string(ncomp) + " above the pseudo-inverse preconditioner's limit of " + std::to_string(CR_MAX_NPRE);
  if (need_bytes > free_bytes)
    return "the pseudo-inverse preconditioner needs " + std::to_string(need_bytes) + " bytes of device memory, " +
           std::to_string(free_bytes) + " are free";
  return "";
}

}  // namespace cmdr
