// The host side of the pseudo-inverse preconditioner of the multi-component CR system (cr_pinv.h: the Jacobi
// pseudo-inverse, the per-l factor tables and the U+ / alpha^2 U+ / P P^t tables) and the argument checks of
// cmdr_cr_set_pseudoinv (check_cr_pseudoinv, cr_plan.h), compiled with g++ for the CPU test-suite.  TEST ONLY.
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../commander_b200/csrc/cr_pinv.h"
#include "../../commander_b200/csrc/cr_plan.h"
using namespace cmdr;

extern "C" void emul_cr_pinv(int rows, int cols, const double *V, double *out) { cr_pinv(rows, cols, V, out); }

// Components: cnm, clmax, Cl[k] (clmax + 1 rows of 3 doubles, row-major) or NULL without prior.  Bands: bnm, blmax,
// bl[q] ((blmax + 1) x 3 row-major).  F_mean[(q * nc + k) * 3 + j], alpha[q * 3 + j].  Writes U and UA
// ([k][q][3][nl], nl = max lmax + 1) and PP ([nmaps_pre][lmax_pre + 1][nc (nc + 1) / 2]).
extern "C" void emul_cr_pinv_tables(int nc, const int *cnm, const int *clmax, const double *const *Cl, int nb, const int *bnm,
                                    const int *blmax, const double *const *bl, const double *F_mean, const double *alpha,
                                    double *U, double *UA, double *PP) {
  int lmax_pre = 0, nmaps_pre = 0, lmax_all = 0;
  unsigned prior = 0;
  for (int k = 0; k < nc; ++k) {
    lmax_pre = std::max(lmax_pre, clmax[k]);
    nmaps_pre = std::max(nmaps_pre, cnm[k]);
    if (Cl[k]) prior |= 1u << k;
  }
  lmax_all = lmax_pre;
  std::vector<int> L(nb);
  for (int q = 0; q < nb; ++q) {
    lmax_all = std::max(lmax_all, blmax[q]);
    L[q] = std::min(blmax[q], lmax_pre);
  }
  const int nl = lmax_all + 1;
  // the columns cmdr_cr_setup_multi receives: sqrt(C_l) per component map, b_l per band map
  std::vector<std::vector<double>> scol, bcol;
  std::vector<const double *> sp, bp;
  for (int k = 0; k < nc; ++k)
    for (int j = 0; j < cnm[k]; ++j) {
      std::vector<double> c;
      if (Cl[k])
        for (int l = 0; l <= clmax[k]; ++l) c.push_back(std::sqrt(std::max(Cl[k][l * 3 + j], 0.0)));
      scol.push_back(c);
    }
  for (int q = 0; q < nb; ++q)
    for (int j = 0; j < bnm[q]; ++j) {
      std::vector<double> c;
      for (int l = 0; l <= blmax[q]; ++l) c.push_back(bl[q][l * 3 + j]);
      bcol.push_back(c);
    }
  for (auto &c : scol) sp.push_back(c.empty() ? nullptr : c.data());
  for (auto &c : bcol) bp.push_back(c.data());
  std::vector<double> sS, f, g, u, ua, pp;
  cr_factor_tables(nc, nb, nl, cnm, clmax, bnm, L.data(), prior, sp.data(), bp.data(), F_mean, sS, f, g);
  cr_pinv_tables(nc, nb, nl, nmaps_pre, lmax_pre, cnm, clmax, prior, g, alpha, u, ua, pp);
  memcpy(U, u.data(), sizeof(double) * u.size());
  memcpy(UA, ua.data(), sizeof(double) * ua.size());
  memcpy(PP, pp.data(), sizeof(double) * pp.size());
}

// Returns 1 when accepted, 0 with the reason in err.
extern "C" int emul_cr_pinv_check(int multi, int ncomp, double need_bytes, double free_bytes, char *err, int errlen) {
  const std::string e = check_cr_pseudoinv(multi != 0, ncomp, (size_t)need_bytes, (size_t)free_bytes);
  snprintf(err, errlen, "%s", e.c_str());
  return e.empty() ? 1 : 0;
}
