// cr_pinv.h -- the host side of the multi-component CR system's per-l factor tables and of its pseudo-inverse
// preconditioner (initDiffPrecond_pseudoinv / updateDiffPrecond_pseudoinv, commander3/src/comm_diffuse_comp_mod.f90:
// 1255-1294, 1560-1658): per (map, l) the (nbands + npre) x npre matrix V = [alpha_q b_l F_mean sqrt(S); P] and its
// pseudo-inverse U+.  Plain C++ (no CUDA) so that the CPU tests compile it with g++.
//
// Tables are [k][q][3][nl] (component, band, map, l), the layout the band and component gathers of cr_multi.cu read.
#pragma once
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <vector>

#include "cr_block.cuh"

namespace cmdr {

// sS[k][j][l] = sqrt(C_l) (0 for l < 2 in polarisation) or 1 without prior, 0 beyond lmax_k;
// f[k][q][j][l] = F_mean b_l where both the component and the band transform hold (j, l); g = f sS.
// sqrtS: NULL or sum_k cnm[k] columns (component-major, NULL columns for a component without prior), b_l: sum_q bnm[q]
// columns, F_mean[(q * nc + k) * 3 + j] (cmdr_cr_setup_multi); L[q]: the band's transform lmax; prior: bit k.
inline void cr_factor_tables(int nc, int nb, int nl, const int *cnm, const int *clmax, const int *bnm, const int *L,
                             unsigned prior, const double *const *sqrtS, const double *const *b_l, const double *F_mean,
                             std::vector<double> &sS, std::vector<double> &f, std::vector<double> &g) {
  std::vector<int> cofs(nc + 1, 0), bofs(nb + 1, 0);   // first sqrtS / b_l column of each
  for (int k = 0; k < nc; ++k) cofs[k + 1] = cofs[k] + cnm[k];
  for (int q = 0; q < nb; ++q) bofs[q + 1] = bofs[q] + bnm[q];
  sS.assign((size_t)nc * 3 * nl, 0.0);
  f.assign((size_t)nc * nb * 3 * nl, 0.0);
  g.assign(f.size(), 0.0);
  for (int k = 0; k < nc; ++k)
    for (int j = 0; j < cnm[k]; ++j)
      for (int l = 0; l <= clmax[k]; ++l) {
        double v = 1.0;
        if ((prior >> k) & 1u) v = (j > 0 && l < 2) ? 0.0 : sqrtS[cofs[k] + j][l];
        sS[((size_t)k * 3 + j) * nl + l] = v;
      }
  for (int k = 0; k < nc; ++k)
    for (int q = 0; q < nb; ++q)
      for (int j = 0; j < std::min(cnm[k], bnm[q]); ++j) {
        const double F = F_mean[((size_t)q * nc + k) * 3 + j];
        for (int l = 0; l <= std::min(clmax[k], L[q]); ++l) {
          const size_t i = (((size_t)k * nb + q) * 3 + j) * nl + l;
          f[i] = F * b_l[bofs[q] + j][l];
          g[i] = f[i] * sS[((size_t)k * 3 + j) * nl + l];
        }
      }
}

// out (cols x rows, row-major) = the pseudo-inverse of V (rows x cols, row-major), by one-sided Jacobi (Hestenes)
// rotations on the columns of V itself: V W = A with W orthogonal and the columns of A orthogonal, so V+ = W diag(1 /
// |a_i|^2) A^t over the columns kept.  Working on V rather than V^t V keeps the relative accuracy of columns whose
// scales span many decades.  Singular values |a_i| <= max(rows, cols) eps sigma_max are dropped (the default of
// torch.linalg.pinv and numpy.linalg.pinv's rcond).  A zero column is never rotated, so it gives an exactly zero row.
inline void cr_pinv(int rows, int cols, const double *V, double *out) {
  std::vector<double> A(V, V + (size_t)rows * cols), W((size_t)cols * cols, 0.0);
  for (int i = 0; i < cols; ++i) W[(size_t)i * cols + i] = 1.0;
  auto a = [&](int r, int c) -> double & { return A[(size_t)r * cols + c]; };
  auto w = [&](int r, int c) -> double & { return W[(size_t)r * cols + c]; };
  for (int sweep = 0; sweep < 80; ++sweep) {
    bool rotated = false;
    for (int i = 0; i < cols - 1; ++i)
      for (int j = i + 1; j < cols; ++j) {
        double al = 0.0, be = 0.0, ga = 0.0;
        for (int r = 0; r < rows; ++r) { al += a(r, i) * a(r, i); be += a(r, j) * a(r, j); ga += a(r, i) * a(r, j); }
        if (ga == 0.0 || std::fabs(ga) <= DBL_EPSILON * std::sqrt(al * be)) continue;
        rotated = true;
        const double zeta = (be - al) / (2.0 * ga);
        const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (std::fabs(zeta) + std::sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / std::sqrt(1.0 + t * t), s = c * t;
        for (int r = 0; r < rows; ++r) {
          const double x = a(r, i), y = a(r, j);
          a(r, i) = c * x - s * y; a(r, j) = s * x + c * y;
        }
        for (int r = 0; r < cols; ++r) {
          const double x = w(r, i), y = w(r, j);
          w(r, i) = c * x - s * y; w(r, j) = s * x + c * y;
        }
      }
    if (!rotated) break;
  }
  std::vector<double> sig(cols, 0.0);
  double smax = 0.0;
  for (int i = 0; i < cols; ++i) {
    double s = 0.0;
    for (int r = 0; r < rows; ++r) s += a(r, i) * a(r, i);
    sig[i] = std::sqrt(s);
    smax = std::max(smax, sig[i]);
  }
  const double tol = (double)std::max(rows, cols) * DBL_EPSILON * smax;
  std::fill(out, out + (size_t)rows * cols, 0.0);
  for (int i = 0; i < cols; ++i) {
    if (!(sig[i] > tol)) continue;
    const double inv2 = 1.0 / (sig[i] * sig[i]);
    for (int k = 0; k < cols; ++k) {
      const double wk = w(k, i) * inv2;
      if (wk == 0.0) continue;
      for (int r = 0; r < rows; ++r) out[(size_t)k * rows + r] += wk * a(r, i);
    }
  }
}

// The tables of the pseudo-inverse preconditioner from g (cr_factor_tables) and alpha[q * 3 + j] (compute_alpha_nu):
//   U[k][q][j][l]  = U+[k][q]               (band gather: a_q = sum_k U+ r_k)
//   UA[k][q][j][l] = alpha_qj^2 U+[k][q]    (component gather: z_k = sum_q alpha^2 U+ a'_q)
//   PP[j][l][cr_tri(k1, k2)] = sum_b U+[k1][nb + b] U+[k2][nb + b]   (the prior term P P^t, P = U+[:, nb:])
// for j < nmaps_pre, l <= lmax_pre, with V[q][k] = alpha_qj g[k][q][j][l] and V[nb + k][k] = 1 on the components with
// a prior that hold (j, l).
inline void cr_pinv_tables(int nc, int nb, int nl, int nmaps_pre, int lmax_pre, const int *cnm, const int *clmax,
                           unsigned prior, const std::vector<double> &g, const double *alpha, std::vector<double> &U,
                           std::vector<double> &UA, std::vector<double> &PP) {
  const int rows = nb + nc, ntri = nc * (nc + 1) / 2;
  U.assign((size_t)nc * nb * 3 * nl, 0.0);
  UA.assign(U.size(), 0.0);
  PP.assign((size_t)nmaps_pre * (lmax_pre + 1) * ntri, 0.0);
  std::vector<double> V((size_t)rows * nc), P((size_t)nc * rows);
  for (int j = 0; j < nmaps_pre; ++j)
    for (int l = 0; l <= lmax_pre; ++l) {
      std::fill(V.begin(), V.end(), 0.0);
      for (int q = 0; q < nb; ++q)
        for (int k = 0; k < nc; ++k) V[(size_t)q * nc + k] = alpha[q * 3 + j] * g[(((size_t)k * nb + q) * 3 + j) * nl + l];
      for (int k = 0; k < nc; ++k)
        if (((prior >> k) & 1u) && j < cnm[k] && l <= clmax[k]) V[(size_t)(nb + k) * nc + k] = 1.0;
      cr_pinv(rows, nc, V.data(), P.data());
      for (int k = 0; k < nc; ++k)
        for (int q = 0; q < nb; ++q) {
          const size_t i = (((size_t)k * nb + q) * 3 + j) * nl + l;
          U[i] = P[(size_t)k * rows + q];
          UA[i] = alpha[q * 3 + j] * alpha[q * 3 + j] * U[i];
        }
      double *pp = PP.data() + ((size_t)j * (lmax_pre + 1) + l) * ntri;
      for (int k1 = 0; k1 < nc; ++k1)
        for (int k2 = k1; k2 < nc; ++k2) {
          double s = 0.0;
          for (int b = 0; b < nc; ++b) s += P[(size_t)k1 * rows + nb + b] * P[(size_t)k2 * rows + nb + b];
          pp[cr_tri(k1, k2, nc)] = s;
        }
    }
}

}  // namespace cmdr
