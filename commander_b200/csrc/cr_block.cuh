// cr_block.cuh -- the per-slot arithmetic of the block-diagonal preconditioner of the multi-component CR system
// (initDiffPrecond_diagonal / updateDiffPrecond_diagonal / applyDiffPrecond_diagonal,
// commander3/src/comm_diffuse_comp_mod.f90:1167-1557, 2186-2235): one symmetric npre x npre block per (map, l, m) slot,
// stored as its upper triangle, element (k1 <= k2) at cr_tri(k1, k2, n) * stride.  Shared with the host emulation test
// (tests/host_emul/emul_crblock.cpp), which compiles it with g++.
#pragma once
#include <math.h>

#ifdef __CUDACC__
#define CR_HD __host__ __device__ __forceinline__
#else
#define CR_HD inline
#endif

namespace cmdr {

CR_HD int cr_tri(int k1, int k2, int n) {
  if (k1 > k2) { const int t = k1; k1 = k2; k2 = t; }
  return k1 * n - k1 * (k1 - 1) / 2 + (k2 - k1);
}

// Finishes and inverts one block in place.  On entry t holds sum_nu N_lm b_l^2 F_k1 F_k2 over the bands; sS[k] is
// sqrt(C_l) of component k at this slot and prior[k] whether it has a prior (sS is ignored without one).  A component
// is active when its diagonal entry is > 0 (comp2ind /= -1); the active block becomes sqrt(S) M sqrt(S) + P and is
// inverted by Cholesky (it is SPD), inactive components pass through as identity rows.
template <int NMAX>
CR_HD void cr_block_finish_invert(double *t, long long stride, int n, const double *sS, const bool *prior) {
  double A[NMAX][NMAX];
  int act[NMAX];
  int na = 0;
  for (int k = 0; k < n; ++k)
    if (t[(long long)cr_tri(k, k, n) * stride] > 0.0) act[na++] = k;
  for (int a = 0; a < na; ++a)
    for (int b = 0; b <= a; ++b) {
      const int k1 = act[a], k2 = act[b];
      double v = t[(long long)cr_tri(k1, k2, n) * stride];
      if (prior[k1]) v *= sS[k1];
      if (prior[k2]) v *= sS[k2];
      if (a == b && prior[k1]) v += 1.0;
      A[a][b] = v;
    }
  // A = L L^t (lower triangle of A), then L^-1 in the upper triangle's mirror B
  for (int j = 0; j < na; ++j) {
    double d = A[j][j];
    for (int k = 0; k < j; ++k) d -= A[j][k] * A[j][k];
    d = sqrt(d);
    A[j][j] = d;
    for (int i = j + 1; i < na; ++i) {
      double s = A[i][j];
      for (int k = 0; k < j; ++k) s -= A[i][k] * A[j][k];
      A[i][j] = s / d;
    }
  }
  double B[NMAX][NMAX];   // B = L^-1 (lower)
  for (int j = 0; j < na; ++j) {
    B[j][j] = 1.0 / A[j][j];
    for (int i = j + 1; i < na; ++i) {
      double s = 0.0;
      for (int k = j; k < i; ++k) s -= A[i][k] * B[k][j];
      B[i][j] = s / A[i][i];
    }
  }
  for (int e = 0; e < n * (n + 1) / 2; ++e) t[(long long)e * stride] = 0.0;
  for (int k = 0; k < n; ++k) t[(long long)cr_tri(k, k, n) * stride] = 1.0;
  for (int a = 0; a < na; ++a)          // A^-1 = L^-t L^-1
    for (int b = a; b < na; ++b) {
      double s = 0.0;
      for (int k = b; k < na; ++k) s += B[k][a] * B[k][b];
      t[(long long)cr_tri(act[a], act[b], n) * stride] = s;
    }
}

// z = M r for one block (NMAX >= n; the loops unroll over NMAX so that r and z stay in registers)
template <int NMAX>
CR_HD void cr_block_apply(const double *t, long long stride, int n, const double *r, double *z) {
#pragma unroll
  for (int k1 = 0; k1 < NMAX; ++k1) {
    if (k1 >= n) break;
    double acc = 0.0;
#pragma unroll
    for (int k2 = 0; k2 < NMAX; ++k2) {
      if (k2 >= n) break;
      acc = fma(t[(long long)cr_tri(k1, k2, n) * stride], r[k2], acc);
    }
    z[k1] = acc;
  }
}

}  // namespace cmdr
