// Host emulation of the SHARP_ALM2MAP_DERIV1 accumulate of the CUDA kernels (commander_b200/csrc/legendre_core.cuh:
// d1_accum / d1_combine), compiled with g++ for the CPU test-suite.  TEST ONLY.  One (ring pair, m): the spin-1
// recurrence as synth_d1_kernel runs it, the phases once through the parity-split sums of the product header and
// once through the plain spin-1 form of synth2_kernel with cp = c, cm = -c.
#include <cmath>
#include <vector>
#include "../../commander_b200/csrc/legendre_core.cuh"
#include "../../commander_b200/csrc/sht_internal.h"
using namespace cmdr;

// c: 2 (lmax+1) doubles, the complex coefficient c_l of every l (only l >= max(m, 1) is read).
// out_d1 / out_ref: {Q.N.re, Q.N.im, Q.S.re, Q.S.im, U.N.re, U.N.im, U.S.re, U.S.im}; out_abs[0] = sum |c| (|P| + |M|).
extern "C" int emul_d1_phases(int lmax, int m, int nside, int north, const double *c, double *out_d1, double *out_ref,
                              double *out_abs) {
  std::vector<int> mval{m};
  std::vector<double> tab; std::vector<long long> ofs;
  build_coef_table(lmax, 1, mval, tab, ofs);
  std::vector<double> Ks;
  build_start_norms_spin(m, 1, Ks);
  long double omc, ns = nside;
  if (north < nside) omc = (long double)north * north / (3.0L * ns * ns);
  else omc = 1.0L - (2.0L * ns - north) * 2.0L / (3.0L * ns);
  RingTrig g{(double)(1.0L - omc), (double)sqrtl(omc * (2.0L - omc)), (double)sqrtl(0.5L * omc), (double)sqrtl(1.0L - 0.5L * omc)};
  const double SD = ldexp(1.0, -SCALE_BITS);
  const int l0 = m > 1 ? m : 1;
  double s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  double sabs = 0.0;
  int k = 0;
  double P = 0, M = 0, Pp = 0, Mp = 0;
  if (l0 <= lmax) start_spin_s(m, 1, Ks[m], g, P, M, k);
  for (int l = l0, cnt = 0; l <= lmax; ++l) {
    const double *t = &tab[4 * (l - l0)];
    const double cr = c[2 * l], ci = c[2 * l + 1];
    const double vp = k == 0 ? P : 0.0, vm = k == 0 ? M : 0.0;
    const bool odd = (l - l0) & 1;
    d1_accum(odd, vp, vm, cr, ci, s);
    // synth2_group with cp = c, cm = -c
    const double cpr = cr, cpi = ci, cmr = -cr, cmi = -ci;
    a[0] = fma(vp, cpr, a[0]); a[1] = fma(vp, cpi, a[1]);
    a[2] = fma(vm, cmr, a[2]); a[3] = fma(vm, cmi, a[3]);
    const double sg = odd ? -1.0 : 1.0;
    a[4] = fma(sg * vm, cpr, a[4]); a[5] = fma(sg * vm, cpi, a[5]);
    a[6] = fma(sg * vp, cmr, a[6]); a[7] = fma(sg * vp, cmi, a[7]);
    sabs += std::hypot(cr, ci) * (std::fabs(vp) + std::fabs(vm));
    double up = fma(t[0], g.cth, t[1]), um = fma(t[0], g.cth, -t[1]);
    double np_ = fma(up, P, -Pp), nm_ = fma(um, M, -Mp);
    Pp = P; P = np_; Mp = M; M = nm_;
    if (++cnt == 8) { cnt = 0; if (k < 0 && (needs_rescale(P) || needs_rescale(M))) { P *= SD; Pp *= SD; M *= SD; Mp *= SD; ++k; } }
  }
  const double sg0 = ((l0 + m) & 1) ? -0.5 : 0.5;
  double q[4], u[4];
  d1_combine(s, sg0, q, u);
  for (int i = 0; i < 4; ++i) { out_d1[i] = q[i]; out_d1[4 + i] = u[i]; }
  // synth2_kernel epilogue
  out_ref[0] = 0.5 * (a[0] + a[2]); out_ref[1] = 0.5 * (a[1] + a[3]);
  out_ref[2] = sg0 * (a[4] + a[6]); out_ref[3] = sg0 * (a[5] + a[7]);
  out_ref[4] = 0.5 * (a[1] - a[3]); out_ref[5] = -0.5 * (a[0] - a[2]);
  out_ref[6] = sg0 * (a[5] - a[7]); out_ref[7] = -sg0 * (a[4] - a[6]);
  out_abs[0] = sabs;
  return k;
}
