// Host emulation of spin 2 as scalar sums (legendre_core.cuh: s2s_coefs / s2s_scatter / s2s_gather; legendre.cu:
// prep_s2s_kernel, post_s2s_kernel), compiled with g++ for the CPU test-suite.  TEST ONLY.
//
// emul_s2s_synth: the north and south phases {Q, U} of one (m, ring) from E_l, B_l (complex, l = 0..lmax, real-packed
//   norm included by the caller) two ways:
//   direct: the spin-2 recurrences of synth2_kernel (coef.cpp tables, start values of start_spin2) in long double and
//           its combination Q = (a1 + a2) / 2, U = -i (a1 - a2) / 2 with cp = -(E + iB), cm = -(E - iB);
//   route:  the scalar sequences d = s2s_scatter(E, B) up to lmax + 2 (double, as the prep kernel forms them), the scalar
//           functions lam_l (long double recurrence, rounded to double as the kernels carry them), the sums in double
//           and the factor 1 / sin^2.
//   out[0..7] = direct {QN, UN, QS, US} (re, im), out[8..15] = route.
// emul_s2s_adjoint: <D a, t> and <a, D^T t> for a = (E, B) and t = (Tq, Tu) as real vectors.
#include <cmath>
#include <complex>
#include <vector>
#include "../../commander_b200/csrc/legendre_core.cuh"
#include "../../commander_b200/csrc/sht_internal.h"
using namespace cmdr;
typedef long double LD;
typedef std::complex<LD> CL;

namespace {
struct Trig { LD cth, sth, sh, ch; };
Trig ring_trig(int nside, int north) {
  LD omc, ns = nside;
  if (north < nside) omc = (LD)north * north / (3.0L * ns * ns);
  else omc = 1.0L - (2.0L * ns - north) * 2.0L / (3.0L * ns);
  return Trig{1.0L - omc, sqrtl(omc * (2.0L - omc)), sqrtl(0.5L * omc), sqrtl(1.0L - 0.5L * omc)};
}

// direct spin-2 sums at (x, sth, sh, ch): returns {Q, U}
void direct(int lmax, int m, const Trig &t, const std::vector<double> &tab, LD K2, const double *E, const double *B, CL &Q, CL &U) {
  const int l0 = m > 2 ? m : 2;
  LD P, M;
  if (m >= 2) { LD b = K2 * powl(t.sth, m - 2); P = b * powl(t.sh, 4); M = b * powl(t.ch, 4); }
  else if (m == 0) { P = M = K2 * t.sth * t.sth; }
  else { P = -K2 * t.ch * t.sh * t.sh * t.sh; M = K2 * t.ch * t.ch * t.ch * t.sh; }
  LD Pp = 0, Mp = 0;
  CL a1 = 0, a2 = 0;
  for (int l = l0; l <= lmax; ++l) {
    const double *c = tab.data() + 4 * (size_t)(l - l0);   // {A', C', g, 0}
    const CL e(E[2 * l], E[2 * l + 1]), b(B[2 * l], B[2 * l + 1]), I(0, 1);
    a1 += -(e + I * b) * ((LD)c[2] * P);
    a2 += -(e - I * b) * ((LD)c[2] * M);
    const LD np = ((LD)c[0] * t.cth + (LD)c[1]) * P - Pp, nm = ((LD)c[0] * t.cth - (LD)c[1]) * M - Mp;
    Pp = P; P = np; Mp = M; M = nm;
  }
  Q = 0.5L * (a1 + a2);
  U = CL(0, -0.5L) * (a1 - a2);
}

// scalar route at x: sum d lam / sin^2, lam from the long double recurrence rounded to double, sums in double
void route(int lmax, int m, const Trig &t, LD K0, const std::vector<double> &d, std::complex<double> &Q, std::complex<double> &U) {
  LD lp = 0, lc = K0 * powl(t.sth, m);
  std::complex<double> sq = 0, su = 0;
  for (int l = m; l <= lmax + 2; ++l) {
    const double lam = (double)lc;
    const size_t o = 4 * (size_t)(l - m);
    sq += std::complex<double>(d[o], d[o + 1]) * lam;
    su += std::complex<double>(d[o + 2], d[o + 3]) * lam;
    const LD e1 = sqrtl(((LD)(l + 1) * (l + 1) - (LD)m * m) / (4.0L * (l + 1) * (l + 1) - 1.0L));
    const LD e0 = l > m ? sqrtl(((LD)l * l - (LD)m * m) / (4.0L * l * l - 1.0L)) : 0.0L;
    const LD nx = (t.cth * lc - e0 * lp) / e1;
    lp = lc; lc = nx;
  }
  const double s = (double)t.sth, f = 1.0 / (s * s);
  Q = sq * f; U = su * f;
}

// d (per l' = m .. lmax + 2: {Q re, Q im, U re, U im}) as prep_s2s_kernel forms it
std::vector<double> premix(int lmax, int m, const double *E, const double *B) {
  std::vector<double> d(4 * (size_t)(lmax + 3 - m), 0.0);
  for (int l = m > 2 ? m : 2; l <= lmax; ++l) {
    double s[2][5][2] = {};
    s2s_scatter(l, m, E[2 * l], E[2 * l + 1], B[2 * l], B[2 * l + 1], s);
    for (int i = 0; i < 5; ++i) {
      const int t = l - 2 + i;
      if (t < m) continue;
      for (int c = 0; c < 2; ++c)
        for (int q = 0; q < 2; ++q) d[4 * (size_t)(t - m) + 2 * c + q] += s[c][i][q];
    }
  }
  return d;
}
}  // namespace

extern "C" void emul_s2s_synth(int nside, int lmax, int m, int north, const double *E, const double *B, double *out) {
  std::vector<int> mval{m};
  std::vector<double> tab; std::vector<long long> ofs;
  build_coef_table(lmax, 2, mval, tab, ofs);
  std::vector<double> K0, K2;
  build_start_norms(m, K0, K2);
  const Trig tn = ring_trig(nside, north), ts{-tn.cth, tn.sth, tn.ch, tn.sh};   // the southern mirror
  const std::vector<double> d = premix(lmax, m, E, B);
  int k = 0;
  for (const Trig *t : {&tn, &ts}) {
    CL Q, U;
    direct(lmax, m, *t, tab, K2[m], E, B, Q, U);
    out[k] = (double)Q.real(); out[k + 1] = (double)Q.imag(); out[k + 2] = (double)U.real(); out[k + 3] = (double)U.imag();
    std::complex<double> q, u;
    route(lmax, m, *t, K0[m], d, q, u);
    out[8 + k] = q.real(); out[9 + k] = q.imag(); out[10 + k] = u.real(); out[11 + k] = u.imag();
    k += 4;
  }
}

// E, B: 2 (lmax + 1) doubles each; T: 4 (lmax + 3 - m) doubles ({Tq re, Tq im, Tu re, Tu im} per l' = m .. lmax + 2)
extern "C" void emul_s2s_adjoint(int lmax, int m, const double *E, const double *B, const double *T, double *out) {
  const std::vector<double> d = premix(lmax, m, E, B);
  LD fwd = 0, adj = 0;
  for (size_t i = 0; i < d.size(); ++i) fwd += (LD)d[i] * T[i];
  for (int l = m > 2 ? m : 2; l <= lmax; ++l) {
    double tq[5][2], tu[5][2];
    for (int i = 0; i < 5; ++i) {
      const int t = l - 2 + i;
      const bool ok = t >= m;
      for (int q = 0; q < 2; ++q) {
        tq[i][q] = ok ? T[4 * (size_t)(t - m) + q] : 0.0;
        tu[i][q] = ok ? T[4 * (size_t)(t - m) + 2 + q] : 0.0;
      }
    }
    double er, ei, br, bi;
    s2s_gather(l, m, tq, tu, er, ei, br, bi);
    adj += (LD)er * E[2 * l] + (LD)ei * E[2 * l + 1] + (LD)br * B[2 * l] + (LD)bi * B[2 * l + 1];
  }
  out[0] = (double)fwd; out[1] = (double)adj;
}
