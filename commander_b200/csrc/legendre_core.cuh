// legendre_core.cuh -- per-ring-pair Legendre / Wigner-d recurrence state shared by the
// synthesis and analysis kernels (and by the host emulation test, which compiles this
// header with a plain C++ compiler: CMDR_HD expands to nothing there).
//
// Replaces the Legendre stage inside libsharp2's sharp_execute, reached from
// commander3/src/sharp.f90:226-240 (SURVEY.md 8a rows a5-a9).  The only Legendre
// arithmetic physically in the reference is commander3/src/math_tools.f90:926-1028.
//
// Formulation (differs from both libsharp2 and the oracle on purpose -- it is the
// cheapest one in FP64 issue slots):
//   lambda_l = g_l * mu_l, where g is chosen so the three-term recurrence reads
//       mu_{l+1} = (A'_l x [+- C'_l]) mu_l - mu_{l-1}          (2 DFMA-pipe ops / l / function)
//   g_l is folded into the a_lm on load (synthesis) or on store (analysis).
//   Tiny values are carried as mu * 2^(SCALE_BITS*k), k<=0; a ring joins the
//   accumulation when k reaches 0, i.e. when |mu| >= 2^-THRESH_BITS.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define CMDR_HD __host__ __device__ __forceinline__
#else
#define CMDR_HD inline
#endif

namespace cmdr {

constexpr int SCALE_BITS = 512;    // one scale step
constexpr int THRESH_BITS = 70;    // accumulate once |mu| >= 2^-70 (libsharp2 starts at 2^-60, sharp_ftol; g_l = O(1..100) leaves margin)
// rescale when the biased exponent reaches (SCALE_BITS-THRESH_BITS)+1023
constexpr int RESCALE_EXP = SCALE_BITS - THRESH_BITS + 1023;

CMDR_HD int hi_word(double v) {
#ifdef __CUDA_ARCH__
  return __double2hiint(v);
#else
  union { double d; uint64_t u; } c; c.d = v; return (int)(c.u >> 32);
#endif
}
CMDR_HD double pow2i(int e) {   // 2^e for -1022 <= e <= 1023
#ifdef __CUDA_ARCH__
  return __hiloint2double((e + 1023) << 20, 0);
#else
  union { double d; uint64_t u; } c; c.u = (uint64_t)(e + 1023) << 52; return c.d;
#endif
}
CMDR_HD bool needs_rescale(double v) { return ((hi_word(v) >> 20) & 0x7ff) >= RESCALE_EXP; }

// base^n as mant * 2^ex with mant in [0.5,1);  0 < base <= 1, n >= 0.
CMDR_HD void pow_scaled(double base, int n, double &mant, int &ex) {
  int be;
  double bm = frexp(base, &be);
  double rm = 0.5; int re = 1;            // 1.0 = 0.5 * 2^1
  while (n) {
    if (n & 1) { rm *= bm; re += be; if (rm < 0.5) { rm *= 2.0; re -= 1; } }
    bm *= bm; be *= 2; if (bm < 0.5) { bm *= 2.0; be -= 1; }
    n >>= 1;
  }
  mant = rm; ex = re;
}

// Splits mant*2^ex (mant in [0.5,1)) into stored = mant*2^(ex-SCALE_BITS*k), k<=0.
CMDR_HD double split_scale(double mant, int ex, int &k) {
  int t = ex + THRESH_BITS;
  // floor division by SCALE_BITS (power of two) for negative t
  int kk = t >= 0 ? 0 : -((-t + SCALE_BITS - 1) / SCALE_BITS);
  k = kk;
  int e = ex - SCALE_BITS * kk;            // in [-THRESH_BITS, SCALE_BITS-THRESH_BITS) or >= -THRESH_BITS when kk==0
  return mant * pow2i(e);
}

// Per-ring geometry the kernels need.
struct RingTrig { double cth, sth, sh, ch; };   // cos/sin(theta), sin/cos(theta/2) of the NORTH ring

// ---- spin 0 --------------------------------------------------------------
// start: lambda_mm = K0[m] * sth^m      (K0 carries (-1)^m sqrt((2m+1)/4pi (2m-1)!!/(2m)!!))
CMDR_HD void start_spin0(int m, double K0m, const RingTrig &g, double &mu, int &k) {
  double mant; int ex;
  pow_scaled(g.sth, m, mant, ex);
  mu = K0m * split_scale(mant, ex, k);
}
// one step: returns mu_{l+1}
CMDR_HD double step0(double A, double x, double cur, double prev) {
  return fma(A * x, cur, -prev);
}

// one step of the two-l-per-step form (coef.cpp, fill_spin0_x2): returns nu_{j+1}; x2 = x^2
CMDR_HD double step0x2(double A, double B, double x2, double cur, double prev) {
  return fma(fma(A, x2, B), cur, -prev);
}

// ---- spin 2 --------------------------------------------------------------
// P = (+2)lambda_{l0,m}, M = (-2)lambda_{l0,m} at l0 = max(m,2).
//   m>=2: P = K2[m] sth^(m-2) sh^4 , M = K2[m] sth^(m-2) ch^4
//   m==0: P = M = c20 * sth^2 ;  m==1: P = -c21 ch sh^3, M = +c21 ch^3 sh
CMDR_HD void start_spin2(int m, double K2m, const RingTrig &g, double &P, double &M, int &k) {
  if (m >= 2) {
    double mant; int ex;
    pow_scaled(g.sth, m - 2, mant, ex);
    double base = K2m * split_scale(mant, ex, k);
    double s2 = g.sh * g.sh, c2 = g.ch * g.ch;
    P = base * (s2 * s2);
    M = base * (c2 * c2);
  } else if (m == 0) {
    k = 0;
    P = M = K2m * g.sth * g.sth;
  } else {
    k = 0;
    P = -K2m * g.ch * (g.sh * g.sh * g.sh);
    M = K2m * (g.ch * g.ch * g.ch) * g.sh;
  }
}

// ---- spin 2 seeded from the scalar recurrence ---------------------------------------------------------
// While every ring of a warp is still far below the accumulation threshold, the spin-2 kernels run the SCALAR
// two-l-per-step recurrence (1 FP64 op per l and ring pair instead of 4 for the two spin-2 recurrences) and convert at a
// group boundary with the classical relations between spin-2 and scalar harmonics (W_lm, X_lm of the polarisation
// literature; checked against the definitional Wigner-d sums in tests/test_host.py):
//   (+2)lam_l = W - X,  (-2)lam_l = W + X,   N = 1 / sqrt((l-1) l (l+1) (l+2)),  c = sqrt((2l+1)/(2l-1) (l-m)/(l+m))
//   W = 2N [ (-(l - m^2)/sin^2 - l(l-1)/2) lam_l + (l+m) (cos/sin^2) c lam_{l-1} ]
//   X = 2N (m/sin^2) [ (l-1) cos lam_l - (l+m) c lam_{l-1} ]
// Linear in the lambdas, so a common scale factor 2^(512 k) passes through.  The smaller of the two functions loses
// log2(large/small) bits (<= 11 for the rings and m this path is used for, i.e. relative errors <= 1e-11 on a function
// that is itself that much smaller than its partner).
CMDR_HD void spin2_from_scalar(int l, int m, double x, double sth, double lam, double lam1, double &P, double &M) {
  const double dl = l, dm = m;
  const double N = 1.0 / sqrt((dl - 1.0) * dl * (dl + 1.0) * (dl + 2.0));
  const double c = sqrt((2.0 * dl + 1.0) / (2.0 * dl - 1.0) * (dl - dm) / (dl + dm));
  const double f = 2.0 * N / (sth * sth);
  const double a = -(dl - dm * dm) - 0.5 * dl * (dl - 1.0) * sth * sth;
  const double b = dm * (dl - 1.0) * x, e = (dl + dm) * c;
  P = f * ((a - b) * lam + e * (x + dm) * lam1);
  M = f * ((a + b) * lam + e * (x - dm) * lam1);
}
// The same relations as a banded map onto the scalar functions (spin-2 Legendre sums run as scalar sums).  With
// S_l = ((+2)lam_l + (-2)lam_l) / 2, A_l = ((+2)lam_l - (-2)lam_l) / 2, the W/X form above and the three-term relation
// x lam_k = eps_{k+1} lam_{k+1} + eps_k lam_{k-1} (eps_k = sqrt((k^2 - m^2) / (4k^2 - 1)); e = (2l+1) eps_l above):
//   sin^2 S_l = kS[0] lam_{l-2} + kS[1] lam_l + kS[2] lam_{l+2},    sin^2 A_l = kA[0] lam_{l-1} + kA[1] lam_{l+1}
//   F = 2 / sqrt((l-1) l (l+1) (l+2)),  kS[0] = F (l+1)(l+2)/2 eps_l eps_{l-1},  kS[2] = F l(l-1)/2 eps_{l+1} eps_{l+2},
//   kS[1] = F [-(l - m^2) - l(l-1)/2 + l(l-1)/2 (eps_{l+1}^2 + eps_l^2) + (2l+1) eps_l^2],
//   kA[0] = F m (l+2) eps_l,  kA[1] = -F m (l-1) eps_{l+1}                                                (l >= 2)
// The identity is polynomial in x = cos(theta), so it holds on the southern mirror too; the 1/sin^2 it leaves costs
// digits near the poles only: ring pairs with sin(theta) < S2S_MIN_STH stay on the spin-2 recurrences.
constexpr double S2S_MIN_STH = 0.05;
CMDR_HD double s2s_eps(int l, int m) {
  const double dl = l, dm = m;
  return l > m ? sqrt((dl * dl - dm * dm) / (4.0 * dl * dl - 1.0)) : 0.0;
}
CMDR_HD void s2s_coefs(int l, int m, double (&kS)[3], double (&kA)[2]) {
  const double dl = l, dm = m;
  const double F = 2.0 / sqrt((dl - 1.0) * dl * (dl + 1.0) * (dl + 2.0));
  const double e0 = s2s_eps(l, m), em = s2s_eps(l - 1, m), e1 = s2s_eps(l + 1, m), e2 = s2s_eps(l + 2, m);
  const double h = 0.5 * dl * (dl - 1.0);
  kS[0] = F * 0.5 * (dl + 1.0) * (dl + 2.0) * e0 * em;
  kS[1] = F * (-(dl - dm * dm) - h + h * (e1 * e1 + e0 * e0) + (2.0 * dl + 1.0) * e0 * e0);
  kS[2] = F * h * e1 * e2;
  kA[0] = F * dm * (dl + 2.0) * e0;
  kA[1] = -F * dm * (dl - 1.0) * e1;
}
// Synthesis of spin 2 (E, B of one l, after the per-l factor and the real-packed norm ns) as the two scalar sequences
// of the map components (Q: dq, U: du) on the slots l-2 .. l+2 (index 0 .. 4), in the combination of synth2_kernel:
//   Q = -sum_l [E_l S_l + i B_l A_l],  U = -sum_l [B_l S_l - i E_l A_l]   (north; the south is the same at -x).
// d[c][i] += {re, im}.
CMDR_HD void s2s_scatter(int l, int m, double er, double ei, double br, double bi, double (&d)[2][5][2]) {
  double kS[3], kA[2];
  s2s_coefs(l, m, kS, kA);
  // S coefficients: Q -E, U -B ; A coefficients: Q -iB = (bi, -br), U +iE = (-ei, er)
  for (int t = 0; t < 3; ++t) {
    d[0][2 * t][0] -= kS[t] * er; d[0][2 * t][1] -= kS[t] * ei;
    d[1][2 * t][0] -= kS[t] * br; d[1][2 * t][1] -= kS[t] * bi;
  }
  for (int t = 0; t < 2; ++t) {
    d[0][2 * t + 1][0] += kA[t] * bi; d[0][2 * t + 1][1] -= kA[t] * br;
    d[1][2 * t + 1][0] -= kA[t] * ei; d[1][2 * t + 1][1] += kA[t] * er;
  }
}
// Its exact transpose for analysis: from the scalar sums Tq_{l+i-2}, Tu_{l+i-2} (i = 0 .. 4; {re, im}) to
//   E_l = -[sum kS Tq + i sum kA Tu],  B_l = -sum kS Tu + i sum kA Tq      (before the real-packed norm and the per-l factor)
CMDR_HD void s2s_gather(int l, int m, const double (&tq)[5][2], const double (&tu)[5][2], double &er, double &ei, double &br,
                        double &bi) {
  double kS[3], kA[2];
  s2s_coefs(l, m, kS, kA);
  double sq[2] = {0.0, 0.0}, su[2] = {0.0, 0.0}, aq[2] = {0.0, 0.0}, au[2] = {0.0, 0.0};
  for (int t = 0; t < 3; ++t)
    for (int c = 0; c < 2; ++c) { sq[c] = fma(kS[t], tq[2 * t][c], sq[c]); su[c] = fma(kS[t], tu[2 * t][c], su[c]); }
  for (int t = 0; t < 2; ++t)
    for (int c = 0; c < 2; ++c) { aq[c] = fma(kA[t], tq[2 * t + 1][c], aq[c]); au[c] = fma(kA[t], tu[2 * t + 1][c], au[c]); }
  er = -(sq[0] - au[1]); ei = -(sq[1] + au[0]);
  br = -su[0] - aq[1];   bi = -su[1] + aq[0];
}

// switch from the scalar to the spin-2 recurrences once a ring's scalar value (stored as true * 2^(-512 k)) is within
// `margin` bits of the accumulation threshold.  The spin-2 functions are larger than the scalar one by at most
// ~2 / sin^2(theta) (the m^2 / sin^2 term of W with m <= l), and a few bits of growth until the next check are allowed for.
CMDR_HD int front_margin_bits(double sth) {
  const int e2 = ((hi_word(sth * sth) >> 20) & 0x7ff) - 1023;   // floor(log2 sin^2): <= 0
  return 8 - e2;
}
CMDR_HD bool front_must_switch(double cur, int k, int margin) {
  return k >= 0 || (k == -1 && ((hi_word(cur) >> 20) & 0x7ff) >= RESCALE_EXP - margin);
}
// State of the spin-2 recurrences at l_b = m + 2 jb (m >= 2) from the scalar state (nu_jb, nu_{jb-1}):
//   mixb = mix row jb {u, v, h, v_{jb-1}}, hprev = h_{jb-1};  c0 / c1 = spin-2 coefficient rows {A', C', g, .} of l_b, l_b + 1.
// Returns mu(l_b) in P / M and mu(l_b - 1) in Pp / Mp (kernel normalisation lam = g mu), same scale factor as nu.
CMDR_HD void spin2_front_convert(int lb, int m, int lmax, double x, double sth, double nu, double nup, const double *mixb, double hprev,
                                 const double *c0, const double *c1, double &P, double &Pp, double &M, double &Mp) {
  const double lam_m1 = x * hprev * nup;                       // lam(l_b - 1)
  const double lam_0 = mixb[0] * nu + mixb[3] * nup;           // lam(l_b)
  const double lam_p1 = x * mixb[2] * nu;                      // lam(l_b + 1)
  double P0, M0, P1 = 0.0, M1 = 0.0;
  spin2_from_scalar(lb, m, x, sth, lam_0, lam_m1, P0, M0);
  P = P0 / c0[2]; M = M0 / c0[2];
  Pp = 0.0; Mp = 0.0;
  if (lb + 1 <= lmax) {
    spin2_from_scalar(lb + 1, m, x, sth, lam_p1, lam_0, P1, M1);
    // mu_{l+1} = (A' x +- C') mu_l - mu_{l-1}  =>  mu_{l-1} = (A' x +- C') mu_l - mu_{l+1}
    Pp = fma(fma(c0[0], x, c0[1]), P, -P1 / c1[2]);
    Mp = fma(fma(c0[0], x, -c0[1]), M, -M1 / c1[2]);
  }
}

// ---- arbitrary spin s >= 1 (conviqt: commander3/src/comm_conviqt_mod.f90:234-239) ---------------
CMDR_HD double ipow(double b, int n) {      // b^n, n >= 0, by repeated squaring
  double r = 1.0;
  while (n) { if (n & 1) r *= b; b *= b; n >>= 1; }
  return r;
}
// P = (+s)lambda_{l0,m}, M = (-s)lambda_{l0,m} at l0 = max(m,s); Ksm from build_start_norms_spin.
// (+-s)lambda_lm(theta) = (-1)^m sqrt((2l+1)/4pi) d^l_{-m,+-s}(theta)   (Goldberg et al. 1967)
CMDR_HD void start_spin_s(int m, int s, double Ksm, const RingTrig &g, double &P, double &M, int &k) {
  if (m >= s) {
    double mant; int ex;
    pow_scaled(g.sth, m - s, mant, ex);
    double base = Ksm * split_scale(mant, ex, k);
    P = base * ipow(g.sh, 2 * s);
    M = base * ipow(g.ch, 2 * s);
    // k was chosen from sin^(m-s) alone; Ksm (which carries 2^s) can lift the start values over the threshold.  Join
    // now: the recurrences only check every 8 l, and with lmax - m < 8 they would never do it.
    if (k < 0 && (needs_rescale(P) || needs_rescale(M))) { P *= pow2i(-SCALE_BITS); M *= pow2i(-SCALE_BITS); ++k; }
  } else {
    k = 0;
    P = Ksm * ipow(g.ch, s - m) * ipow(g.sh, s + m);
    M = (((s - m) & 1) ? -Ksm : Ksm) * ipow(g.ch, s + m) * ipow(g.sh, s - m);
  }
}

// ---- SHARP_ALM2MAP_DERIV1: gradient of a spin-0 map through the spin-1 functions ---------------------------
// d_theta T = spin-1 synthesis with E = -sqrt(l(l+1)) a, B = 0, so both spin-1 coefficients are multiples of one
// number c_l: cp = c, cm = -c.  The four phase sums of the spin-s kernels (north: sum cp P, sum cm M; south:
// sum sg cp M, sum sg cm P, sg = (-1)^(l - l0) relative to l0) then follow from sum c P and sum c M, each split by
// the parity of l - l0.  s[0..1] = even c P, s[2..3] = even c M, s[4..5] = odd c P, s[6..7] = odd c M (re, im):
// 4 accumulate FMAs per l and ring pair instead of 8.
CMDR_HD void d1_accum(bool odd, double P, double M, double cr, double ci, double (&s)[8]) {
  if (odd) { s[4] = fma(P, cr, s[4]); s[5] = fma(P, ci, s[5]); s[6] = fma(M, cr, s[6]); s[7] = fma(M, ci, s[7]); }
  else     { s[0] = fma(P, cr, s[0]); s[1] = fma(P, ci, s[1]); s[2] = fma(M, cr, s[2]); s[3] = fma(M, ci, s[3]); }
}
// Phases {N.re, N.im, S.re, S.im} of the two map components from the parity sums, in the combination of the spin-s
// synthesis epilogue (a1 = sum cp P, a2 = sum cm M, a3 = sum sg cp M, a4 = sum sg cm P; Q = (a1 + a2)/2,
// U = -i (a1 - a2)/2, south with sg0 = (-1)^(l0 + m) / 2).
CMDR_HD void d1_combine(const double (&s)[8], double sg0, double (&q)[4], double (&u)[4]) {
  const double a1r = s[0] + s[4], a1i = s[1] + s[5];
  const double a2r = -(s[2] + s[6]), a2i = -(s[3] + s[7]);
  const double a3r = s[2] - s[6], a3i = s[3] - s[7];
  const double a4r = s[4] - s[0], a4i = s[5] - s[1];
  q[0] = 0.5 * (a1r + a2r); q[1] = 0.5 * (a1i + a2i);
  u[0] = 0.5 * (a1i - a2i); u[1] = -0.5 * (a1r - a2r);
  q[2] = sg0 * (a3r + a4r); q[3] = sg0 * (a3i + a4i);
  u[2] = sg0 * (a3i - a4i); u[3] = -sg0 * (a3r - a4r);
}

// libsharp-style per-ring m cut-off (contributions above it are far below FP64
// resolution).  Same form as the oracle's get_mlim.
inline int mlim_for_ring(int lmax, int spin, double sth, double cth) {
  double ofs = lmax * 0.01; if (ofs < 100.) ofs = 100.;
  double b = -2 * spin * fabs(cth);
  double t1 = lmax * sth + ofs;
  double c = (double)spin * spin - t1 * t1;
  double discr = b * b - 4 * c;
  if (discr <= 0) return lmax;
  double res = (-b + sqrt(discr)) / 2.;
  if (res > lmax) res = lmax;
  return (int)(res + 0.5);
}

}  // namespace cmdr
