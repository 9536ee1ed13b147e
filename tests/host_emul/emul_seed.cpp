// Host emulation of the seed tables of the spin-0 Legendre kernels (legendre.cu: seed0_kernel, synth0_kernel), compiled
// with g++ for the CPU test-suite.  TEST ONLY.  One warp of `n` ring pairs (north ring indices, -1 = invalid slot) runs
//   unseeded: closed-form start values at row 0, groups of 4 rows, the kernel's warp-uniform choice between "all on",
//             "none on" and the predicated mode (invalid slots count as on, as in the kernel), synthesis sums per ring;
//   seeded:   the seed loop up to the first group at which a VALID ring is on, then the same group loop from there.
// Returns the seeded start row; `same` is set when every ring's sums and final recurrence state agree bit for bit.
#include <cmath>
#include <cstring>
#include <vector>
#include "../../commander_b200/csrc/legendre_core.cuh"
#include "../../commander_b200/csrc/sht_internal.h"
using namespace cmdr;

namespace {
struct Ring { bool valid; double x2, cur, prev; int k; double s[4]; };

RingTrig trig(int nside, int north) {
  long double omc, ns = nside;
  if (north < nside) omc = (long double)north * north / (3.0L * ns * ns);
  else omc = 1.0L - (2.0L * ns - north) * 2.0L / (3.0L * ns);
  return RingTrig{(double)(1.0L - omc), (double)sqrtl(omc * (2.0L - omc)), (double)sqrtl(0.5L * omc), (double)sqrtl(1.0L - 0.5L * omc)};
}

// groups of 4 rows from row j0 to J as synth0_group runs them, with a fixed pseudo a_lm combination c per row
void groups(std::vector<Ring> &w, const double *rec, int j0, int J, bool accumulate) {
  const double SD = ldexp(1.0, -SCALE_BITS);
  for (int j = j0; j < J; j += 4) {
    bool all_on = true, none_on = true;
    for (auto &r : w) { all_on &= r.k == 0; none_on &= r.k < 0; }
    const int mode = all_on ? 2 : (none_on ? 0 : 1);
    for (int q = 0; q < 4; ++q) {
      const double c[4] = {std::sin(1.0 + j + q), std::cos(2.0 + j + q), std::sin(3.0 * (j + q)), std::cos(0.5 * (j + q))};
      for (auto &r : w) {
        if (accumulate && mode >= 1) {
          const double v = (mode == 2 || r.k == 0) ? r.cur : 0.0;
          for (int i = 0; i < 4; ++i) r.s[i] = std::fma(v, c[i], r.s[i]);
        }
        const double nxt = step0x2(rec[2 * (j + q)], rec[2 * (j + q) + 1], r.x2, r.cur, r.prev);
        r.prev = r.cur; r.cur = nxt;
      }
    }
    if (mode < 2)
      for (auto &r : w)
        if (r.k < 0 && needs_rescale(r.cur)) { r.cur *= SD; r.prev *= SD; ++r.k; }
  }
}
}  // namespace

extern "C" int emul_seed0(int nside, int lmax, int m, int n, const int *north, int *same) {
  std::vector<int> mval{m};
  std::vector<double> rec, mix; std::vector<long long> ofs;
  build_coef_table_x2(lmax, mval, rec, mix, ofs);
  rec.resize(rec.size() + 8, 0.0);   // the device table is zero padded past the last row
  std::vector<double> K0, K2;
  build_start_norms(m, K0, K2);
  const int J = (lmax - m) / 2 + 1;
  std::vector<Ring> w(n);
  for (int i = 0; i < n; ++i) {
    Ring &r = w[i];
    std::memset(&r, 0, sizeof r);
    r.valid = north[i] > 0;
    if (r.valid) { const RingTrig g = trig(nside, north[i]); r.x2 = g.cth * g.cth; start_spin0(m, K0[m], g, r.cur, r.k); }
  }
  std::vector<Ring> ref = w;
  groups(ref, rec.data(), 0, J, true);
  // seed loop (seed0_kernel): stop at the first group at which a valid ring is on
  int j0 = 0;
  for (; j0 < J; j0 += 4) {
    bool on = false;
    for (auto &r : w) on |= r.valid && r.k == 0;
    if (on) break;
    groups(w, rec.data(), j0, j0 + 4, false);
  }
  groups(w, rec.data(), j0, J, true);
  bool eq = true;
  for (int i = 0; i < n; ++i)
    eq &= std::memcmp(w[i].s, ref[i].s, sizeof w[i].s) == 0 && std::memcmp(&w[i].cur, &ref[i].cur, sizeof(double)) == 0 &&
          w[i].k == ref[i].k;
  *same = eq ? 1 : 0;
  return j0;
}
