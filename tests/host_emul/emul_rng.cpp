// The draw stream of the constrained-realisation fluctuation terms (commander_b200/csrc/rng.cuh), the local -> global ring
// table and the argument checks of cmdr_cr_compute_rhs_draw (commander_b200/csrc/cr_draw.h), compiled with g++
// (-ffp-contract=off) for the CPU test-suite.  TEST ONLY.
#include <cstdio>
#include <cstring>
#include "../../commander_b200/csrc/cr_draw.h"
#include "../../commander_b200/csrc/rng.cuh"
using namespace cmdr;

// out[4 i .. 4 i + 3] = Philox4x32-10 of counter ctr[4 i .. 4 i + 3] and key (k0, k1)
extern "C" void emul_philox(long long n, const uint32_t *ctr, uint32_t k0, uint32_t k1, uint32_t *out) {
  for (long long i = 0; i < n; ++i) {
    const RngWords r = philox4x32_10(RngWords{ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3]}, k0, k1);
    out[4 * i] = r.x; out[4 * i + 1] = r.y; out[4 * i + 2] = r.z; out[4 * i + 3] = r.w;
  }
}

// out[i] = the Gaussian of the four words w[4 i .. 4 i + 3]
extern "C" void emul_gauss(long long n, const uint32_t *w, double *out) {
  for (long long i = 0; i < n; ++i) out[i] = rng_gauss(RngWords{w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]});
}

extern "C" void emul_eta_pix(unsigned long long seed, unsigned long long draw, unsigned q, unsigned j, long long n,
                             const uint32_t *pix, double *out) {
  for (long long i = 0; i < n; ++i) out[i] = rng_eta_pix(seed, draw, q, j, pix[i]);
}

extern "C" void emul_eta_alm(unsigned long long seed, unsigned long long draw, unsigned k, unsigned j, long long n, const int *l,
                             const int *ms, double *out) {
  for (long long i = 0; i < n; ++i) out[i] = rng_eta_alm(seed, draw, k, j, l[i], ms[i]);
}

// cr_ring_table of a ring list: row r into loc[r], glob[r], nph[r]; returns the number of rows
extern "C" int emul_ring_table(int nside, int nrings, const int *rings, long long *loc, long long *glob, int *nph) {
  const std::vector<CrRing> t = cr_ring_table(nside, std::vector<int>(rings, rings + nrings));
  for (size_t r = 0; r < t.size(); ++r) { loc[r] = t[r].loc; glob[r] = t[r].glob; nph[r] = t[r].nph; }
  return (int)t.size();
}

// check_cr_draw: 1 when accepted, 0 with the reason in `err`
extern "C" int emul_check_draw(int terms, char *err, int errlen) {
  const std::string e = check_cr_draw(terms);
  snprintf(err, errlen, "%s", e.c_str());
  return e.empty() ? 1 : 0;
}

extern "C" void emul_draw_words(unsigned long long seed, unsigned long long draw, int terms, int ok, int *w) {
  cr_draw_words(seed, draw, terms, ok != 0, w);
}
