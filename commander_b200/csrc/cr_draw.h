// cr_draw.h -- host side of the fluctuation terms drawn on the device (cr_draw.cu): the local -> global pixel table of a
// geometry and the argument checks of cmdr_cr_compute_rhs_draw.  Plain C++ (no CUDA) so that the CPU tests compile it
// with g++ (tests/host_emul/emul_rng.cpp).
#pragma once
#include <string>
#include <vector>

#include "conviqt_interp.cuh"
#include "sht_internal.h"

namespace cmdr {

// One local ring of a geometry: its first local pixel, its first global RING pixel, its pixel count.  The draw kernel runs
// one CTA per row, so a local pixel finds its global index without a search.
struct CrRing {
  long long loc, glob;
  int nph, pad;
};

// The rows of a geometry given by its ring list (1-based ring numbers in map storage order: local pixels follow the
// rings in that order, each ring's after the previous one's, as sharp_make_subset_healpix_geom_info lays them out)
inline std::vector<CrRing> cr_ring_table(int nside, const std::vector<int> &rings) {
  std::vector<CrRing> t;
  long long loc = 0;
  for (int r : rings) {
    const long long n = cvq_ring_npix(nside, r);
    t.push_back(CrRing{loc, cvq_ring_start(nside, r), (int)n, 0});
    loc += n;
  }
  return t;
}

// Checks the `terms` of cmdr_cr_compute_rhs_draw.  Returns the reason of a refusal, or an empty string.
inline std::string check_cr_draw(int terms) {
  if (terms < 0 || terms > (CMDR_CR_ETA_PIX | CMDR_CR_ETA_ALM))
    return "terms " + std::to_string(terms) + " out of range (0..3: CMDR_CR_ETA_PIX | CMDR_CR_ETA_ALM)";
  return "";
}

// The words every rank compares before a drawn right-hand side: seed and draw in 30-bit pieces (comm_all_equal compares
// non-negative ints exactly), then terms; all -1 when this rank's arguments were refused.
constexpr int CR_DRAW_WORDS = 7;
inline void cr_draw_words(unsigned long long seed, unsigned long long draw, int terms, bool ok, int w[CR_DRAW_WORDS]) {
  const unsigned long long v[2] = {seed, draw};
  for (int i = 0; i < 2; ++i)
    for (int k = 0; k < 3; ++k) w[3 * i + k] = (int)((v[i] >> (30 * k)) & 0x3fffffffULL);
  w[6] = terms;
  if (!ok)
    for (int i = 0; i < CR_DRAW_WORDS; ++i) w[i] = -1;
}

}  // namespace cmdr
