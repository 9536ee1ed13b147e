// The argument checks of cmdr_cr_set_mixing_map (check_cr_mixing, commander_b200/csrc/cr_plan.h), compiled with g++ for
// the CPU test-suite.  TEST ONLY.
#include <cstdio>

#include "../../commander_b200/csrc/cr_plan.h"
using namespace cmdr;

// F_given = 0: F = NULL; else three column pointers of which `null_col` (if >= 0) is NULL.  Returns 1 when accepted, 0
// with the reason in err.
extern "C" int emul_cr_mix_check(int multi, int ncomp, int nbands, const int *comp_nmaps, const int *band_nmaps, int band,
                                 int comp, int F_given, int null_col, char *err, int errlen) {
  static const double one = 1.0;
  const double *cols[3] = {&one, &one, &one};
  if (null_col >= 0 && null_col < 3) cols[null_col] = nullptr;
  const std::string e = check_cr_mixing(multi != 0, ncomp, nbands, comp_nmaps, band_nmaps, band, comp, F_given ? cols : nullptr);
  snprintf(err, errlen, "%s", e.c_str());
  return e.empty() ? 1 : 0;
}
