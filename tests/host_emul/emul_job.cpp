// The job resolution of the entry points (commander_b200/csrc/job.h), compiled with g++ for the CPU test-suite.  TEST ONLY.
#include <cstring>
#include "../../commander_b200/csrc/job.h"
using namespace cmdr;

// out: {spin, alm_cols, map_cols, synth, weighted, add, deriv1}.  Returns 1 for a valid job, 0 with the reason in `err`.
extern "C" int emul_resolve_job(int type, int spin, int flags, int iqu, int *out, char *err, int errlen) {
  const JobOrError r = resolve_job(type, spin, flags, iqu != 0);
  const Job &j = r.job;
  const int v[7] = {j.spin, j.alm_cols, j.map_cols, j.synth, j.weighted, j.add, j.deriv1};
  memcpy(out, v, sizeof(v));
  snprintf(err, errlen, "%s", r.error.c_str());
  return r.error.empty() ? 1 : 0;
}
