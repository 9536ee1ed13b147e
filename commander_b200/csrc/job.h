// job.h -- one transform job: what a (type, spin, flags) call runs, resolved and checked once by each entry point.
// Plain C++ (no CUDA) so that the CPU tests compile it with g++.
#pragma once
#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../include/cmdr_sht.h"

namespace cmdr {

constexpr int CMDR_MAX_SPIN = 32;   // start values use plain powers sh^(2s), ch^(2s): fine in FP64 up to here

// SHARP_ALM2MAP_DERIV1 is a synthesis from ONE spin-0 a_lm column to TWO maps {d_theta T, d_phi T / sin theta}; it runs on
// the spin-1 tables whatever spin the caller passes.
struct Job {
  int type = SHARP_Y;
  int spin = 0;                      // spin of the tables that run
  int alm_cols = 1, map_cols = 1;    // caller columns; map_cols is also the number of phase components
  bool synth = true;                 // a_lm -> map
  bool weighted = false;             // ring weights applied (SHARP_WY, SHARP_YtW)
  bool add = false;                  // SHARP_ADD: accumulate into the output
  bool deriv1 = false;               // SHARP_ALM2MAP_DERIV1
};

struct JobOrError {
  Job job;
  std::string error;                 // empty: `job` is valid
};

// The job of (type, spin, flags), or why the library does not run it.  `iqu`: the fused T + (Q,U) entry points, which
// run the four map <-> a_lm jobs only -- DERIV1 has one a_lm column and two maps per transform, which their
// three-column pointer tables cannot carry.
inline JobOrError resolve_job(int type, int spin, int flags, bool iqu = false) {
  JobOrError r;
  if (type < 0 || type > (iqu ? SHARP_WY : SHARP_ALM2MAP_DERIV1)) {
    r.error = "job type " + std::to_string(type) + " unsupported";
    return r;
  }
  Job &j = r.job;
  j.type = type;
  j.deriv1 = type == SHARP_ALM2MAP_DERIV1;
  j.spin = j.deriv1 ? 1 : spin;
  if (j.spin < 0 || j.spin > CMDR_MAX_SPIN) {
    r.error = "spin " + std::to_string(j.spin) + " unsupported (0.." + std::to_string(CMDR_MAX_SPIN) + ")";
    return r;
  }
  if (flags & SHARP_NO_FFT) {
    r.error = "SHARP_NO_FFT unsupported";
    return r;
  }
  j.synth = type == SHARP_Y || type == SHARP_WY || j.deriv1;
  j.weighted = type == SHARP_WY || type == SHARP_YtW;
  j.add = (flags & SHARP_ADD) != 0;
  j.alm_cols = j.deriv1 || j.spin == 0 ? 1 : 2;
  j.map_cols = j.deriv1 || j.spin != 0 ? 2 : 1;
  return r;
}

// resolve_job for an entry point of the library: prints the reason and aborts when the job is refused
inline Job job_or_abort(const char *who, int type, int spin, int flags, bool iqu = false) {
  JobOrError r = resolve_job(type, spin, flags, iqu);
  if (!r.error.empty()) { fprintf(stderr, "cmdr_sht: %s: %s\n", who, r.error.c_str()); abort(); }
  return r.job;
}

}  // namespace cmdr
