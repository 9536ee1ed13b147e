// The per-sample psi lookup and the table placement of the conviqt sampler (commander_b200/csrc/conviqt_interp.cuh),
// compiled with g++ (-ffp-contract=off) for the CPU test-suite.  TEST ONLY.
#include <cstdio>
#include <cstring>
#include "../../commander_b200/csrc/conviqt_interp.cuh"
using namespace cmdr;

// out[i] = what conviqt_interp_kernel computes for sample i of the table tab[2 bmax][npix]
extern "C" void emul_conviqt_interp(const float *tab, long long npix, int bmax, int optim, long long n, const int *pix,
                                    const float *psi, float *out) {
  const int psisteps = 2 * bmax;
  const float psires = cvq_psires(psisteps), twopi = cvq_twopi();
  for (long long i = 0; i < n; ++i) out[i] = conviqt_interp_sample(tab, npix, psisteps, psires, twopi, optim, pix[i], psi[i]);
}

extern "C" float emul_conviqt_psires(int psisteps) { return cvq_psires(psisteps); }

static std::vector<std::vector<int>> split(int nranks, const int *nrings, const int *rings) {
  std::vector<std::vector<int>> rr(nranks);
  for (int r = 0, k = 0; r < nranks; ++r)
    for (int i = 0; i < nrings[r]; ++i) rr[r].push_back(rings[k++]);
  return rr;
}

// cvq_check_rings over the ranks' ring lists (concatenated); returns 1 when accepted, 0 with the reason in `err`
extern "C" int emul_conviqt_check_rings(int nside, int nranks, const int *nrings, const int *rings, int whole, char *err,
                                        int errlen) {
  const std::string e = cvq_check_rings(nside, split(nranks, nrings, rings), whole != 0);
  snprintf(err, errlen, "%s", e.c_str());
  return e.empty() ? 1 : 0;
}

// The all-gather + scatter of the sampler on one table row: rank r's local pixel i sits at r * stride + i of the gathered
// buffer; the runs move it to the table.  owner[p] / local[p] receive the rank and local index that landed in global pixel p
// (-1 where none did).  Returns the number of runs.
extern "C" long long emul_conviqt_scatter(int nside, int nranks, const int *nrings, const int *rings, long long stride,
                                          int *owner, long long *local) {
  const long long npix = 12LL * nside * nside;
  for (long long p = 0; p < npix; ++p) { owner[p] = -1; local[p] = -1; }
  const std::vector<CvqRun> runs = cvq_scatter_runs(nside, split(nranks, nrings, rings), stride);
  for (const CvqRun &r : runs)
    for (int j = 0; j < r.n; ++j) {
      owner[r.dst + j] = (int)((r.src + j) / stride);
      local[r.dst + j] = (r.src + j) % stride;
    }
  return (long long)runs.size();
}
