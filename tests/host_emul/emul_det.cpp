// Host emulation of the deterministic analysis indexing (commander_b200/csrc/det.h), compiled with g++ by
// tests/test_det_cpu.py: the partials slots the kernels store, the order in which the reduce reads them, and the cut of
// pipelined launches on warp blocks.
#include <cstring>
#include <vector>

#include "../../commander_b200/csrc/det.h"

using namespace cmdr;

extern "C" {

// One launch of nslots work slots over local m's mval[0..nm) (starts mvstart, real-packed or complex), l0 = max(m, spin),
// blocks of bs slots.  first[b * nm + im]: the first l block b stores for m (DET_EMPTY: nothing), as the kernels record
// it.  Stores every (component, block, m, l >= first, part) entry the kernels store, then reduces every destination
// slot with det_sum and checks: each stored entry is read exactly once, by the slot of its (m, l, part); no entry that
// was not stored is read; blocks are read in ascending order; destination indices are distinct and inside [0, ndst).
// Returns 0, or a code naming the first failed check.
int emul_det_check(int nslots, int bs, int nm, const int *mval, const long long *mvstart, int real_packed, int s2s,
                   int lmax, int spin, int ncomp, const int *first, long long ndst) {
  DetLayout d;
  d.nb = (nslots + bs - 1) / bs; d.nm = nm; d.im0 = 0; d.lmax = lmax;
  const size_t n = d.comp_stride() * ncomp;
  std::vector<int> stored(n, 0), read(n, 0), rec((size_t)d.nb * nm);
  std::vector<int> dst_hits(ndst > 0 ? ndst : 1, 0);
  for (int b = 0; b < d.nb; ++b)
    for (int im = 0; im < nm; ++im) rec[d.rec_index(b, im)] = first[(size_t)b * nm + im];
  long long cofs = 0;   // s2s scratch: {re, im} of l at 2 (cofs + l - m), cofs the two-l-per-step table offsets (doubles)
  for (int im = 0; im < nm; ++im) {
    const int m = mval[im], l0 = m > spin ? m : spin;
    for (int b = 0; b < d.nb; ++b) {
      const int f = rec[d.rec_index(b, im)];
      if (f == DET_EMPTY) continue;
      for (int l = f; l <= lmax; ++l)
        for (int part = 0; part < 2; ++part) {
          if (m == 0 && part) continue;
          for (int c = 0; c < ncomp; ++c) {
            const size_t i = d.index(c, b, im, l, part);
            if (i >= n) return 1;
            if (stored[i]++) return 2;
          }
        }
    }
    const long long xofs = 2 * (cofs - m);
    for (int l = l0; l <= lmax; ++l)
      for (int part = 0; part < 2; ++part) {
        if (m == 0 && part) continue;
        const long long di = det_dst_index(s2s, real_packed, m, mvstart[im], xofs, l, part);
        if (di < 0 || di >= ndst) return 3;
        if (dst_hits[di]++) return 4;
        for (int c = 0; c < ncomp; ++c) {
          const size_t base = d.index(c, 0, im, l, part), bstride = (size_t)d.nm * d.row();
          int last = -1;
          bool order_ok = true;
          det_sum(&rec[d.rec_index(0, im)], 1, d.nb, l, [&](int b) {
            if (b <= last) order_ok = false;
            last = b;
            read[base + (size_t)b * bstride]++;
            return 0.0;
          });
          if (!order_ok) return 5;
        }
      }
    cofs += 2 * ((lmax - m) / 2 + 1);
  }
  for (size_t i = 0; i < n; ++i)
    if (read[i] != stored[i]) return stored[i] ? 6 : 7;
  return 0;
}

// The launches of a pipelined analysis over chunk cuts wcut[0..nch] (wcut[0] = 0, wcut[nch] = nslots): owner[s] = the
// launch (chunk) whose det_cut range holds slot s (-1: none, -2: more than one); begin / end of each launch.
void emul_det_cut(int nslots, int bs, int nch, const int *wcut, int *owner, int *begin, int *end) {
  for (int s = 0; s < nslots; ++s) owner[s] = -1;
  for (int c = 0; c < nch; ++c) {
    det_cut(wcut[c], wcut[c + 1], c == nch - 1, nslots, bs, begin[c], end[c]);
    for (int s = begin[c]; s < end[c]; ++s) owner[s] = owner[s] == -1 ? c : -2;
  }
}

}  // extern "C"
