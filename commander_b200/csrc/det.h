// det.h -- indexing of the deterministic analysis (cmdr_sht_set_deterministic), shared by the Legendre and N_lm kernels,
// their ordered reduce and the pipelined launchers; plain C++ so that tests/host_emul/emul_det.cpp compiles it with g++.
//
// In deterministic mode an analysis warp does not add its per-tile sums to the a_lm with atomics.  It stores them into a
// partials buffer with one row of 2 (lmax + 1) doubles ({re, im} per l) per (component, warp block, local m), and records
// per (warp block, local m) the first l it stored.  A warp block is `32 R` consecutive work slots counted from slot 0 of
// the whole geometry (work index / 32 R), whatever slot range a launch covers, so that a slot belongs to the same block,
// and its ring to the same lane and register, in a whole-geometry launch and in every cut of it.  The reduce then sums,
// for each a_lm slot, the blocks in ascending block order starting from +0.0 and adds the sum once to the destination.
// Entries a warp did not store (l below its record, or a record of DET_EMPTY) count as exact zeros: adding +-0.0 to a sum
// that starts at +0.0 never changes it, so an unseeded warp that adds zeros for the rows before its first accumulating
// one gives the same bits as a seeded warp that starts there.
#pragma once
#include <cstddef>

#ifdef __CUDACC__
#define DET_HD __host__ __device__ __forceinline__
#else
#define DET_HD inline
#endif

namespace cmdr {

constexpr int DET_EMPTY = 0x7fffffff;   // record of a (block, m) that stored nothing

// Partials buffer of one launch: nb warp blocks (the whole geometry), nm local m's from im0, rows of 2 (lmax + 1) doubles
struct DetLayout {
  int nb = 0, nm = 0, im0 = 0, lmax = 0;
  DET_HD size_t row() const { return 2 * (size_t)(lmax + 1); }
  DET_HD size_t comp_stride() const { return (size_t)nb * nm * row(); }
  // {re, im} (part 0, 1) of l in the row of (component c, block b, local m im)
  DET_HD size_t index(int c, int b, int im, int l, int part) const {
    return (((size_t)c * nb + b) * nm + (im - im0)) * row() + 2 * (size_t)l + part;
  }
  DET_HD size_t rec_index(int b, int im) const { return (size_t)(im - im0) * nb + b; }
};

// a_lm index of (l, part) of local m (start mvs) written by the analysis kernels: real-packed (m = 0 has no imaginary
// part), complex, or the scalar-sum scratch of the spin-2 route ({re, im} of l at xofs + 2 l)
DET_HD long long det_dst_index(bool s2s, bool real_packed, int m, long long mvs, long long xofs, int l, int part) {
  return s2s ? xofs + 2 * (long long)l + part
             : real_packed ? (m == 0 ? mvs + l : mvs + 2 * (long long)l + part) : 2 * (mvs + l) + part;
}

// Sum over the nb blocks of one slot, in ascending block order; rec[b * rstride] is block b's record, part_at(b) its entry.
template <typename F>
DET_HD double det_sum(const int *rec, size_t rstride, int nb, int l, F part_at) {
  double s = 0.0;
  for (int b = 0; b < nb; ++b)
    if (l >= rec[(size_t)b * rstride]) s += part_at(b);
  return s;
}

// Cut of a pipelined launch over work slots [s0, s1) of an nslots-slot geometry to whole warp blocks of bs slots: a block
// that straddles two chunks goes with the later one, and the last chunk (by index, `last`, even when it is empty) takes
// every block from its start to nslots.  Every slot of the geometry then falls into exactly one launch when the chunks
// tile [0, nslots).
DET_HD void det_cut(int s0, int s1, bool last, int nslots, int bs, int &b, int &e) {
  b = s0 / bs * bs;
  e = last ? nslots : s1 / bs * bs;
  if (e < b) e = b;
}

}  // namespace cmdr
