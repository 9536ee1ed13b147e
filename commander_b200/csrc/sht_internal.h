// sht_internal.h -- internal types of libcmdr_sht (not part of the ABI).
#pragma once
#include <cstddef>
#include <cstdint>
#include <map>
#include <vector>

#include "../../include/cmdr_sht.h"

namespace cmdr {

// ---- host-side table builders (coef.cpp)
void build_coef_table(int lmax, int spin, const std::vector<int> &mval, std::vector<double> &tab,
                      std::vector<long long> &ofs);
// spin 0 in steps of two l (x^2 recurrence, coef.cpp): rec rows {a_j, b'_j} (ofs in doubles, 2 per row), mix rows {u_j, v_j, h_j, v_{j-1}}
void build_coef_table_x2(int lmax, const std::vector<int> &mval, std::vector<double> &rec, std::vector<double> &mix,
                         std::vector<long long> &ofs);
constexpr int COEF_KEY_S0X2 = -1;   // key of that table in sharp_alm_info::coef (key 0 stays the one-step table of invn.cu)
constexpr int COEF_KEY_S0X2P2 = -2; // the same up to lmax + 2: spin 2 run as scalar sums (legendre.cu, launch_s2s_*)
void build_start_norms(int mmax, std::vector<double> &K0, std::vector<double> &K2);
void build_start_norms_spin(int mmax, int spin, std::vector<double> &Ks);

struct CoefDev {            // device copy of one (alm_info, spin) coefficient table
  bool ready = false;
  double *tab = nullptr;    // spin 0: {A', g} per l ; spin 2: {A', C', g, 0} per l ; COEF_KEY_S0X2: {a_j, b'_j} per two l
  double *tab2 = nullptr;   // COEF_KEY_S0X2 only: mix rows {u_j, v_j, h_j, v_{j-1}}, row index = ofs / 2 + j
  long long *ofs = nullptr; // per local m: offset (in doubles) of l = l0
  long long *tofs = nullptr; // per local m: first synthesis tile row (rows padded to a multiple of 8)
  long long trows = 0;       // total synthesis tile rows
  long long nofs = 0;        // offset past the last local m (doubles)
};

// Region of the ring-FFT work buffer: pairs [first, first+np) share one FFT length.
struct FftRegion {
  int first = 0, np = 0;
  int len = 0;              // FFT length (nph for direct, power of two M for Bluestein)
  bool bluestein = false;
  long long base = 0;       // complex elements before this region, for ONE component
};

}  // namespace cmdr

// The opaque handles of the ABI.
struct sharp_alm_info {
  int lmax = 0, nm = 0, stride = 1, flags = 0;
  bool real_packed = true;
  std::vector<int> mval;
  std::vector<long long> mvstart;   // element index of (l=0) for each m (may be negative)
  long long nalm = 0;               // reals (real-packed) or complex elements (general)
  int mmax = -1;
  // device
  int *d_mval = nullptr;
  long long *d_mvstart = nullptr;
  int *d_m2im = nullptr;            // size mmax+1, -1 when m is not local
  std::map<int, double *> d_K;      // per spin: start-value normalisation per m
  std::map<int, cmdr::CoefDev> coef; // per spin: coefficient table
  int device = -1;
};

struct sharp_geom_info {
  int nside = 0, nrings = 0;
  std::vector<int> ring;            // as given (1-based), map storage order
  long long npix = 0;               // local pixel count
  // ring pairs sorted by colatitude of the northern member
  int npairs = 0;
  std::vector<int> north;           // northern ring number 1..2nside
  std::vector<double> cth, sth, sh, ch, wgt;
  std::vector<int> nph, shifted;
  std::vector<long long> ofsN, ofsS;
  std::vector<cmdr::FftRegion> regions;
  long long zlen_total = 0;         // complex elements of the FFT buffer per component
  long long vlen_total = 0;         // complex elements of the Bluestein filter table
  // device
  double *d_trig = nullptr;         // npairs * 4: cth, sth, sh, ch
  double *d_wgt = nullptr;
  int *d_nph = nullptr, *d_shifted = nullptr;
  long long *d_ofsN = nullptr, *d_ofsS = nullptr;
  long long *d_zbase = nullptr;     // per pair: region base
  int *d_zidx = nullptr, *d_znp = nullptr, *d_zlen = nullptr, *d_zblue = nullptr;
  double *d_vtab = nullptr;         // Bluestein filter spectra (complex), built lazily
  double *d_vtab_br = nullptr;      // the same in bit-reversed order for the classes of the fused kernel (ringfft.cu)
  std::map<int, double *> d_vsub;   // per split region: filter spectra of the length-n/4 sub-transforms (ringfft.cu)
  bool vtab_ready = false;
  std::map<long long, int> plans;   // key (region<<8 | ncomp) -> cufftHandle
  std::map<long long, int *> mlim;  // key (lmax<<8 | spin) -> device int[npairs]
  int device = -1;
  // ring-pair sub-ranges used to pipeline host<->device copies with compute (abi.cu)
  int pair0 = 0;                       // first parent pair (sub-geometries only)
  bool subs_built = false;
  std::vector<sharp_geom_info *> subs; // empty when the ring list is not chunkable
};
