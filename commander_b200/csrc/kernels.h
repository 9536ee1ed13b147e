// kernels.h -- launcher interface between the ABI layer (abi.cu) and the CUDA stages.
#pragma once
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <vector>

#include "sht_internal.h"

namespace cmdr {

constexpr int CMDR_MAX_PEERS = 8;
constexpr int CMDR_MAX_SPIN = 32;   // start values use plain powers sh^(2s), ch^(2s): fine in FP64 up to here

void count_launch(int n = 1);

// Geometry as the Legendre stage sees it: `nslots` ring-pair slots stored as [owner][NPL].
// The kernels walk WORK indices; `trig` (cth,sth,sh,ch) and the per-ring m cut-off `mlim`
// (-1 = empty slot) are in work order and `wslot` maps a work index to its storage slot.  On
// several GPUs the work order is by colatitude, so that the 32 R rings of a warp are neighbours
// on the sphere whoever owns them (identity on one GPU, where storage is already sorted).
struct LegGeom {
  int nslots = 0, NPL = 0, nowners = 1;
  int slot_begin = 0, slot_end = -1;   // sub-range of slots to process (-1: all)
  int NML = 0;                    // padded number of local m's (phase buffer row count per comp)
  int ncomp_tot = 1, comp0 = 0;   // components in the phase buffer / first one written here
  const double *trig = nullptr;   // nslots*4
  const int *mlim = nullptr;      // nslots
  const int *wslot = nullptr;     // nslots, or nullptr for the identity
  // Fused exchange (multi-GPU): when npeer > 0, peer[o] is the phase buffer of ring owner o
  // (peer-mapped memory over NVLink) and `src_rank` the block of this rank in it.  Synthesis
  // stores the phases of owner o's slots straight into peer[o]; analysis loads them from there.
  // No send buffer and no all-to-all in either direction.
  int npeer = 0, src_rank = 0;
  double4 *peer[CMDR_MAX_PEERS] = {};
};

// alm side of the Legendre stage (local m's of this rank)
struct LegAlm {
  int lmax = 0, nm = 0, real_packed = 1;
  int spin = 0;                    // 0, or s >= 1 (two components; coefficient table and start norms of that spin)
  int im_begin = 0, im_end = -1;   // sub-range of local m's to process (-1: all)
  const int *mval = nullptr;
  const long long *mvstart = nullptr;
  const double *coef = nullptr;    // spin 0: rec rows {a_j, b'_j} of the two-l-per-step scheme; spin s: {A', C', g, 0}
  const double *coef2 = nullptr;   // spin 0: mix rows {u_j, v_j, h_j, v_{j-1}}
  const long long *cofs = nullptr;
  const double *Kstart = nullptr;  // start-value normalisation of this spin, indexed by m
  // spin 2: scalar (spin-0, two l per step) tables and start norms for the front phase of the kernels (nullptr: off)
  const double *front_coef = nullptr, *front_mix = nullptr, *front_K0 = nullptr;
  const long long *front_cofs = nullptr;
  const long long *tofs = nullptr; // first synthesis tile row of each local m (rows padded to 8 per m)
  long long trows = 0;             // total tile rows
  // optional factor per l for each component of this spin (device, lmax+1 entries; nullptr = 1): applied to the
  // a_lm on load (synthesis) and on store (analysis) -- how cr_matmulA's sqrt(S), beam and F_mean passes
  // (commander3/src/comm_cr_mod.f90:797-836, 957-1008; comm_B_bl_mod.f90:108-127) ride in the Legendre kernels
  const double *lscale[2] = {nullptr, nullptr};
  bool deriv1 = false;             // SHARP_ALM2MAP_DERIV1 (spin 1 tables, one a_lm column): prep_d1 / synth_d1 kernels
};

// Column counts of a job.  SHARP_ALM2MAP_DERIV1 is a synthesis from ONE spin-0 a_lm column to TWO maps
// {d_theta T, d_phi T / sin theta}; it runs on the spin-1 tables whatever spin the caller passes.
inline bool job_synth(int type) { return type == SHARP_Y || type == SHARP_WY || type == SHARP_ALM2MAP_DERIV1; }
inline int job_spin(int type, int spin) { return type == SHARP_ALM2MAP_DERIV1 ? 1 : spin; }
inline int job_alm_cols(int type, int spin) { return type == SHARP_ALM2MAP_DERIV1 ? 1 : (spin == 0 ? 1 : 2); }
inline int job_map_cols(int type, int spin) { return type == SHARP_ALM2MAP_DERIV1 ? 2 : (spin == 0 ? 1 : 2); }
unsigned long long job_opcnt(const sharp_geom_info *g, const sharp_alm_info *a, int type, int spin);
// The fused T + (Q,U) entry points (execute_iqu[_batch|_dist]) run the four map <-> a_lm jobs only: DERIV1 has one
// a_lm column and two maps per transform, which their three-column pointer tables cannot carry.
inline void require_iqu_job(int type, const char *who) {
  if (type < SHARP_YtW || type > SHARP_WY) { fprintf(stderr, "cmdr_sht: %s: job type %d unsupported\n", who, type); abort(); }
}

// Optional element-wise factors fused into a transform (cr.cu): per l on the a_lm side, per local pixel on the map
// side of a synthesis (N^-1 of commander3/src/comm_N_rms_mod.f90:264-273 in the ring-FFT epilogue).
struct XformOpts {
  const double *lscale[3] = {nullptr, nullptr, nullptr};
  const double *pixscale[3] = {nullptr, nullptr, nullptr};
};

// Phase buffer element: {north re, north im, south re, south im}.  One block of NML x NPL elements per (ring owner /
// m owner, component); inside a block the element of (local m `im`, local ring pair `pair`) sits at
//   ring-major (default):  pair * NML + im   -- the phases of ONE ring pair for consecutive m are contiguous, so the
//                          ring-FFT kernels (one CTA per ring pair) read and write whole rows; the Legendre kernels'
//                          one-element-per-ring accesses become 32-byte scatters, which their low bandwidth need
//                          (1 GB over >= 20 ms) does not notice
//   m-major (CMDR_SHT_PH_LAYOUT=m, the round-1 layout):  im * NPL + pair
bool phase_ring_major();
__host__ __device__ inline size_t ph_index(int block, int ncomp_tot, int comp, int NML, int NPL, int im, int pair, bool ring_major) {
  const size_t base = (size_t)(block * ncomp_tot + comp) * NML * NPL;
  return ring_major ? base + (size_t)pair * NML + im : base + (size_t)im * NPL + pair;
}
//
// synthesis: alm (device, ncomp pointers) -> ph ; analysis: ph -> alm (atomic accumulate)
// `prep`: (re)build the pre-scaled a_lm tile rows first; false when the same a_lm were already
// prepared by an earlier launch of this transform (ring-pair chunks of the pipelined host path)
void launch_legendre_synth(int spin, const LegGeom &g, const LegAlm &a, const double *const *alm,
                           double4 *ph, cudaStream_t st, bool prep = true);
void launch_legendre_anal(int spin, const LegGeom &g, const LegAlm &a, double *const *alm,
                          const double4 *ph, cudaStream_t st);

// Ring-FFT stage on the LOCAL rings of `geom` (ringfft.cu).
// The phase buffer on this side is indexed
//   ((src*ncomp_tot + comp0 + c)*NML + im_src)*NPL + local_pair
// with the (m -> src, im) lookup tables below (src = rank that owns m).
struct PhaseLayout {
  int NPL = 0, NML = 0, ncomp_tot = 1, comp0 = 0;
  int pair0 = 0;                 // phase-buffer index of this geometry's first ring pair
  int mmax = -1;                 // largest m present anywhere
  const int *m2src = nullptr;    // size mmax+1 (-1: m absent)
  const int *m2im = nullptr;     // size mmax+1
  int nm_total = 0;              // number of (src, im) entries (all ranks)
  const int *mlist = nullptr;    // nm_total: m value
  const int *mlist_src = nullptr, *mlist_im = nullptr;
};

void ringfft_synth(sharp_geom_info *geom, int ncomp, const PhaseLayout &L, const double4 *ph,
                   double *const *map, bool weighted, bool add, cudaStream_t st,
                   const double *const *pixscale = nullptr);
size_t ringfft_scratch_elems(const sharp_geom_info *geom);   // FFT work elements per component the cuFFT regions need (0: none)
void ringfft_anal(sharp_geom_info *geom, int ncomp, const PhaseLayout &L, double4 *ph,
                  const double *const *map, bool weighted, cudaStream_t st);

// scratch memory arena and shared engine helpers (abi.cu)
void *scratch_get(const char *name, size_t bytes);
void ensure_alm_device(sharp_alm_info *a);
void ensure_geom_device(sharp_geom_info *g);
LegAlm make_legalm(sharp_alm_info *a, int spin, bool classic = false);
void ring_trig_ld(int nside, int north, long double &cth, long double &sth, long double &sh, long double &ch);
bool is_device_ptr(const void *p);
extern thread_local int g_profiling;
void prof_begin(int spin, int dir, cudaStream_t st);
void prof_end(cudaStream_t st);
void prof_collect();
// pinned-host pipelining helpers (abi.cu), shared with the distributed path
sharp_geom_info *make_subgeom(const sharp_geom_info *g, int a, int b);
bool pairs_contiguous(const sharp_geom_info *g);
void sub_ranges(const sharp_geom_info *s, long long &nb, long long &ne, long long &sb, long long &se);
bool is_pinned_host(const void *p);
// start offsets of the local m columns in a dense packed a_lm array and a cut of the m range into nch pieces of about equal
// size (false for layouts that are not dense or have fewer than 64 m's)
bool alm_m_chunks(const sharp_alm_info *a, long long nalm_d, int nch, std::vector<long long> &mstart, std::vector<int> &mcut);
cudaStream_t copy_stream();
cudaEvent_t pooled_event(size_t i);
// host staging for pageable caller arrays (hostio.cu)
enum class HostKind { Device, Pinned, Pageable };
HostKind host_kind(const void *p);
void *pinned_get(const char *name, size_t bytes, bool write_combined = false);
void pinned_release();
void host_copy(void *dst, const void *src, size_t bytes);   // multi-threaded memcpy (blocking)
int host_copy_threads();
void host_copy_set_ranks(int ranks_on_this_node);   // sizes the copy-thread pool so that all ranks fit the node's CPUs
// The columns of one caller array (alm or map) as the pipelined paths move them: pinned columns are copied in
// place; pageable columns go through the library's pinned arena (same offsets), uploads staged by the copy
// threads before the H2D is queued, downloads landing in the arena and moved to the caller by drain().
class HostIO {
 public:
  void init(const char *tag, double *const *cols, int ncols, long long count, bool upload_ring = false);
  bool pageable() const { return pageable_; }
  void h2d(double *dev, int c, long long ofs, long long n, cudaStream_t s);
  void d2h(const double *dev, int c, long long ofs, long long n, cudaStream_t s);
  void commit(cudaStream_t s);   // marks the downloads queued so far on `s` as one completion group
  void drain();                  // waits for the groups in order and hands the data to the caller (call before returning)
 private:
  struct Drain { cudaEvent_t ev; double *dst; const double *src; size_t bytes; bool done = false; bool deferred = false; };
  double *stage_dn();
  double *stage_up();
  double *user_[4] = {};
  double *stage_ = nullptr, *stage_up_ = nullptr;
  const char *tag_ = "";
  int ncols_ = 0;
  long long count_ = 0;
  bool pageable_ = false, ring_ = false;
  std::vector<Drain> drains_;
  std::vector<cudaEvent_t> events_;
};

struct Staged {
  std::vector<double *> dev;
  std::vector<double *> host;
  bool staged = false;
};
Staged stage_in(const char *tag, double *const *ptrs, int n, long long count, bool copy_in, cudaStream_t st);
void stage_out(Staged &s, long long count, cudaStream_t st);
void execute_any(int type, int spin, void *alm_v, void *map_v, sharp_geom_info *g, sharp_alm_info *a,
                 int flags, double *time, unsigned long long *opcnt, cudaStream_t st);
// device-pointer transforms with fused factors (single GPU: abi.cu; any registered comm: dist.cu)
void run_single(int type, int spin, double *const *alm, double *const *map, sharp_geom_info *g,
                sharp_alm_info *a, int flags, cudaStream_t st, const XformOpts *opts = nullptr, int comp_off = 0);
int effective_comm(int comm, const sharp_geom_info *g, const sharp_alm_info *a, const char *who);
void execute_iqu_opts(int comm, int type, int nmaps, double *const *alm, double *const *map, sharp_geom_info *gT,
                      sharp_geom_info *gP, sharp_alm_info *a, int flags, const XformOpts *opts, cudaStream_t st);

}  // namespace cmdr

#define CMDR_CUDA_CHECK(x)                                                                   \
  do {                                                                                       \
    cudaError_t e_ = (x);                                                                    \
    if (e_ != cudaSuccess) {                                                                 \
      fprintf(stderr, "cmdr_sht: CUDA error %s at %s:%d: %s\n", cudaGetErrorName(e_), __FILE__, \
              __LINE__, cudaGetErrorString(e_));                                             \
      abort();                                                                               \
    }                                                                                        \
  } while (0)
