// kernels.h -- launcher interface between the ABI layer (abi.cu) and the CUDA stages.
#pragma once
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <vector>

#include "cr_draw.h"
#include "cr_plan.h"
#include "job.h"
#include "sht_internal.h"

namespace cmdr {

constexpr int CMDR_MAX_PEERS = 8;

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
  // Handles that key the per-plan seed tables of the Legendre kernels (legendre.cu), set by a caller that launches every
  // slot of the geometry on one GPU; nullptr: every warp starts from the closed-form start values.
  const void *seed_geom = nullptr, *seed_alm = nullptr;
  // spin 2 as scalar sums (legendre.cu, launch_s2s_*): slots [0, s2s_npolar) have sin(theta) < S2S_MIN_STH and stay on
  // the spin-2 kernels; -1: the route is off.  Set by a caller that launches every slot of the geometry on one GPU.
  int s2s_npolar = -1;
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
  // spin 2 as scalar sums: the two-l-per-step spin-0 tables up to lmax + 2 (rec, mix, offsets in doubles, tile rows),
  // the spin-0 start norms and the number of l slots of the table (nullptr: the route is off)
  const double *s2s_coef = nullptr, *s2s_mix = nullptr, *s2s_K0 = nullptr;
  const long long *s2s_cofs = nullptr, *s2s_tofs = nullptr;
  long long s2s_trows = 0, s2s_nl = 0;
};
// spin 2 as scalar sums on (default) or off (cmdr_sht_set_spin2_scalar)
bool spin2_scalar_on();

unsigned long long job_opcnt(const sharp_geom_info *g, const sharp_alm_info *a, const Job &job);

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
void launch_legendre_synth(const LegGeom &g, const LegAlm &a, const double *const *alm, double4 *ph, cudaStream_t st,
                           bool prep = true);
// In deterministic mode (deterministic(), det.h) the analysis kernels store per-warp-block partials and an ordered reduce
// adds them to the a_lm.  reduce = false: one piece of an analysis that a pipelined caller launches over several cuts of
// the slot range (det_cut on det_block_slots(spin)); the caller then runs legendre_anal_reduce for each m range once all
// pieces covering it are queued.  Outside deterministic mode `reduce` is ignored and legendre_anal_reduce does nothing.
void launch_legendre_anal(const LegGeom &g, const LegAlm &a, double *const *alm, const double4 *ph, cudaStream_t st,
                          bool reduce = true);
void legendre_anal_reduce(const LegGeom &g, const LegAlm &a, double *const *alm, cudaStream_t st);
bool deterministic();              // cmdr_sht_set_deterministic / CMDR_SHT_DETERMINISTIC
// SHARP_ADD analysis in deterministic mode (abi.cu): det_add_begin returns zeroed scratch columns for the analysis to
// write (else `alm` itself), det_add_end adds them once to `alm`, a = a + r, so that an ADD gives the prior values plus
// the plain result on every route (the spin-2 scalar-sum route adds to the a_lm twice)
double *const *det_add_begin(bool add, double *const *alm, int ncols, size_t nd, cudaStream_t st);
void det_add_end(double *const *out, double *const *alm, int ncols, size_t nd, cudaStream_t st);
int det_block_slots(int spin);     // work slots per warp block of the deterministic analysis kernels
// Seed tables (legendre.cu): dropped with the geometry or alm handle they were built for, or all at once.
void seed_forget(const void *h);
void seed_release();

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
// The Legendre-stage view of `a` for `job`, with lscale[c] (nullptr: none) as the factor per l of a_lm component c.
// `classic`: spin 0 with the one-step table {A', g} (invn.cu); the transforms use the two-l-per-step tables.
LegAlm make_legalm(sharp_alm_info *a, const Job &job, const double *const *lscale = nullptr, bool classic = false);
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
void execute_any(const Job &job, void *alm_v, void *map_v, sharp_geom_info *g, sharp_alm_info *a, double *time,
                 unsigned long long *opcnt, cudaStream_t st);
// device-pointer transforms with fused factors (single GPU: abi.cu; any registered comm: dist.cu)
void run_single(const Job &job, double *const *alm, double *const *map, sharp_geom_info *g, sharp_alm_info *a,
                cudaStream_t st, const XformOpts *opts = nullptr, int comp_off = 0);
int effective_comm(int comm, const sharp_geom_info *g, const sharp_alm_info *a, const char *who);
void execute_iqu_opts(int comm, int type, int nmaps, double *const *alm, double *const *map, sharp_geom_info *gT,
                      sharp_geom_info *gP, sharp_alm_info *a, int flags, const XformOpts *opts, cudaStream_t st);

// constrained-realisation pieces shared by the one-component system (cr.cu) and the multi-component one (cr_multi.cu)
// m = N^-1 d (+ sqrt(N^-1) eta): the map of one band and map column in cr_computeRHS
void cr_rhs_map(double *m, const double *invN, const double *d, const double *eta, long long n, cudaStream_t st);
// Where the fluctuation terms of cr_computeRHS come from: the caller's columns, or the device stream of rng.cuh
struct RhsEta {
  const double *const *pix = nullptr;   // caller eta_pix columns (per band and map), nullptr: no pixel term (draw = false)
  bool draw = false;                    // draw on the device: (seed, index) of the stream, `terms` CMDR_CR_ETA_PIX | _ALM
  unsigned long long seed = 0, index = 0;
  int terms = 0;
};
// The RHS map of band q, map j (column `col` of data and eta_pix) into m: N^-1 d (data_col nullptr: d = 0) plus the pixel
// term of `eta`.  `rings`, `nrings`: the band's table (cr_ring_table_device); tmp: 2 np doubles of device scratch (cr_draw.cu)
void cr_rhs_column(double *m, const double *invN, const double *data_col, const RhsEta &eta, int col, int q, int j, long long np,
                   const CrRing *rings, int nrings, double *tmp, cudaStream_t st);
CrRing *cr_ring_table_device(const sharp_geom_info *g);   // the caller frees it
// eta of band q, map j at every local pixel into dst (np doubles, host or device)
void cr_draw_pix(double *dst, const CrRing *rings, int nrings, long long np, unsigned long long seed, unsigned long long draw,
                 int q, int j, cudaStream_t st);
// eta_0 of component k at every local slot of `a` into out[j * stride + slot], j < nmaps (device)
void cr_draw_alm(double *out, long long stride, sharp_alm_info *a, int nmaps, unsigned long long seed, unsigned long long draw,
                 int k, cudaStream_t st);
// nlm ([nmaps][nalm] device) = N^-1_{lm,lm} of one band from its N^-1 maps ([nmaps][npix] device): compute_invN_lm
void cr_invn_lm(int comm, int nmaps, double *invN, sharp_geom_info *gT, sharp_geom_info *gP, sharp_alm_info *a, double *nlm,
                cudaStream_t st);
struct CrMulti;
CrMulti *cr_multi_create(int comm, const CrPlan &plan, const sharp_alm_info *const *comp_alm, const int *comp_nmaps,
                         const double *const *sqrtS,
                         const sharp_geom_info *const *band_geom_T, const sharp_geom_info *const *band_geom_P,
                         const sharp_alm_info *const *band_alm, const int *band_nmaps, const double *const *invN,
                         const double *const *b_l, const double *F_mean, int precond, cudaStream_t st);
void cr_multi_destroy(CrMulti *S);
long long cr_multi_length(const CrMulti *S);
void cr_multi_columns(const CrMulti *S, std::vector<long long> &len);   // a_lm per column of a CG vector
bool cr_multi_has_precond(const CrMulti *S);   // a preconditioner other than the identity is selected
void cr_multi_matmulA(CrMulti *S, const double *x, double *y, cudaStream_t st);
void cr_multi_rhs(CrMulti *S, const double *const *data, const RhsEta &eta, const double *eta_alm, double *b, cudaStream_t st);
// The draws of the stream for this handle: eta_pix (per band and map, host or device; nullptr: none) and eta_alm (a device
// CG vector, zeros on the components without a prior; nullptr: none)
void cr_multi_draw_eta(CrMulti *S, unsigned long long seed, unsigned long long draw, double *const *eta_pix, double *eta_alm,
                       cudaStream_t st);
// z = M^-1 r with the selected preconditioner (pseudo-inverse or block diagonal; collective with the pseudo-inverse)
void cr_multi_precond(CrMulti *S, const double *r, double *z, cudaStream_t st);
// cmdr_cr_set_pseudoinv on a multi-component handle: checks (collectively), builds the tables on first use, selects
void cr_multi_set_pseudoinv(CrMulti *S, int on, cudaStream_t st);
// cmdr_cr_set_mixing_map on a multi-component handle: checks (collectively), then installs or removes the map
void cr_multi_set_mixing(CrMulti *S, int band, int comp, const double *const *F, cudaStream_t st);
// true when every rank of `comm` passed the same v (one 8-byte max all-reduce of (v, -v)); true on one GPU
bool comm_all_equal(int comm, int v, cudaStream_t st);
// rank and size of `comm` when it is a registered group of several ranks (true); else rank 0 of 1 (false)
bool comm_group(int comm, int &rank, int &nranks);
// NCCL all-gather of `bytes` per rank on a registered group of several ranks: out (device) receives the ranks' blocks
// in rank order
void comm_allgather(int comm, const void *in, void *out, size_t bytes, cudaStream_t st);

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

namespace cmdr {

// device copy of a host vector (one element allocated for an empty one); the caller frees it
template <typename T>
T *upload(const std::vector<T> &v) {
  T *d = nullptr;
  size_t n = v.size() ? v.size() : 1;
  CMDR_CUDA_CHECK(cudaMalloc(&d, sizeof(T) * n));
  if (v.size()) CMDR_CUDA_CHECK(cudaMemcpy(d, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice));
  return d;
}

}  // namespace cmdr
