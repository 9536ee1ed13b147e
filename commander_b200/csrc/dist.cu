// dist.cu -- multi-GPU SHT: one process per GPU, libsharp-MPI layout.
//
// Replaces sharp_execute_mpi (reached through sharp_execute_mpi_fortran,
// commander3/src/sharp.f90:96-104,226-232) where libsharp2 does: Allgather of the
// per-rank m lists and ring-pair colatitudes, Legendre for local m over ALL ring pairs,
// one MPI_Alltoallv of complex phases, FFT on local rings.  Layout of m's and rings per
// rank is whatever the caller's handles say (comm_mapinfo uses round-robin,
// commander3/src/comm_map_mod.f90:197-261); it is discovered with NCCL all-gathers.
//
// Default exchange: FUSED into the producing kernels.  Every rank owns two receive buffers
// (synthesis side, analysis side) that all other ranks map through CUDA IPC; the synthesis
// Legendre kernel stores each warp's phases straight into the ring owner's buffer and the analysis
// Legendre kernel loads each warp's phases straight from the ring owner's buffer (coalesced
// NVLink/NVSwitch peer accesses), so the m <-> ring transpose overlaps the math warp by warp and
// there is no send buffer, no pack pass and no separate all-to-all.  Two 4-byte NCCL all-reduces per transform act as the cross-GPU
// stream barriers (buffer free / buffer complete).
// Fallback (CMDR_SHT_P2P=0, more than 8 ranks, or IPC mapping unavailable): an NCCL all-to-all
// (grouped ncclSend/ncclRecv) between a send and a receive buffer in the same block layout
// ([owner][comp][m][ring pair]); still no pack/unpack passes.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <chrono>
#include <cstring>
#include <map>
#include <tuple>

#include "det.h"
#include "kernels.h"
#include "legendre_core.cuh"

namespace cmdr {

#define CMDR_NCCL_CHECK(x)                                                                  \
  do {                                                                                      \
    ncclResult_t r_ = (x);                                                                  \
    if (r_ != ncclSuccess) {                                                                \
      fprintf(stderr, "cmdr_sht: NCCL error %s at %s:%d\n", nccl_api()->GetErrorString(r_), __FILE__, __LINE__); \
      abort();                                                                              \
    }                                                                                       \
  } while (0)

// NCCL is bound at first use with dlopen so that (a) loading this library never drags a
// second libnccl into a process that already has one (PyTorch bundles its own), and (b) a
// single-GPU Commander run needs no NCCL at all.  Order: an already-loaded libnccl.so.2,
// $CMDR_SHT_NCCL_LIB, then the system libnccl.so.2.
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId *);
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int);
  ncclResult_t (*CommDestroy)(ncclComm_t);
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*GroupStart)();
  ncclResult_t (*GroupEnd)();
  const char *(*GetErrorString)(ncclResult_t);
};
static NcclApi *nccl_api() {
  static NcclApi api;
  static bool ready = false;
  if (ready) return &api;
  void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
  if (!h) { const char *e = getenv("CMDR_SHT_NCCL_LIB"); if (e && *e) h = dlopen(e, RTLD_NOW | RTLD_GLOBAL); }
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) { fprintf(stderr, "cmdr_sht: cannot load libnccl.so.2 (%s)\n", dlerror()); abort(); }
  auto need = [&](const char *name) {
    void *s = dlsym(h, name);
    if (!s) { fprintf(stderr, "cmdr_sht: libnccl lacks %s\n", name); abort(); }
    return s;
  };
  api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(need("ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(need("ncclCommInitRank"));
  api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(need("ncclCommDestroy"));
  api.AllGather = reinterpret_cast<decltype(api.AllGather)>(need("ncclAllGather"));
  api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(need("ncclAllReduce"));
  api.Send = reinterpret_cast<decltype(api.Send)>(need("ncclSend"));
  api.Recv = reinterpret_cast<decltype(api.Recv)>(need("ncclRecv"));
  api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(need("ncclGroupStart"));
  api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(need("ncclGroupEnd"));
  api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(need("ncclGetErrorString"));
  ready = true;
  return &api;
}

struct DistPlan {
  int NPL = 0, NML = 0, mmax = -1, nm_total = 0;
  int nslots = 0;
  // Legendre work order: all ranks' ring pairs sorted by colatitude, empty (padding) slots last
  double *d_trig = nullptr;                 // [nranks*NPL][4], work order
  int *d_wslot = nullptr;                   // work index -> storage slot owner*NPL + local
  std::map<int, int *> d_mlim;              // per spin: [nranks*NPL], work order
  std::vector<double> h_sth, h_cth;         // per work index (0 for empty)
  std::vector<int> h_valid;
  int *d_m2src = nullptr, *d_m2im = nullptr, *d_mlist = nullptr, *d_mlist_src = nullptr, *d_mlist_im = nullptr;
  // pinned-host pipeline: the valid work slots cut into chunks (multiples of 128 slots, the same on every
  // rank) and, per chunk, this rank's local ring pairs in it (a contiguous range) as a sub-geometry
  int nvalid = 0;
  std::vector<int> wcut;                      // work-slot boundaries, size nchunk + 1
  std::vector<int> lcut;                      // this rank's local pair boundaries, size nchunk + 1
  std::vector<sharp_geom_info *> subs;        // per chunk (nullptr when this rank has no pair in it)
  bool subs_built = false;
  int pipe_ok = 0;                            // chunked host pipeline usable on EVERY rank (agreed in get_plan)
};

struct PeerBuf {                       // one receive buffer per rank, mapped by every rank
  double *mine = nullptr;
  size_t bytes = 0;
  std::vector<double *> peer;          // [nranks], peer[rank] == mine
};

struct DistComm {
  ncclComm_t nccl = nullptr;
  int rank = 0, nranks = 1, device = 0;
  std::map<std::tuple<const sharp_geom_info *, const sharp_alm_info *>, DistPlan *> plans;
  int p2p = -1;                        // -1 undecided, 0 NCCL all-to-all, 1 fused peer stores
  PeerBuf pb[2];                       // [0] analysis side (written by unfold), [1] synthesis side
  PeerBuf pbflag;                      // flag words of the peer-flag barrier (one int per rank, zero-initialised)
  int flag_state = 0;                  // 0 not set up, 1 usable, -1 unavailable (NCCL barrier)
  int epoch = 0;
  int *d_flag = nullptr;               // token of the NCCL barrier
};

static std::map<int, DistComm *> g_comms;

static DistComm *find_comm(int comm) {
  auto it = g_comms.find(comm);
  return it == g_comms.end() ? nullptr : it->second;
}

static void free_plan(DistPlan *P) {
  cudaFree(P->d_trig); cudaFree(P->d_wslot); cudaFree(P->d_m2src); cudaFree(P->d_m2im); cudaFree(P->d_mlist);
  cudaFree(P->d_mlist_src); cudaFree(P->d_mlist_im);
  for (auto &m : P->d_mlim) cudaFree(m.second);
  for (sharp_geom_info *sub : P->subs) if (sub) sharp_destroy_geom_info(sub);
  delete P;
}

// Called by sharp_destroy_geom_info / sharp_destroy_alm_info (abi.cu): every cached plan that was built for the
// handle goes with it, so that a later handle that happens to get the same heap address (comm_mapinfo%dealloc
// followed by a new comm_mapinfo, commander3/src/comm_map_mod.f90:419-431) can never hit a stale plan.
void dist_forget_handle(const void *h) {
  for (auto &kc : g_comms) {
    DistComm *C = kc.second;
    for (auto it = C->plans.begin(); it != C->plans.end();) {
      if ((const void *)std::get<0>(it->first) == h || (const void *)std::get<1>(it->first) == h) {
        DistPlan *P = it->second;
        it = C->plans.erase(it);
        CMDR_CUDA_CHECK(cudaDeviceSynchronize());       // the plan's tables may still be in use by queued kernels
        free_plan(P);
      } else {
        ++it;
      }
    }
  }
}

// An unknown communicator handle must never run silently as a local transform: under `mpirun -np 8` every rank
// holds a strict subset of the rings and m's and the result would be wrong without a message.  The only
// communicator-less case that is well defined is a group of one, where the handles cover the whole sphere.
constexpr int CMDR_COMM_SELF = -1;
static bool covers_sphere(const sharp_geom_info *g, const sharp_alm_info *a) {
  if (g->nrings != 4 * g->nside - 1 || a->nm != a->lmax + 1) return false;
  std::vector<char> seen(a->lmax + 1, 0);
  for (int m : a->mval) seen[m] = 1;
  for (char c : seen) if (!c) return false;
  return true;
}
static DistComm *comm_or_local(int comm, const sharp_geom_info *g, const sharp_alm_info *a, const char *who) {
  DistComm *C = find_comm(comm);
  if (C) return C->nranks == 1 ? nullptr : C;
  if (comm == CMDR_COMM_SELF || covers_sphere(g, a)) return nullptr;     // a group of one
  fprintf(stderr, "cmdr_sht: %s called with communicator %d that was never registered with cmdr_sht_comm_register, and the "
          "handles hold only part of the sphere (%d of %d rings, %d of %d m's): refusing to run a local transform.  "
          "Register every communicator that reaches sharp_execute (INTEGRATION.md section 2).\n",
          who, comm, g->nrings, 4 * g->nside - 1, a->nm, a->lmax + 1);
  abort();
}

// all-gather a vector of ints padded to `n` entries per rank
static std::vector<int> allgather_ints(DistComm *C, const std::vector<int> &mine, int n, cudaStream_t st) {
  std::vector<int> pad(n, -1);
  std::copy(mine.begin(), mine.end(), pad.begin());
  int *d_in = upload(pad), *d_out = nullptr;
  CMDR_CUDA_CHECK(cudaMalloc(&d_out, sizeof(int) * (size_t)n * C->nranks));
  CMDR_NCCL_CHECK(nccl_api()->AllGather(d_in, d_out, n, ncclInt32, C->nccl, st));
  std::vector<int> out((size_t)n * C->nranks);
  CMDR_CUDA_CHECK(cudaMemcpyAsync(out.data(), d_out, sizeof(int) * out.size(), cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  cudaFree(d_in); cudaFree(d_out);
  return out;
}

static DistPlan *get_plan(DistComm *C, sharp_geom_info *g, sharp_alm_info *a, cudaStream_t st) {
  auto key = std::make_tuple((const sharp_geom_info *)g, (const sharp_alm_info *)a);
  auto it = C->plans.find(key);
  if (it != C->plans.end()) return it->second;
  DistPlan *P = new DistPlan;
  const int R = C->nranks;
  // sizes: {nm, npairs, nside, lmax, this rank can take the chunked host pipeline}.  The last entry is agreed here,
  // where every rank is anyway, rather than in try_dist_pipelined: a rank without rings or m's gets null columns, which
  // look like device arrays, and must not skip a collective the other ranks enter.
  const int pipe_mine = (g->npairs > 0 && a->nm > 0 && pairs_contiguous(g)) ? 1 : 0;
  std::vector<int> sz = allgather_ints(C, {a->nm, g->npairs, g->nside, a->lmax, pipe_mine}, 5, st);
  int NML = 1, NPL = 1;
  P->pipe_ok = 1;
  for (int r = 0; r < R; ++r) {
    if (sz[5 * r + 2] != g->nside || sz[5 * r + 3] != a->lmax) {
      fprintf(stderr, "cmdr_sht: ranks disagree on nside/lmax\n"); abort();
    }
    NML = std::max(NML, sz[5 * r]); NPL = std::max(NPL, sz[5 * r + 1]);
    P->pipe_ok = std::min(P->pipe_ok, sz[5 * r + 4]);
  }
  P->NML = NML; P->NPL = NPL; P->nslots = R * NPL;
  std::vector<int> all_m = allgather_ints(C, a->mval, NML, st);
  std::vector<int> all_north = allgather_ints(C, g->north, NPL, st);
  // global slot geometry in work order
  std::vector<std::pair<int, int>> order;   // (north ring, storage slot)
  for (int r = 0; r < R; ++r)
    for (int j = 0; j < sz[5 * r + 1]; ++j) order.emplace_back(all_north[(size_t)r * NPL + j], r * NPL + j);
  std::sort(order.begin(), order.end());
  std::vector<int> wslot(P->nslots, 0);
  std::vector<char> used(P->nslots, 0);
  std::vector<double> trig(4 * (size_t)P->nslots, 0.0);
  P->h_sth.assign(P->nslots, 0.0); P->h_cth.assign(P->nslots, 0.0); P->h_valid.assign(P->nslots, 0);
  int w = 0;
  for (auto &o : order) {
    long double c, sn, sh, ch;
    ring_trig_ld(g->nside, o.first, c, sn, sh, ch);
    trig[4 * w] = (double)c; trig[4 * w + 1] = (double)sn; trig[4 * w + 2] = (double)sh; trig[4 * w + 3] = (double)ch;
    P->h_sth[w] = (double)sn; P->h_cth[w] = (double)c; P->h_valid[w] = 1;
    wslot[w] = o.second; used[o.second] = 1;
    ++w;
  }
  P->nvalid = w;
  {
    // chunks per transform of the host-buffer pipeline (one exchange barrier each; the first chunk's upload and the last
    // chunk's download are not hidden behind kernels, so smaller chunks shorten both ends): CMDR_SHT_DIST_CHUNKS, default 8
    static const int K = (getenv("CMDR_SHT_DIST_CHUNKS") && atoi(getenv("CMDR_SHT_DIST_CHUNKS")) > 0) ? std::min(24, atoi(getenv("CMDR_SHT_DIST_CHUNKS"))) : 8;
    int per = ((P->nvalid + K - 1) / K + 127) / 128 * 128;
    if (per < 128) per = 128;
    for (int b = 0; b < P->nvalid; b += per) P->wcut.push_back(b);
    P->wcut.push_back(P->nvalid);
    // my local pairs are sorted by ring number like the work order: the pairs of a chunk are a contiguous range
    P->lcut.assign(P->wcut.size(), 0);
    int mine = 0, ci = 1;
    for (int wi = 0; wi < P->nvalid; ++wi) {
      while (ci < (int)P->wcut.size() && wi >= P->wcut[ci]) P->lcut[ci++] = mine;
      if (order[wi].second / NPL == C->rank) ++mine;
    }
    while (ci < (int)P->wcut.size()) P->lcut[ci++] = mine;
  }
  for (int s2 = 0; s2 < P->nslots; ++s2) if (!used[s2]) wslot[w++] = s2;   // padding slots: zero-filled, never read
  P->d_trig = upload(trig);
  P->d_wslot = upload(wslot);
  // global m tables
  int mmax = -1;
  for (int r = 0; r < R; ++r) for (int i = 0; i < sz[5 * r]; ++i) mmax = std::max(mmax, all_m[(size_t)r * NML + i]);
  P->mmax = mmax;
  std::vector<int> m2src(mmax + 2, -1), m2im(mmax + 2, -1), mlist, mlist_src, mlist_im;
  for (int r = 0; r < R; ++r)
    for (int i = 0; i < sz[5 * r]; ++i) {
      int m = all_m[(size_t)r * NML + i];
      if (m2src[m] >= 0) { fprintf(stderr, "cmdr_sht: m=%d owned by two ranks\n", m); abort(); }
      m2src[m] = r; m2im[m] = i;
      mlist.push_back(m); mlist_src.push_back(r); mlist_im.push_back(i);
    }
  P->nm_total = (int)mlist.size();
  P->d_m2src = upload(m2src); P->d_m2im = upload(m2im);
  P->d_mlist = upload(mlist); P->d_mlist_src = upload(mlist_src); P->d_mlist_im = upload(mlist_im);
  C->plans[key] = P;
  return P;
}

static const int *plan_mlim(DistPlan *P, int lmax, int spin) {
  auto it = P->d_mlim.find(spin);
  if (it != P->d_mlim.end()) return it->second;
  std::vector<int> ml(P->nslots, -1);
  for (int s = 0; s < P->nslots; ++s)
    if (P->h_valid[s]) ml[s] = mlim_for_ring(lmax, spin, P->h_sth[s], P->h_cth[s]);
  int *d = upload(ml);
  P->d_mlim[spin] = d;
  return d;
}

// Cross-GPU stream barrier: work enqueued after it on any rank starts only after everything
// enqueued before it on every rank has completed (kernel completion makes its peer stores
// visible).  Two implementations:
//  * peer flags (default once the IPC mappings exist): a one-warp kernel stores this barrier's epoch into the flag
//    word it owns in every peer's flag array (system-scope release over NVLink) and spins until all peers' epochs
//    have arrived in its own array -- ~5 us instead of the ~30 us of a 4-byte NCCL all-reduce, which matters at 8
//    GPUs where a transform is 1-3 ms and has 2 barriers (K + 1 in the chunked host pipeline);
//  * a 4-byte NCCL all-reduce (CMDR_SHT_FLAG_BARRIER=0, or while the mappings are being set up).
static void nccl_barrier(DistComm *C, cudaStream_t st) {
  if (!C->d_flag) { CMDR_CUDA_CHECK(cudaMalloc(&C->d_flag, sizeof(int))); CMDR_CUDA_CHECK(cudaMemset(C->d_flag, 0, sizeof(int))); }
  CMDR_NCCL_CHECK(nccl_api()->AllReduce(C->d_flag, C->d_flag, 1, ncclInt32, ncclMax, C->nccl, st));
  count_launch(1);
}

struct FlagPeers { int *p[CMDR_MAX_PEERS]; };

__global__ void flag_barrier_kernel(FlagPeers peers, int *mine, int rank, int nranks, int epoch) {
  const int t = threadIdx.x;
  if (t >= nranks) return;
  __threadfence_system();
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(peers.p[t] + rank), "r"(epoch) : "memory");
  const long long t0 = clock64();
  int v;
  do {
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(mine + t) : "memory");
    if (v - epoch < 0 && clock64() - t0 > 240000000000LL) {    // ~2 min: a rank never arrived (crashed or mismatched collective)
      printf("cmdr_sht: flag barrier timed out on rank %d waiting for rank %d (epoch %d, have %d)\n", rank, t, epoch, v);
      __trap();
    }
  } while (v - epoch < 0);
}

static bool ensure_peerbuf(DistComm *C, PeerBuf &B, size_t bytes, cudaStream_t st);

static void stream_barrier(DistComm *C, cudaStream_t st) {
  static const bool flags_on = !(getenv("CMDR_SHT_FLAG_BARRIER") && atoi(getenv("CMDR_SHT_FLAG_BARRIER")) == 0);
  if (flags_on && C->flag_state == 0 && C->p2p != 0 && C->nranks <= CMDR_MAX_PEERS) {
    C->flag_state = -1;                                        // (ensure_peerbuf uses the NCCL barrier itself)
    C->flag_state = ensure_peerbuf(C, C->pbflag, sizeof(int) * 64, st) ? 1 : -1;
  }
  if (C->flag_state != 1) { nccl_barrier(C, st); return; }
  FlagPeers fp;
  for (int r = 0; r < CMDR_MAX_PEERS; ++r) fp.p[r] = r < C->nranks ? reinterpret_cast<int *>(C->pbflag.peer[r]) : nullptr;
  ++C->epoch;
  flag_barrier_kernel<<<1, 32, 0, st>>>(fp, reinterpret_cast<int *>(C->pbflag.mine), C->rank, C->nranks, C->epoch);
  count_launch(1);
}

static void close_peerbuf(DistComm *C, PeerBuf &B) {
  for (int r = 0; r < (int)B.peer.size(); ++r)
    if (r != C->rank && B.peer[r]) cudaIpcCloseMemHandle(B.peer[r]);
  B.peer.clear();
  if (B.mine) cudaFree(B.mine);
  B.mine = nullptr; B.bytes = 0;
}

// Collective: (re)allocates this rank's receive buffer and maps everybody else's.  Sizes are
// functions of the global maxima NML / NPL, so every rank grows at the same call.
// Returns false (on all ranks) if any rank could not map a peer.
static bool ensure_peerbuf(DistComm *C, PeerBuf &B, size_t bytes, cudaStream_t st) {
  if (B.bytes >= bytes) return true;
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  nccl_barrier(C, st);                         // nobody still uses the old mapping
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  close_peerbuf(C, B);
  size_t want = bytes + bytes / 16 + 256;
  CMDR_CUDA_CHECK(cudaMalloc(&B.mine, want));
  CMDR_CUDA_CHECK(cudaMemset(B.mine, 0, want));
  CMDR_CUDA_CHECK(cudaDeviceSynchronize());    // zeroed before any peer can learn the handle
  B.bytes = want;
  cudaIpcMemHandle_t h;
  CMDR_CUDA_CHECK(cudaIpcGetMemHandle(&h, B.mine));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  char *d_in = nullptr, *d_out = nullptr;
  CMDR_CUDA_CHECK(cudaMalloc(&d_in, 64)); CMDR_CUDA_CHECK(cudaMalloc(&d_out, 64 * (size_t)C->nranks));
  CMDR_CUDA_CHECK(cudaMemcpyAsync(d_in, &h, 64, cudaMemcpyHostToDevice, st));
  CMDR_NCCL_CHECK(nccl_api()->AllGather(d_in, d_out, 64, ncclChar, C->nccl, st));
  std::vector<cudaIpcMemHandle_t> all(C->nranks);
  CMDR_CUDA_CHECK(cudaMemcpyAsync(all.data(), d_out, 64 * (size_t)C->nranks, cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  cudaFree(d_in); cudaFree(d_out);
  B.peer.assign(C->nranks, nullptr);
  int ok = 1;
  for (int r = 0; r < C->nranks; ++r) {
    if (r == C->rank) { B.peer[r] = B.mine; continue; }
    void *ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, all[r], cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); ok = 0; break; }
    B.peer[r] = static_cast<double *>(ptr);
  }
  // agree on the outcome
  int *d_ok = nullptr;
  CMDR_CUDA_CHECK(cudaMalloc(&d_ok, sizeof(int)));
  CMDR_CUDA_CHECK(cudaMemcpyAsync(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice, st));
  CMDR_NCCL_CHECK(nccl_api()->AllReduce(d_ok, d_ok, 1, ncclInt32, ncclMin, C->nccl, st));
  CMDR_CUDA_CHECK(cudaMemcpyAsync(&ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  cudaFree(d_ok);
  if (!ok) {
    if (C->rank == 0) fprintf(stderr, "cmdr_sht: CUDA IPC peer mapping unavailable, using the NCCL all-to-all exchange\n");
    close_peerbuf(C, B);
    return false;
  }
  return true;
}

static bool use_p2p(DistComm *C) {
  if (C->p2p < 0) {
    const char *e = getenv("CMDR_SHT_P2P");
    C->p2p = (e && atoi(e) == 0) || C->nranks > CMDR_MAX_PEERS ? 0 : 1;
  }
  return C->p2p == 1;
}

// all-to-all of equal-sized blocks (in doubles)
static void alltoall_blocks(DistComm *C, const double *send, double *recv, size_t block, cudaStream_t st) {
  CMDR_NCCL_CHECK(nccl_api()->GroupStart());
  for (int r = 0; r < C->nranks; ++r) {
    if (r == C->rank) continue;
    CMDR_NCCL_CHECK(nccl_api()->Send(send + (size_t)r * block, block, ncclDouble, r, C->nccl, st));
    CMDR_NCCL_CHECK(nccl_api()->Recv(recv + (size_t)r * block, block, ncclDouble, r, C->nccl, st));
  }
  CMDR_NCCL_CHECK(nccl_api()->GroupEnd());
  CMDR_CUDA_CHECK(cudaMemcpyAsync(recv + (size_t)C->rank * block, send + (size_t)C->rank * block,
                                  sizeof(double) * block, cudaMemcpyDeviceToDevice, st));
  count_launch(1);
}

struct Part {
  Job job; int comp0; sharp_geom_info *g; double *const *alm; double *const *map;
  const double *lscale[2] = {nullptr, nullptr}, *pixscale[2] = {nullptr, nullptr};   // fused factors (XformOpts)
  bool has_ps() const { return pixscale[0] || pixscale[1]; }
};

// Distributed transform over `parts` (one part = one spin with its geometry; all of the same job type); all parts
// share one phase buffer of ncomp_tot components and one exchange.
static void run_dist(DistComm *C, const Part *parts, int nparts, int ncomp_tot, sharp_alm_info *a, cudaStream_t st) {
  const Job &job = parts[0].job;
  const bool synth = job.synth, add = job.add;
  sharp_geom_info *g0 = parts[0].g;
  for (int i = 0; i < nparts; ++i) {
    ensure_geom_device(parts[i].g);
    if (parts[i].g->north != g0->north) { fprintf(stderr, "cmdr_sht: parts use different ring sets\n"); abort(); }
  }
  ensure_alm_device(a);
  DistPlan *P = get_plan(C, g0, a, st);
  const size_t block = (size_t)ncomp_tot * P->NML * P->NPL * 4;   // doubles per peer block
  PhaseLayout L;
  L.NPL = P->NPL; L.NML = P->NML; L.ncomp_tot = ncomp_tot; L.mmax = P->mmax;
  L.m2src = P->d_m2src; L.m2im = P->d_m2im; L.nm_total = P->nm_total;
  L.mlist = P->d_mlist; L.mlist_src = P->d_mlist_src; L.mlist_im = P->d_mlist_im;
  LegGeom G;
  G.nslots = P->nslots; G.NPL = P->NPL; G.nowners = C->nranks; G.NML = P->NML; G.ncomp_tot = ncomp_tot;
  G.trig = P->d_trig; G.wslot = P->d_wslot;
  // receive buffers are sized for 3 components so that T, QU and IQU calls share one mapping
  const size_t cap = sizeof(double) * (size_t)3 * P->NML * P->NPL * 4 * C->nranks;
  bool fused = use_p2p(C);
  if (fused && !(ensure_peerbuf(C, C->pb[0], cap, st) && ensure_peerbuf(C, C->pb[1], cap, st))) { C->p2p = 0; fused = false; }

  if (fused && synth) {
    PeerBuf &B = C->pb[1];
    G.npeer = C->nranks; G.src_rank = C->rank;
    for (int r = 0; r < C->nranks; ++r) G.peer[r] = reinterpret_cast<double4 *>(B.peer[r]);
    prof_begin(200, 0, st);
    stream_barrier(C, st);                       // every rank has finished reading its buffer
    prof_end(st);
    for (int i = 0; i < nparts; ++i) {
      const Part &p = parts[i];
      LegAlm A = make_legalm(a, p.job, p.lscale);
      G.comp0 = p.comp0; G.mlim = plan_mlim(P, a->lmax, p.job.spin);
      prof_begin(p.job.spin, 0, st);
      launch_legendre_synth(G, A, p.alm, reinterpret_cast<double4 *>(B.mine), st);
      prof_end(st);
    }
    prof_begin(201, 0, st);
    stream_barrier(C, st);                       // every rank's phases have landed
    prof_end(st);
    for (int i = 0; i < nparts; ++i) {
      const Part &p = parts[i];
      L.comp0 = p.comp0;
      if (p.g->npairs == 0) continue;
      prof_begin(100 + p.job.spin, 0, st);
      ringfft_synth(p.g, p.job.map_cols, L, reinterpret_cast<double4 *>(B.mine), p.map, job.weighted, add, st,
                    p.has_ps() ? p.pixscale : nullptr);
      prof_end(st);
    }
    return;
  }
  if (fused) {
    // analysis: FFT + unfold fill this rank's buffer ([m owner][comp][m][pair]); after the barrier
    // every rank's Legendre kernel loads its block from the ring owners' buffers over NVLink
    PeerBuf &B = C->pb[0];
    G.npeer = C->nranks; G.src_rank = C->rank;
    for (int r = 0; r < C->nranks; ++r) G.peer[r] = reinterpret_cast<double4 *>(B.peer[r]);
    prof_begin(200, 1, st);
    stream_barrier(C, st);                       // every rank has finished reading my buffer
    prof_end(st);
    for (int i = 0; i < nparts; ++i) {
      const Part &p = parts[i];
      L.comp0 = p.comp0;
      if (p.g->npairs == 0) continue;
      prof_begin(100 + p.job.spin, 1, st);
      ringfft_anal(p.g, p.job.map_cols, L, reinterpret_cast<double4 *>(B.mine), p.map, job.weighted, st);
      prof_end(st);
    }
    prof_begin(201, 1, st);
    stream_barrier(C, st);                       // every rank's phases are complete
    prof_end(st);
    for (int i = 0; i < nparts; ++i) {
      const Part &p = parts[i];
      LegAlm A = make_legalm(a, p.job, p.lscale);
      G.comp0 = p.comp0; G.mlim = plan_mlim(P, a->lmax, p.job.spin);
      const size_t nd = (size_t)a->nalm * (a->real_packed ? 1 : 2);
      double *const *out = det_add_begin(add, p.alm, p.job.alm_cols, nd, st);
      if (!add && nd)
        for (int c = 0; c < p.job.alm_cols; ++c) CMDR_CUDA_CHECK(cudaMemsetAsync(p.alm[c], 0, sizeof(double) * nd, st));
      prof_begin(p.job.spin, 1, st);
      launch_legendre_anal(G, A, out, reinterpret_cast<const double4 *>(B.mine), st);
      prof_end(st);
      det_add_end(out, p.alm, p.job.alm_cols, nd, st);
    }
    return;
  }

  double *bufA = static_cast<double *>(scratch_get("dist_phA", sizeof(double) * block * C->nranks));
  double *bufB = static_cast<double *>(scratch_get("dist_phB", sizeof(double) * block * C->nranks));
  if (synth) {
    // padded m rows are never written by the kernels: keep them defined
    if (a->nm < P->NML) CMDR_CUDA_CHECK(cudaMemsetAsync(bufA, 0, sizeof(double) * block * C->nranks, st));
    for (int i = 0; i < nparts; ++i) {
      const Part &p = parts[i];
      LegAlm A = make_legalm(a, p.job, p.lscale);
      G.comp0 = p.comp0; G.mlim = plan_mlim(P, a->lmax, p.job.spin);
      prof_begin(p.job.spin, 0, st);
      launch_legendre_synth(G, A, p.alm, reinterpret_cast<double4 *>(bufA), st);
      prof_end(st);
    }
    prof_begin(200, 0, st);
    alltoall_blocks(C, bufA, bufB, block, st);
    prof_end(st);
    for (int i = 0; i < nparts; ++i) {
      const Part &p = parts[i];
      L.comp0 = p.comp0;
      if (p.g->npairs == 0) continue;
      prof_begin(100 + p.job.spin, 0, st);
      ringfft_synth(p.g, p.job.map_cols, L, reinterpret_cast<double4 *>(bufB), p.map, job.weighted, add, st,
                    p.has_ps() ? p.pixscale : nullptr);
      prof_end(st);
    }
  } else {
    CMDR_CUDA_CHECK(cudaMemsetAsync(bufA, 0, sizeof(double) * block * C->nranks, st));
    for (int i = 0; i < nparts; ++i) {
      const Part &p = parts[i];
      L.comp0 = p.comp0;
      if (p.g->npairs == 0) continue;
      prof_begin(100 + p.job.spin, 1, st);
      ringfft_anal(p.g, p.job.map_cols, L, reinterpret_cast<double4 *>(bufA), p.map, job.weighted, st);
      prof_end(st);
    }
    prof_begin(200, 1, st);
    alltoall_blocks(C, bufA, bufB, block, st);
    prof_end(st);
    for (int i = 0; i < nparts; ++i) {
      const Part &p = parts[i];
      LegAlm A = make_legalm(a, p.job, p.lscale);
      G.comp0 = p.comp0; G.mlim = plan_mlim(P, a->lmax, p.job.spin);
      const size_t nd = (size_t)a->nalm * (a->real_packed ? 1 : 2);
      double *const *out = det_add_begin(add, p.alm, p.job.alm_cols, nd, st);
      if (!add && nd)
        for (int c = 0; c < p.job.alm_cols; ++c) CMDR_CUDA_CHECK(cudaMemsetAsync(p.alm[c], 0, sizeof(double) * nd, st));
      prof_begin(p.job.spin, 1, st);
      launch_legendre_anal(G, A, out, reinterpret_cast<const double4 *>(bufB), st);
      prof_end(st);
      det_add_end(out, p.alm, p.job.alm_cols, nd, st);
    }
  }
}

// Host-buffer form of one distributed transform (one spin) with pinned caller arrays and the fused exchange:
// the work slots are processed in chunks with one exchange barrier per chunk, so that the PCIe copy of the map
// rows of chunk c runs beside the Legendre kernel of chunk c+-1 (synthesis: D2H after each chunk's FFT;
// analysis: H2D ahead of each chunk's FFT).  Every rank walks the same chunks, so the barriers match.
static bool try_dist_pipelined(DistComm *C, const Job &job, double *const *alm, double *const *map,
                               sharp_geom_info *g, sharp_alm_info *a, cudaStream_t st) {
  static const bool disabled = getenv("CMDR_SHT_NO_PIPELINE") != nullptr;
  const int spin = job.spin, nca = job.alm_cols, ncomp = job.map_cols;
  if (disabled || job.add || !use_p2p(C)) return false;
  // Every rank must take the same decision (the chunked path has K + 1 exchange barriers, the plain one 2).
  // Global sizes are equal everywhere by construction.  What can differ from rank to rank -- a rank without
  // rings or m's, a ring list that is not contiguous -- was agreed when the plan was built (get_plan, which
  // every rank reaches here).  Once that holds, every rank has non-null columns, and host-versus-device buffers
  // is a property of the call site, the same on all ranks of a collective call (pinned or pageable does not
  // matter: both take this path).
  if ((long long)g->nside * g->nside * 12 < (1LL << 20) * C->nranks) return false;
  const bool synth = job.synth;
  ensure_geom_device(g);
  ensure_alm_device(a);
  DistPlan *P = get_plan(C, g, a, st);
  if (!P->pipe_ok) return false;
  for (int c = 0; c < nca; ++c)
    if (host_kind(alm[c]) == HostKind::Device) return false;
  for (int c = 0; c < ncomp; ++c)
    if (host_kind(map[c]) == HostKind::Device) return false;
  const int K = (int)P->wcut.size() - 1;
  if (!P->subs_built) {
    P->subs_built = true;
    for (int c = 0; c < K; ++c)
      P->subs.push_back(P->lcut[c + 1] > P->lcut[c] ? make_subgeom(g, P->lcut[c], P->lcut[c + 1]) : nullptr);
  }
  const size_t cap = sizeof(double) * (size_t)3 * P->NML * P->NPL * 4 * C->nranks;
  if (!(ensure_peerbuf(C, C->pb[0], cap, st) && ensure_peerbuf(C, C->pb[1], cap, st))) { C->p2p = 0; return false; }
  const long long nalm_d = a->nalm * (a->real_packed ? 1 : 2);
  double *alm_buf = static_cast<double *>(scratch_get("stage_alm", sizeof(double) * (size_t)nalm_d * nca));
  double *map_buf = static_cast<double *>(scratch_get("stage_map", sizeof(double) * (size_t)g->npix * ncomp));
  size_t maxz = 0;
  for (sharp_geom_info *sub : P->subs) if (sub) { ensure_geom_device(sub); maxz = std::max(maxz, ringfft_scratch_elems(sub)); }
  if (maxz) scratch_get("fftbuf", sizeof(double2) * maxz * ncomp);
  double *alm_dev[2], *map_dev[2];
  for (int c = 0; c < nca; ++c) alm_dev[c] = alm_buf + (size_t)c * nalm_d;
  for (int c = 0; c < ncomp; ++c) map_dev[c] = map_buf + (size_t)c * g->npix;
  PhaseLayout L;
  L.NPL = P->NPL; L.NML = P->NML; L.ncomp_tot = ncomp; L.comp0 = 0; L.mmax = P->mmax;
  L.m2src = P->d_m2src; L.m2im = P->d_m2im; L.nm_total = P->nm_total;
  L.mlist = P->d_mlist; L.mlist_src = P->d_mlist_src; L.mlist_im = P->d_mlist_im;
  LegGeom G;
  G.nslots = P->nslots; G.NPL = P->NPL; G.nowners = C->nranks; G.NML = P->NML; G.ncomp_tot = ncomp; G.comp0 = 0;
  G.trig = P->d_trig; G.wslot = P->d_wslot; G.mlim = plan_mlim(P, a->lmax, spin);
  PeerBuf &B = C->pb[synth ? 1 : 0];
  G.npeer = C->nranks; G.src_rank = C->rank;
  for (int r = 0; r < C->nranks; ++r) G.peer[r] = reinterpret_cast<double4 *>(B.peer[r]);
  LegAlm A = make_legalm(a, job);
  cudaStream_t cs = copy_stream();
  const size_t ev0 = 32;                                  // events 0..31 belong to the single-GPU pipeline
  HostIO ioA, ioM;                                        // pageable caller arrays go through the pinned arena (hostio.cu)
  ioA.init("hstage_alm", alm, nca, nalm_d);
  ioM.init("hstage_map", map, ncomp, g->npix);
  // The a_lm move in NMCH chunks of local m's beside the kernels of ONE work-slot chunk (rank-local: no barrier inside):
  // synthesis runs the first chunk's Legendre kernel m-chunk by m-chunk as the upload lands, analysis the last chunk's,
  // sending finished columns back while the next m-chunk is accumulated.
  constexpr int NMCH = 4;
  std::vector<long long> mstart;
  std::vector<int> mcut;
  const int nmch = alm_m_chunks(a, nalm_d, NMCH, mstart, mcut) ? NMCH : 1;
  const size_t evm = 200;                                 // events of the m-chunks
  if (synth) {
    if (nmch == 1) for (int c = 0; c < nca; ++c) ioA.h2d(alm_dev[c], c, 0, nalm_d, st);
    else {
      cudaEvent_t e0 = pooled_event(evm + 2 * NMCH);       // the staging a_lm may still be read by earlier work on `st`
      CMDR_CUDA_CHECK(cudaEventRecord(e0, st));
      CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, e0, 0));
    }
    stream_barrier(C, st);                                 // every rank has finished reading its buffer
    for (int c = K - 1; c >= 0; --c) {                     // belt first, polar caps last
      G.slot_begin = P->wcut[c]; G.slot_end = P->wcut[c + 1];
      if (c == K - 1 && nmch > 1) {
        for (int j = 0; j < nmch; ++j) {
          const long long b = mstart[mcut[j]], e = mstart[mcut[j + 1]];
          for (int k = 0; k < nca; ++k) ioA.h2d(alm_dev[k] + b, k, b, e - b, cs);
          cudaEvent_t ej = pooled_event(evm + j);
          CMDR_CUDA_CHECK(cudaEventRecord(ej, cs));
          CMDR_CUDA_CHECK(cudaStreamWaitEvent(st, ej, 0));
          LegAlm Aj = A;
          Aj.im_begin = mcut[j]; Aj.im_end = mcut[j + 1];
          launch_legendre_synth(G, Aj, alm_dev, reinterpret_cast<double4 *>(B.mine), st, true);
        }
      } else {
        launch_legendre_synth(G, A, alm_dev, reinterpret_cast<double4 *>(B.mine), st, c == K - 1);
      }
      stream_barrier(C, st);                               // chunk c has landed everywhere
      sharp_geom_info *sub = P->subs[c];
      if (!sub) continue;
      L.pair0 = sub->pair0;
      ringfft_synth(sub, ncomp, L, reinterpret_cast<double4 *>(B.mine), map_dev, job.weighted, false, st);
      cudaEvent_t e = pooled_event(ev0 + c);
      CMDR_CUDA_CHECK(cudaEventRecord(e, st));
      CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, e, 0));
      long long nb, ne, sb, se;
      sub_ranges(sub, nb, ne, sb, se);
      for (int k = 0; k < ncomp; ++k) {
        ioM.d2h(map_dev[k] + nb, k, nb, ne - nb, cs);
        ioM.d2h(map_dev[k] + sb, k, sb, se - sb, cs);
      }
      ioM.commit(cs);
    }
    ioM.drain();
    CMDR_CUDA_CHECK(cudaStreamSynchronize(cs));
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  } else {
    const bool det = deterministic();
    cudaEvent_t e0 = pooled_event(ev0 + K);                // staging rows may still be read by earlier work on `st`
    CMDR_CUDA_CHECK(cudaEventRecord(e0, st));
    CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, e0, 0));
    for (int c = 0; c < nca; ++c) CMDR_CUDA_CHECK(cudaMemsetAsync(alm_dev[c], 0, sizeof(double) * nalm_d, st));
    stream_barrier(C, st);                                 // every rank has finished reading my buffer
    for (int c = 0; c < K; ++c) {                          // polar chunks (short rows) first
      sharp_geom_info *sub = P->subs[c];
      if (sub) {
        long long nb, ne, sb, se;
        sub_ranges(sub, nb, ne, sb, se);
        for (int k = 0; k < ncomp; ++k) {
          ioM.h2d(map_dev[k] + nb, k, nb, ne - nb, cs);
          ioM.h2d(map_dev[k] + sb, k, sb, se - sb, cs);
        }
        cudaEvent_t e = pooled_event(ev0 + c);
        CMDR_CUDA_CHECK(cudaEventRecord(e, cs));
        CMDR_CUDA_CHECK(cudaStreamWaitEvent(st, e, 0));
        L.pair0 = sub->pair0;
        ringfft_anal(sub, ncomp, L, reinterpret_cast<double4 *>(B.mine), map_dev, job.weighted, st);
      }
      stream_barrier(C, st);                               // chunk c is complete on every rank
      G.slot_begin = P->wcut[c]; G.slot_end = P->wcut[c + 1];
      // deterministic mode: whole warp blocks per launch (a block that straddles two chunks waits for the later one, whose
      // barrier completes its phases) and one ordered reduce per m range after the last chunk, before its download
      if (det) det_cut(P->wcut[c], P->wcut[c + 1], c == K - 1, P->nslots, det_block_slots(spin), G.slot_begin, G.slot_end);
      if (c == K - 1 && nmch > 1) {
        for (int j = 0; j < nmch; ++j) {
          LegAlm Aj = A;
          Aj.im_begin = mcut[j]; Aj.im_end = mcut[j + 1];
          launch_legendre_anal(G, Aj, alm_dev, reinterpret_cast<const double4 *>(B.mine), st, !det);
          legendre_anal_reduce(G, Aj, alm_dev, st);
          cudaEvent_t ej = pooled_event(evm + NMCH + j);
          CMDR_CUDA_CHECK(cudaEventRecord(ej, st));
          CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, ej, 0));
          const long long b = mstart[mcut[j]], e = mstart[mcut[j + 1]];
          for (int k = 0; k < nca; ++k) ioA.d2h(alm_dev[k] + b, k, b, e - b, cs);
          ioA.commit(cs);
        }
      } else {
        launch_legendre_anal(G, A, alm_dev, reinterpret_cast<const double4 *>(B.mine), st, !det);
        if (c == K - 1) legendre_anal_reduce(G, A, alm_dev, st);
      }
    }
    if (nmch == 1) {
      for (int c = 0; c < nca; ++c) ioA.d2h(alm_dev[c], c, 0, nalm_d, st);
      ioA.commit(st);
    }
    ioA.drain();
    CMDR_CUDA_CHECK(cudaStreamSynchronize(cs));
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  return true;
}

// `jobs`: one per part, all of the same type (T alone, or T and P of a fused IQU call)
static void execute_dist_any(DistComm *C, const Job *jobs, int nparts, double *const *alm, double *const *map,
                             sharp_geom_info *const *geoms, sharp_alm_info *a, cudaStream_t st,
                             const XformOpts *opts = nullptr) {
  const bool synth = jobs[0].synth, add = jobs[0].add;
  // a_lm and map columns: equal except for DERIV1 (one part: 1 a_lm column, 2 maps)
  int ncomp_tot = 0, nalm_tot = 0;
  for (int i = 0; i < nparts; ++i) { ncomp_tot += jobs[i].map_cols; nalm_tot += jobs[i].alm_cols; }
  const long long nalm_d = a->nalm * (a->real_packed ? 1 : 2);
  if (nparts == 1 && !opts && try_dist_pipelined(C, jobs[0], alm, map, geoms[0], a, st)) return;
  Staged sa = stage_in("stage_alm", alm, nalm_tot, nalm_d, synth || add, st);
  Staged sm = stage_in("stage_map", map, ncomp_tot, geoms[0]->npix, !synth || add, st);
  Part parts[4];
  int c0 = 0, ca = 0;
  for (int i = 0; i < nparts; ++i) {
    const int nc = jobs[i].map_cols;
    parts[i] = Part{jobs[i], c0, geoms[i], sa.dev.data() + ca, sm.dev.data() + c0};
    ca += jobs[i].alm_cols;
    if (opts)
      for (int c = 0; c < nc; ++c) { parts[i].lscale[c] = opts->lscale[c0 + c]; parts[i].pixscale[c] = opts->pixscale[c0 + c]; }
    c0 += nc;
  }
  run_dist(C, parts, nparts, ncomp_tot, a, st);
  if (synth) stage_out(sm, geoms[0]->npix, st); else stage_out(sa, nalm_d, st);
  if (sa.staged || sm.staged) CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
}

// the communicator a component should keep using: `comm` when it is a registered group of several ranks, else
// CMDR_COMM_SELF (aborts for an unknown communicator whose handles hold only part of the sphere)
int effective_comm(int comm, const sharp_geom_info *g, const sharp_alm_info *a, const char *who) {
  return comm_or_local(comm, g, a, who) ? comm : CMDR_COMM_SELF;
}

// T (nmaps = 1) or IQU (nmaps = 3) transform on device pointers with fused factors, on one GPU or collectively
// on a registered communicator (cr.cu)
void execute_iqu_opts(int comm, int type, int nmaps, double *const *alm, double *const *map, sharp_geom_info *gT,
                      sharp_geom_info *gP, sharp_alm_info *a, int flags, const XformOpts *opts, cudaStream_t st) {
  const Job jobs[2] = {job_or_abort("execute_iqu_opts", type, 0, flags, true),
                       job_or_abort("execute_iqu_opts", type, 2, flags, true)};
  DistComm *C = comm_or_local(comm, gT, a, "cmdr_cr");
  if (!C) {
    run_single(jobs[0], alm, map, gT, a, st, opts, 0);
    if (nmaps == 3) run_single(jobs[1], alm + 1, map + 1, gP, a, st, opts, 1);
    return;
  }
  sharp_geom_info *gs[2] = {gT, gP};
  execute_dist_any(C, jobs, nmaps == 3 ? 2 : 1, alm, map, gs, a, st, opts);
}

bool comm_all_equal(int comm, int v, cudaStream_t st) {
  DistComm *C = find_comm(comm);
  if (!C || C->nranks == 1) return true;
  const int h[2] = {v, -v};
  int *d = nullptr, r[2];
  CMDR_CUDA_CHECK(cudaMalloc(&d, sizeof(h)));
  CMDR_CUDA_CHECK(cudaMemcpyAsync(d, h, sizeof(h), cudaMemcpyHostToDevice, st));
  CMDR_NCCL_CHECK(nccl_api()->AllReduce(d, d, 2, ncclInt32, ncclMax, C->nccl, st));
  CMDR_CUDA_CHECK(cudaMemcpyAsync(r, d, sizeof(r), cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  cudaFree(d);
  count_launch(1);
  return r[0] == -r[1];   // max v == min v
}

bool comm_group(int comm, int &rank, int &nranks) {
  DistComm *C = find_comm(comm);
  rank = 0; nranks = 1;
  if (!C || C->nranks == 1) return false;
  rank = C->rank; nranks = C->nranks;
  return true;
}

void comm_allgather(int comm, const void *in, void *out, size_t bytes, cudaStream_t st) {
  DistComm *C = find_comm(comm);
  CMDR_NCCL_CHECK(nccl_api()->AllGather(in, out, bytes, ncclChar, C->nccl, st));
  count_launch(1);
}

// out[i] = sum over ranks r in ascending order of all[r n + i]: the deterministic form of cmdr_sht_allreduce_sum
__global__ void __launch_bounds__(256) rank_order_sum_kernel(double *out, const double *all, int n, int nranks) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s = all[i];
  for (int r = 1; r < nranks; ++r) s += all[(size_t)r * n + i];
  out[i] = s;
}

// map *= F, the pixel-space mixing step between Y and YtW (HBM-bound: 24 bytes per pixel)
__global__ void __launch_bounds__(256) scale_map_kernel(double *__restrict__ m, const double *__restrict__ f, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) m[i] *= f[i];
}

}  // namespace cmdr

using namespace cmdr;

extern "C" {

void cmdr_sht_get_unique_id(void *id128) {
  ncclUniqueId id;
  CMDR_NCCL_CHECK(nccl_api()->GetUniqueId(&id));
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id128, &id, sizeof(id));
}

int cmdr_sht_comm_register(int comm, int rank, int nranks, const void *id128) {
  if (find_comm(comm)) return 0;
  DistComm *C = new DistComm;
  C->rank = rank; C->nranks = nranks;
  CMDR_CUDA_CHECK(cudaGetDevice(&C->device));
  if (nranks > 1) {
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    CMDR_NCCL_CHECK(nccl_api()->CommInitRank(&C->nccl, nranks, id, rank));
  }
  g_comms[comm] = C;
  host_copy_set_ranks(nranks);           // one process per GPU on one node: the copy threads of all ranks share its CPUs
  return 0;
}

void cmdr_sht_comm_destroy(int comm) {
  DistComm *C = find_comm(comm);
  if (!C) return;
  std::vector<DistPlan *> plans;
  for (auto &kv : C->plans) plans.push_back(kv.second);
  C->plans.clear();                      // free_plan destroys sub-geometries, whose destructor walks the plan maps
  for (DistPlan *P : plans) free_plan(P);
  close_peerbuf(C, C->pb[0]); close_peerbuf(C, C->pb[1]); close_peerbuf(C, C->pbflag);
  if (C->d_flag) cudaFree(C->d_flag);
  if (C->nccl) nccl_api()->CommDestroy(C->nccl);
  g_comms.erase(comm);
  delete C;
}

void cmdr_sht_comm_set_exchange(int comm, int mode) {
  DistComm *C = find_comm(comm);
  if (!C) return;
  CMDR_CUDA_CHECK(cudaDeviceSynchronize());
  C->p2p = mode < 0 ? -1 : ((mode && C->nranks <= CMDR_MAX_PEERS) ? 1 : 0);
}

void cmdr_sht_execute_dist(int comm, int type, int spin, void *alm, void *map, const sharp_geom_info *geom_info,
                           const sharp_alm_info *alm_info, int flags, void *stream) {
  const Job job = job_or_abort("cmdr_sht_execute_dist", type, spin, flags);
  sharp_geom_info *g = const_cast<sharp_geom_info *>(geom_info);
  sharp_alm_info *a = const_cast<sharp_alm_info *>(alm_info);
  DistComm *C = comm_or_local(comm, g, a, "cmdr_sht_execute_dist");
  if (!C) {
    execute_any(job, alm, map, g, a, nullptr, nullptr, (cudaStream_t)stream);
    return;
  }
  execute_dist_any(C, &job, 1, static_cast<double *const *>(alm), static_cast<double *const *>(map), &g, a,
                   (cudaStream_t)stream);
}

void cmdr_sht_execute_iqu_dist(int comm, int type, double *const *alm3, double *const *map3,
                               const sharp_geom_info *geom_T, const sharp_geom_info *geom_P,
                               const sharp_alm_info *alm_info, int flags, void *stream) {
  const Job jobs[2] = {job_or_abort("cmdr_sht_execute_iqu_dist", type, 0, flags, true),
                       job_or_abort("cmdr_sht_execute_iqu_dist", type, 2, flags, true)};
  DistComm *C = comm_or_local(comm, geom_T, alm_info, "cmdr_sht_execute_iqu_dist");
  if (!C) {
    cmdr_sht_execute_iqu(type, alm3, map3, geom_T, geom_P, alm_info, flags, stream);
    return;
  }
  sharp_geom_info *gs[2] = {const_cast<sharp_geom_info *>(geom_T), const_cast<sharp_geom_info *>(geom_P)};
  execute_dist_any(C, jobs, 2, alm3, map3, gs, const_cast<sharp_alm_info *>(alm_info), (cudaStream_t)stream);
}

void cmdr_sht_allreduce_sum(int comm, double *dev_buf, int n, void *stream) {
  DistComm *C = find_comm(comm);
  if (!C && comm != CMDR_COMM_SELF) {
    fprintf(stderr, "cmdr_sht_allreduce_sum: communicator %d was never registered (cmdr_sht_comm_register); a silent no-op "
            "would leave every rank with its local partial sum\n", comm);
    abort();
  }
  if (!C || C->nranks == 1) return;
  if (deterministic()) {
    // NCCL fixes no reduction order: gather every rank's n values and sum them in rank order, the same bits on every rank
    cudaStream_t st = (cudaStream_t)stream;
    double *all = static_cast<double *>(scratch_get("det_allreduce", sizeof(double) * (size_t)std::max(n, 1) * C->nranks));
    CMDR_NCCL_CHECK(nccl_api()->AllGather(dev_buf, all, n, ncclDouble, C->nccl, st));
    if (n > 0) rank_order_sum_kernel<<<(n + 255) / 256, 256, 0, st>>>(dev_buf, all, n, C->nranks);
    count_launch(2);
    CMDR_CUDA_CHECK(cudaGetLastError());
    return;
  }
  CMDR_NCCL_CHECK(nccl_api()->AllReduce(dev_buf, dev_buf, n, ncclDouble, ncclSum, C->nccl, (cudaStream_t)stream));
  count_launch(1);
}

// Pixel-space mixing: alm <- YtW( F .* Y(alm) ), the spatially varying branch of evalDiffuseBand /
// projectDiffuseBand (commander3/src/comm_diffuse_comp_mod.f90:2078-2080, 2148-2150: `call m%Y();
// m%map = m%map * F%map; call m%YtW()`).  The reference makes four sharp_execute calls and multiplies
// on the host; here the map never leaves the device: only the a_lm (and F, when the caller keeps it
// on the host) cross PCIe.  nmaps = 1 (T) or 3 (IQU); alm and F are arrays of nmaps pointers, host
// or device; with a registered `comm` the call is collective like sharp_execute_mpi_fortran.
void cmdr_sht_mix(int comm, int nmaps, double *const *alm, const double *const *F,
                  const sharp_geom_info *geom_T, const sharp_geom_info *geom_P,
                  const sharp_alm_info *alm_info, void *stream) {
  if (nmaps != 1 && nmaps != 3) { fprintf(stderr, "cmdr_sht_mix: nmaps %d unsupported (1 or 3)\n", nmaps); abort(); }
  cudaStream_t st = (cudaStream_t)stream;
  const sharp_alm_info *a = alm_info;
  const long long nalm_d = a->nalm * (a->real_packed ? 1 : 2);
  const long long npix = geom_T->npix;
  if (nmaps == 3 && geom_P->npix != npix) { fprintf(stderr, "cmdr_sht_mix: T and P geometries differ in size\n"); abort(); }
  bool alm_on_dev = true, f_on_dev = true;
  for (int c = 0; c < nmaps; ++c) {
    alm_on_dev = alm_on_dev && (nalm_d == 0 || is_device_ptr(alm[c]));
    f_on_dev = f_on_dev && (npix == 0 || is_device_ptr(F[c]));
  }
  double *ad[3], *md[3];
  const double *fd[3];
  double *map_buf = static_cast<double *>(scratch_get("mix_map", sizeof(double) * (size_t)std::max<long long>(1, npix) * nmaps));
  for (int c = 0; c < nmaps; ++c) md[c] = map_buf + (size_t)c * npix;
  if (alm_on_dev) {
    for (int c = 0; c < nmaps; ++c) ad[c] = alm[c];
  } else {
    double *alm_buf = static_cast<double *>(scratch_get("mix_alm", sizeof(double) * (size_t)std::max<long long>(1, nalm_d) * nmaps));
    for (int c = 0; c < nmaps; ++c) {
      ad[c] = alm_buf + (size_t)c * nalm_d;
      if (nalm_d) CMDR_CUDA_CHECK(cudaMemcpyAsync(ad[c], alm[c], sizeof(double) * nalm_d, cudaMemcpyHostToDevice, st));
    }
  }
  cudaEvent_t ef = nullptr;
  if (f_on_dev) {
    for (int c = 0; c < nmaps; ++c) fd[c] = F[c];
  } else {
    // F goes up on the copy stream while the synthesis runs
    double *f_buf = static_cast<double *>(scratch_get("mix_F", sizeof(double) * (size_t)std::max<long long>(1, npix) * nmaps));
    cudaStream_t cs = copy_stream();
    cudaEvent_t e0 = pooled_event(60);          // an earlier call on `st` may still read the buffer
    CMDR_CUDA_CHECK(cudaEventRecord(e0, st));
    CMDR_CUDA_CHECK(cudaStreamWaitEvent(cs, e0, 0));
    for (int c = 0; c < nmaps; ++c) {
      fd[c] = f_buf + (size_t)c * npix;
      if (npix) CMDR_CUDA_CHECK(cudaMemcpyAsync(f_buf + (size_t)c * npix, F[c], sizeof(double) * npix, cudaMemcpyHostToDevice, cs));
    }
    ef = pooled_event(61);
    CMDR_CUDA_CHECK(cudaEventRecord(ef, cs));
  }
  auto transform = [&](int type) {
    if (nmaps == 3) {
      cmdr_sht_execute_iqu_dist(comm, type, ad, md, geom_T, geom_P, alm_info, SHARP_DP, st);
    } else {
      cmdr_sht_execute_dist(comm, type, 0, ad, md, geom_T, alm_info, SHARP_DP, st);
    }
  };
  transform(SHARP_Y);
  if (ef) CMDR_CUDA_CHECK(cudaStreamWaitEvent(st, ef, 0));
  if (npix) {
    int nsm = 148;
    int dev = 0;
    CMDR_CUDA_CHECK(cudaGetDevice(&dev));
    CMDR_CUDA_CHECK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    for (int c = 0; c < nmaps; ++c) {
      scale_map_kernel<<<nsm * 8, 256, 0, st>>>(md[c], fd[c], npix);
      count_launch(1);
    }
    CMDR_CUDA_CHECK(cudaGetLastError());
  }
  transform(SHARP_YtW);
  if (!alm_on_dev) {
    for (int c = 0; c < nmaps; ++c)
      if (nalm_d) CMDR_CUDA_CHECK(cudaMemcpyAsync(alm[c], ad[c], sizeof(double) * nalm_d, cudaMemcpyDeviceToHost, st));
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  } else if (!f_on_dev) {
    CMDR_CUDA_CHECK(cudaStreamSynchronize(st));     // the caller may free or rewrite the host F after return
  }
}

// commander3/src/sharp.f90:96-104.  `comm` is the MPI_Fint; the group must have been
// registered (INTEGRATION.md shows the MPI_Bcast of the NCCL id the Fortran side adds).
void sharp_execute_mpi_fortran(int comm, int type, int spin, void *alm, void *map,
                               const sharp_geom_info *geom_info, const sharp_alm_info *alm_info, int flags,
                               double *time, unsigned long long *opcnt) {
  const Job job = job_or_abort("sharp_execute_mpi_fortran", type, spin, flags);
  sharp_geom_info *g = const_cast<sharp_geom_info *>(geom_info);
  sharp_alm_info *a = const_cast<sharp_alm_info *>(alm_info);
  DistComm *C = comm_or_local(comm, g, a, "sharp_execute_mpi_fortran");
  if (!C) {
    execute_any(job, alm, map, g, a, time, opcnt, (cudaStream_t)0);
    return;
  }
  auto t0 = std::chrono::steady_clock::now();
  execute_dist_any(C, &job, 1, static_cast<double *const *>(alm), static_cast<double *const *>(map), &g, a,
                   (cudaStream_t)0);
  if (time || opcnt) CMDR_CUDA_CHECK(cudaStreamSynchronize(0));
  if (time) *time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();   // wall seconds, as libsharp2 reports
  if (opcnt) *opcnt = job_opcnt(geom_info, alm_info, job);
}

}  // extern "C"
