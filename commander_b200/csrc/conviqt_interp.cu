// conviqt_interp.cu -- sampling the conviqt cube on the device: comm_conviqt%interp (commander3/src/comm_conviqt_mod.f90:
// 155-205), which the TOD sidelobe correction calls for every sample of every detector.
//
// The reference keeps the cube of ALL pixels in one node-shared MPI window (:140-141), so that any rank can interpolate
// any pixel.  The sampler is the device counterpart: a float table [2 bmax][12 nside^2] in global RING order on every
// GPU of the group, built once from the local cubes that cmdr_sht_conviqt_cube wrote:
//
//   conviqt_scatter_kernel   (pack) local cube -> float block [2 bmax][max n_pix]        (a double cube is rounded here)
//   NCCL all-gather          every rank's block, bit for bit (no reduction: -0.0 stays -0.0)
//   conviqt_scatter_kernel   each rank's rings -> their RING-scheme positions in the table
//
// conviqt_interp_kernel then evaluates one sample per thread with the reference's single-precision operations
// (conviqt_interp.cuh).  Algorithmic bytes per sample: 4 (pix) + 4 (psi) + 4 (out) + 4 per table read (1 or 2).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "conviqt_interp.cuh"
#include "kernels.h"

using namespace cmdr;

struct cmdr_conviqt_sampler {
  int device = 0, nside = 0, bmax = 0, psisteps = 0;
  long long npix = 0;
  float psires = 0.0f, twopi = 0.0f;
  float *tab = nullptr;                 // [psisteps][npix]
  unsigned long long *d_bad = nullptr;  // out-of-range pixels of the last interp call
};

namespace {

constexpr int INTERP_BLOCK = 256;

// The 2-D copy described by `runs` (conviqt_interp.cuh): one CTA per (run, row).
template <typename T>
__global__ void __launch_bounds__(256) conviqt_scatter_kernel(const CvqRun *__restrict__ runs, const T *__restrict__ src,
                                                              long long src_pitch, float *__restrict__ dst, long long dst_pitch) {
  const CvqRun r = runs[blockIdx.x];
  const long long k = blockIdx.y;
  const T *s = src + r.src + k * src_pitch;
  float *d = dst + r.dst + k * dst_pitch;
  for (int j = threadIdx.x; j < r.n; j += blockDim.x) d[j] = (float)s[j];
}

__global__ void __launch_bounds__(INTERP_BLOCK) conviqt_interp_kernel(const float *__restrict__ tab, long long npix,
                                                                       int psisteps, float psires, float twopi, int optim,
                                                                       long long n, const int *__restrict__ pix,
                                                                       const float *__restrict__ psi, float *__restrict__ out,
                                                                       unsigned long long *__restrict__ bad) {
  unsigned nbad = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int p = pix[i];
    nbad += (p < 0 || (long long)p >= npix) ? 1u : 0u;
    out[i] = conviqt_interp_sample(tab, npix, psisteps, psires, twopi, optim, p, psi[i]);
  }
  if (nbad) atomicAdd(bad, (unsigned long long)nbad);
}

template <typename T>
void launch_scatter(const std::vector<CvqRun> &runs, int nrow, const void *src, long long src_pitch, float *dst,
                    long long dst_pitch, cudaStream_t st) {
  if (runs.empty()) return;
  CvqRun *d_runs = upload(runs);
  conviqt_scatter_kernel<T><<<dim3((unsigned)runs.size(), (unsigned)nrow), 256, 0, st>>>(
      d_runs, static_cast<const T *>(src), src_pitch, dst, dst_pitch);
  CMDR_CUDA_CHECK(cudaGetLastError());
  count_launch(1);
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  cudaFree(d_runs);
}

void scatter(bool f64, const std::vector<CvqRun> &runs, int nrow, const void *src, long long src_pitch, float *dst,
             long long dst_pitch, cudaStream_t st) {
  if (f64) launch_scatter<double>(runs, nrow, src, src_pitch, dst, dst_pitch, st);
  else launch_scatter<float>(runs, nrow, src, src_pitch, dst, dst_pitch, st);
}

// all-gather of n ints per rank
std::vector<int> gather_ints(int comm, int nranks, std::vector<int> mine, int n, cudaStream_t st) {
  mine.resize(n, 0);
  int *d_in = upload(mine), *d_out = nullptr;
  CMDR_CUDA_CHECK(cudaMalloc(&d_out, sizeof(int) * (size_t)n * nranks));
  comm_allgather(comm, d_in, d_out, sizeof(int) * n, st);
  std::vector<int> all((size_t)n * nranks);
  CMDR_CUDA_CHECK(cudaMemcpyAsync(all.data(), d_out, sizeof(int) * all.size(), cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  cudaFree(d_in); cudaFree(d_out);
  return all;
}

[[noreturn]] void refuse(const std::string &why) {
  fprintf(stderr, "cmdr_sht: cmdr_sht_conviqt_sampler: %s\n", why.c_str());
  abort();
}

}  // namespace

extern "C" {

cmdr_conviqt_sampler *cmdr_sht_conviqt_sampler(int comm, int bmax, const void *cube, int cube_f64,
                                               const sharp_geom_info *geom_T, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  std::string err;
  const int nside = geom_T ? geom_T->nside : 0;
  const long long np = geom_T ? geom_T->npix : 0;
  if (!geom_T) err = "geom_T is NULL";
  else if (bmax < 1 || bmax > CMDR_MAX_SPIN) err = "bmax " + std::to_string(bmax) + " outside 1.." + std::to_string(CMDR_MAX_SPIN);
  else err = cvq_check_rings(nside, {geom_T->ring}, false);   // coverage is checked once all ranks' rings are known
  if (err.empty() && np > 0 && !cube) err = "cube is NULL";
  int rank = 0, nranks = 1;
  const bool group = comm_group(comm, rank, nranks);
  // every rank learns whether all passed the same (nside, bmax, cube_f64) and all were valid before any of them aborts
  const int code = err.empty() ? (nside * (CMDR_MAX_SPIN + 1) + bmax) * 2 + (cube_f64 ? 1 : 0) : -1;
  const bool same = comm_all_equal(comm, code, st);
  if (!err.empty()) refuse(err);
  if (!same) refuse("the ranks passed different nside, bmax or cube_f64, or one of them an invalid argument; every rank of "
                    "the communicator must make the same call");

  std::vector<std::vector<int>> rings;
  long long maxnp = np;
  if (group) {
    const std::vector<int> cnt = gather_ints(comm, nranks, {geom_T->nrings, (int)np}, 2, st);
    int maxr = 1;
    maxnp = 1;
    for (int r = 0; r < nranks; ++r) { maxr = std::max(maxr, cnt[2 * r]); maxnp = std::max<long long>(maxnp, cnt[2 * r + 1]); }
    const std::vector<int> all = gather_ints(comm, nranks, geom_T->ring, maxr, st);
    for (int r = 0; r < nranks; ++r) rings.emplace_back(all.begin() + (size_t)r * maxr, all.begin() + (size_t)r * maxr + cnt[2 * r]);
  } else {
    rings.push_back(geom_T->ring);
  }
  err = cvq_check_rings(nside, rings, true);
  if (!err.empty()) {
    if (!group)
      err = "communicator " + std::to_string(comm) + " is not a registered group of several ranks, so geom_T must hold the "
            "whole sphere: " + err;
    refuse(err);
  }

  cmdr_conviqt_sampler *s = new cmdr_conviqt_sampler;
  CMDR_CUDA_CHECK(cudaGetDevice(&s->device));
  s->nside = nside; s->bmax = bmax; s->psisteps = 2 * bmax;
  s->npix = 12LL * nside * nside;
  s->psires = cvq_psires(s->psisteps);
  s->twopi = cvq_twopi();
  const int nrow = s->psisteps;
  CMDR_CUDA_CHECK(cudaMalloc(&s->tab, sizeof(float) * (size_t)nrow * s->npix));
  CMDR_CUDA_CHECK(cudaMalloc(&s->d_bad, sizeof(unsigned long long)));

  // this rank's cube on the device
  const size_t esz = cube_f64 ? sizeof(double) : sizeof(float);
  const void *cd = cube;
  void *staged = nullptr;
  if (np > 0 && !is_device_ptr(cube)) {
    CMDR_CUDA_CHECK(cudaMalloc(&staged, esz * (size_t)nrow * np));
    CMDR_CUDA_CHECK(cudaMemcpyAsync(staged, cube, esz * (size_t)nrow * np, cudaMemcpyHostToDevice, st));
    cd = staged;
  }
  if (!group) {
    scatter(cube_f64, cvq_scatter_runs(nside, rings, 0), nrow, cd, np, s->tab, s->npix, st);
  } else {
    float *send = nullptr, *recv = nullptr;
    CMDR_CUDA_CHECK(cudaMalloc(&send, sizeof(float) * (size_t)nrow * maxnp));
    CMDR_CUDA_CHECK(cudaMalloc(&recv, sizeof(float) * (size_t)nrow * maxnp * nranks));
    std::vector<CvqRun> pack;
    cvq_add_runs(pack, 0, 0, np);
    scatter(cube_f64, pack, nrow, cd, np, send, maxnp, st);
    comm_allgather(comm, send, recv, sizeof(float) * (size_t)nrow * maxnp, st);
    scatter(false, cvq_scatter_runs(nside, rings, (long long)nrow * maxnp), nrow, recv, maxnp, s->tab, s->npix, st);
    cudaFree(send); cudaFree(recv);
  }
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  if (staged) cudaFree(staged);
  return s;
}

long long cmdr_sht_conviqt_interp(const cmdr_conviqt_sampler *s, long long nsamp, const int *pix, const float *psi,
                                  int optim, float *out, void *stream) {
  if (!s) { fprintf(stderr, "cmdr_sht: cmdr_sht_conviqt_interp: sampler is NULL\n"); abort(); }
  if (nsamp < 0 || (nsamp > 0 && (!pix || !psi || !out))) {
    fprintf(stderr, "cmdr_sht: cmdr_sht_conviqt_interp: nsamp %lld with a NULL array, or negative\n", nsamp);
    abort();
  }
  int dev = 0;
  CMDR_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev != s->device) {
    fprintf(stderr, "cmdr_sht: cmdr_sht_conviqt_interp: the sampler lives on device %d, the current device is %d\n",
            s->device, dev);
    abort();
  }
  if (nsamp == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)nsamp;
  const int *pd = pix;
  const float *qd = psi;
  float *od = out;
  if (!is_device_ptr(pix)) {
    int *b = static_cast<int *>(scratch_get("cvq_pix", sizeof(int) * n));
    CMDR_CUDA_CHECK(cudaMemcpyAsync(b, pix, sizeof(int) * n, cudaMemcpyHostToDevice, st));
    pd = b;
  }
  if (!is_device_ptr(psi)) {
    float *b = static_cast<float *>(scratch_get("cvq_psi", sizeof(float) * n));
    CMDR_CUDA_CHECK(cudaMemcpyAsync(b, psi, sizeof(float) * n, cudaMemcpyHostToDevice, st));
    qd = b;
  }
  const bool out_host = !is_device_ptr(out);
  if (out_host) od = static_cast<float *>(scratch_get("cvq_out", sizeof(float) * n));
  CMDR_CUDA_CHECK(cudaMemsetAsync(s->d_bad, 0, sizeof(unsigned long long), st));
  const long long blocks = std::min<long long>((nsamp + INTERP_BLOCK - 1) / INTERP_BLOCK, 1LL << 30);
  conviqt_interp_kernel<<<(unsigned)blocks, INTERP_BLOCK, 0, st>>>(s->tab, s->npix, s->psisteps, s->psires, s->twopi, optim,
                                                                   nsamp, pd, qd, od, s->d_bad);
  CMDR_CUDA_CHECK(cudaGetLastError());
  count_launch(1);
  if (out_host) CMDR_CUDA_CHECK(cudaMemcpyAsync(out, od, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
  unsigned long long bad = 0;
  CMDR_CUDA_CHECK(cudaMemcpyAsync(&bad, s->d_bad, sizeof(bad), cudaMemcpyDeviceToHost, st));
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));
  return (long long)bad;
}

void cmdr_sht_conviqt_sampler_destroy(cmdr_conviqt_sampler *s) {
  if (!s) return;
  cudaFree(s->tab);
  cudaFree(s->d_bad);
  delete s;
}

}  // extern "C"
