// legendre.cu -- hand-written sm_100a FP64 Legendre / Wigner-d kernels.
//
// Replaces the Legendre stage of libsharp2's sharp_execute (reached from
// commander3/src/sharp.f90:226-240) for the job types of commander3/src/sharp.f90:8-14:
//   synthesis (SHARP_Y, SHARP_WY):   ph[m][ring] = sum_l a_lm lambda_lm(theta_ring)
//   analysis  (SHARP_Yt, SHARP_YtW): a_lm       = sum_ring lambda_lm(theta_ring) ph[m][ring]
// for spin 0 (T), spin 2 (Q,U <-> E,B; HEALPix "COSMO" convention,
// commander3/src/comm_map_mod.f90:1002) and any other spin up to CMDR_MAX_SPIN
// (commander3/src/comm_conviqt_mod.f90:234-239).
//
// Work decomposition: grid = (ring-pair chunks, local m), ONE WARP PER CTA, no block-level
// synchronisation.  A thread owns R adjacent ring pairs (spin-2 analysis: 32 apart; north ring + its southern mirror
// share one recurrence through the l+m parity), runs the recurrence in registers over l, and
// reads per-l data (recurrence coefficients and, for synthesis, the pre-scaled a_lm) as
// warp-uniform broadcasts from a shared-memory tile of TL consecutive l that the warp stages
// itself with cp.async.  FP64-pipe cost per (l, m, ring pair):
//   spin 0: 1 (recurrence) + 2 (accumulate) -- two l per step, recurrence in x^2 (coef.cpp) ; spin s: 4 + 8.
// Spin 2 runs that scalar recurrence too while every ring of a warp is still far below the accumulation threshold
// (1 instead of 4 per l and ring pair) and converts to the two spin-2 recurrences at the hand-over (spin2_front_phase).
// On one GPU, spin 2 runs as two scalar sums of premixed coefficients everywhere but near the poles (launch_s2s_*).
// Analysis reduces over the rings of the warp with a select-free, software-pipelined register
// butterfly and adds the sums to the a_lm with coalesced atomics (DESIGN.md 3.1).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <tuple>

#include "det.h"
#include "kernels.h"
#include "legendre_core.cuh"

namespace cmdr {

constexpr int TL = 128;    // l per shared-memory tile (per warp, double buffered)
constexpr unsigned FULL = 0xffffffffu;
constexpr double SCALE_DOWN = 7.458340731200207e-155;   // 2^-512

static_assert(SCALE_BITS == 512, "SCALE_DOWN must equal 2^-SCALE_BITS");

struct KParams {
  int lmax, nm, real_packed;
  int spin;          // 0, or s >= 1 for the two-component kernels
  double spinsign;   // sign of (+s)a = spinsign (E + iB): -1 for even s (HEALPix COSMO for s = 2), +1 for odd s
  int nslots, NPL, NML, ncomp_tot, comp0;
  int ring_major;    // phase layout inside a block (kernels.h: ph_index)
  int slot_begin;   // first slot handled by this launch (nslots = one past the last)
  int im0;          // first local m handled by this launch (grid.y counts from it)
  const int *mval;
  const long long *mvstart;
  const double *coef;
  const double *coef2;               // spin 0: mix rows {u_j, v_j, h_j, v_{j-1}} of the two-l-per-step scheme (coef.cpp)
  const long long *cofs;
  const double *Kstart;
  // spin 2 only: scalar tables for the front phase (spin2_front_phase); fcoef == nullptr disables it
  const double *fcoef, *fmix, *fK0;   // rec rows {a_j, b'_j}, mix rows {u, v, h, v_prev}, spin-0 start norms
  const long long *fcofs;
  const long long *tofs;             // synthesis: first tile row of each local m (rows padded to 8 per m)
  double *trows;                     // synthesis: tile rows (TileS0<NC> / TileS2), written by the prep kernels
  const double *trig;
  const int *mlim;
  const int *wslot;                  // work index -> storage slot (nullptr: identity)
  // spin-0 kernels running a spin-2 job as scalar sums (launch_s2s_*; -1: off): the phases are scaled by 1 / sin^2 on
  // store (synthesis, synth0_kernel<2, ...>) or load (analysis), the slots below this one are left to the spin-2 kernels
  // (analysis: weight 0), and the analysis writes the unnormalised sums per (m, l) into a scratch buffer laid out like the coefficient table
  int s2s_npolar;
  // seeded kernels only (seed tables, see seed0_kernel / seed2_kernel): first row (spin 0) / l - l0 (spin 2) each warp
  // accumulates at, per (local m, warp); recurrence state and scale exponent there, per (local m, slot)
  const int *sl;
  const double *ss;
  const int *sk;
  double *alm0, *alm1;
  const double *lscale0, *lscale1;   // optional factor per l on component 0 / 1 (nullptr: 1)
  double4 *ph;
  int src_rank;                      // fused exchange: block of this rank in the ring owners' buffers (-1: local buffer, block = owner)
  double4 *peer[CMDR_MAX_PEERS];     // phase buffer of each ring owner (all = ph without the fused exchange)
};

// Partials buffer (component 0 at det), records and their layout of the deterministic analysis kernels (det.h): a
// parameter of its own, so that KParams and the kernels that do not use it keep their parameter layout
struct DetArgs {
  double *det = nullptr;
  int *drec = nullptr;
  DetLayout dl;
};

// one row = two l (l_j = m + 2j, l_j + 1): the shared recurrence coefficients and {c1r, c1i, c2r, c2i} of each of NC
// components (1: T; 2: Q and U of a spin-2 job run as scalar sums)
template <int NC>
struct __align__(16) TileS0 { double A, B, c[NC][4]; };
struct __align__(16) TileS2 { double A, C, cpr, cpi, cmr, cmi; };
struct __align__(16) TileA0 { double A, B; };
struct __align__(16) TileA2 { double A, C, g, pad; };

// analysis input: blocks indexed by the rank that owns the rings in the local buffer; with the
// fused exchange the block of THIS rank in the ring owner's buffer, read over NVLink
__device__ __forceinline__ const double4 *ph_in(const KParams &p, int comp, int im, int work) {
  const int slot = p.wslot ? p.wslot[work] : work;
  int owner = slot / p.NPL, local = slot - owner * p.NPL;
  const int blk = p.src_rank >= 0 ? p.src_rank : owner;
  return p.peer[owner] + ph_index(blk, p.ncomp_tot, p.comp0 + comp, p.NML, p.NPL, im, local, p.ring_major);
}
// synthesis output: the ring owner's buffer (its own on one GPU, peer-mapped over NVLink
// otherwise), block of the writing rank
__device__ __forceinline__ double4 *ph_out(const KParams &p, int comp, int im, int work) {
  const int slot = p.wslot ? p.wslot[work] : work;
  int owner = slot / p.NPL, local = slot - owner * p.NPL;
  const int blk = p.src_rank >= 0 ? p.src_rank : owner;
  return p.peer[owner] + ph_index(blk, p.ncomp_tot, p.comp0 + comp, p.NML, p.NPL, im, local, p.ring_major);
}

// Spin-2 analysis only: ring pair r of lane `lane` is slot chunk0 + 32 r + lane, so that the 32 ring pairs with the same r
// (a "slice") are neighbours in colatitude and cross the accumulation threshold together; in the transient phase (some
// rings on, some not) the accumulate FMAs of a slice none of whose rings is on yet are skipped with a warp-uniform test:
// bit r of the mask (anal2 28.31 -> 27.88 ms).  The other three kernels keep R adjacent ring pairs per thread and the
// default mask: the same change cost them registers (synth2 162 -> 226) and made them slower.
template <int R>
__device__ __forceinline__ unsigned slices_on(const int (&k)[R]) {
  unsigned m = 0;
#pragma unroll
  for (int r = 0; r < R; ++r)
    if (__any_sync(FULL, k[r] == 0)) m |= 1u << r;
  return m;
}

// 16-byte asynchronous global -> shared copies (LDGSTS): every kernel stages its per-l
// tiles as raw rows of a global table (coefficient tables for analysis, the pre-scaled a_lm rows
// written by the prep kernels for synthesis), so staging needs no registers and no barrier.
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
  unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// ------------------------------------------------------------------------------------
// spin-0 synthesis, two l per recurrence step (coef.cpp, fill_spin0_x2):
//   nu_{j+1} = (A_j x^2 + B_j) nu_j - nu_{j-1};  sum_l a_l lam_l = sum_j nu_j c1_j + x sum_j nu_j c2_j
//   c1_j = u_j a_{l_j} + v_j a_{l_j+2} (even l - m),  c2_j = h_j a_{l_j+1} (odd l - m);  south ring: x -> -x.
// One group = 4 rows = 8 l.  NC components share the recurrence: each row's nu feeds 4 NC accumulate FMAs, and every
// component's chain is the same fma sequence whatever NC and R are.
// ------------------------------------------------------------------------------------
template <int MODE, int NC, int R>
__device__ __forceinline__ void synth0_group(const TileS0<NC> *t, const double (&x2)[R], double (&cur)[R],
                                             double (&prev)[R], double (&acc)[NC][4][R], int (&k)[R]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double A = t[j].A, B = t[j].B;
    double c[NC][4];
#pragma unroll
    for (int n = 0; n < NC; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) c[n][i] = t[j].c[n][i];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (MODE != 0) {
        double v = (MODE == 2 || k[r] == 0) ? cur[r] : 0.0;
#pragma unroll
        for (int n = 0; n < NC; ++n)
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[n][i][r] = fma(v, c[n][i], acc[n][i][r]);
      }
      double nxt = step0x2(A, B, x2[r], cur[r], prev[r]);
      prev[r] = cur[r]; cur[r] = nxt;
    }
  }
  if (MODE < 2) {
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (k[r] < 0 && needs_rescale(cur[r])) { cur[r] *= SCALE_DOWN; prev[r] *= SCALE_DOWN; ++k[r]; }
  }
}

// Tile rows for synthesis: {A_j, B_j, c1_j, c2_j} per (m, j), written once per transform by a prep kernel so
// that every warp of the Legendre kernel can stage them with plain asynchronous copies.  Rows of one
// m are padded with zero rows to a multiple of 8 (the kernels walk the rows in groups of 4).
__global__ void __launch_bounds__(256) prep_s0_kernel(KParams p) {
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int j = blockIdx.x * blockDim.x + threadIdx.x, l = m + 2 * j;
  const int J = p.lmax >= m ? (p.lmax - m) / 2 + 1 : 0;
  const int npad = (J + 7) & ~7;
  if (j >= npad) return;
  TileS0<1> e{0.0, 0.0, {{0.0, 0.0, 0.0, 0.0}}};
  if (j < J) {
    const double2 rc = reinterpret_cast<const double2 *>(p.coef + p.cofs[im])[j];        // {A_j, B_j}
    const double4 mx = reinterpret_cast<const double4 *>(p.coef2 + 2 * p.cofs[im])[j];   // {u_j, v_j, h_j, v_{j-1}}
    const double *a = p.alm0;
    const long long mvs = p.mvstart[im];
    const double nrm = (p.real_packed && m > 0) ? 0.70710678118654752440 : 1.0;
    auto load = [&](int ll, double &re, double &imv) {
      re = 0.0; imv = 0.0;
      if (ll > p.lmax) return;
      const double f = p.lscale0 ? nrm * p.lscale0[ll] : nrm;
      if (p.real_packed) {
        if (m == 0) re = f * a[mvs + ll];
        else { re = f * a[mvs + 2 * (long long)ll]; imv = f * a[mvs + 2 * (long long)ll + 1]; }
      } else {
        re = f * a[2 * (mvs + ll)];
        if (m > 0) imv = f * a[2 * (mvs + ll) + 1];
      }
    };
    double r0, i0, r1, i1, r2, i2;
    load(l, r0, i0); load(l + 1, r1, i1); load(l + 2, r2, i2);
    e.A = rc.x; e.B = rc.y;
    e.c[0][0] = fma(mx.x, r0, mx.y * r2); e.c[0][1] = fma(mx.x, i0, mx.y * i2);
    e.c[0][2] = mx.z * r1; e.c[0][3] = mx.z * i1;
  }
  reinterpret_cast<TileS0<1> *>(p.trows)[p.tofs[im] + j] = e;
}

// Synthesis kernels: ONE WARP PER CTA like the analysis kernels (no block barriers; a thread owns R
// adjacent ring pairs; whole warps beyond the m cut-off only write zeros).
// SEED: start each ring from the seed table at the warp's first accumulating row instead of from the closed-form start
// values at row 0 (the rows in between add exact zeros; seed0_kernel).
// NC = 2 runs a spin-2 job as scalar sums (launch_s2s_synth): components comp0 and comp0 + 1, phases scaled by
// 1 / sin^2 on store (sum d lam = sin^2 x the spin-2 sum).  Its 80-byte rows take tiles of TL_S2S rows: 2 x 128 rows
// would be 20 KB of shared memory per one-warp CTA, 10 CTAs per SM instead of the 12 the 160 registers allow
// (measured: 64 and 96 rows alike, 128 rows 1.3 % and 32 rows 0.6 % slower).
constexpr int TL_S2S = 64;
template <int NC, int R, int MINB, bool SEED = false>
__global__ void __launch_bounds__(32, MINB) synth0_kernel(KParams p) {
  constexpr int TLN = NC == 1 ? TL : TL_S2S;
  static_assert(TLN * sizeof(TileS0<NC>) % 512 == 0, "a tile is staged in whole 16-byte copies of the warp");
  __shared__ __align__(16) TileS0<NC> tile[2][TLN];
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int lane = threadIdx.x;
  const int chunk0 = p.slot_begin + blockIdx.x * (32 * R);
  const int J = p.lmax >= m ? (p.lmax - m) / 2 + 1 : 0;   // rows (steps of two l) of this m
  double x[R], x2[R], cur[R], prev[R], acc[NC][4][R];
  int k[R], slot[R];
  bool any = false;
  const double K = p.Kstart[m];
  const int j0 = SEED ? p.sl[(size_t)im * gridDim.x + blockIdx.x] : 0;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    slot[r] = chunk0 + lane * R + r;
    bool valid = slot[r] < p.nslots && m <= p.mlim[min(slot[r], p.nslots - 1)];
#pragma unroll
    for (int n = 0; n < NC; ++n) acc[n][0][r] = acc[n][1][r] = acc[n][2][r] = acc[n][3][r] = 0.0;
    prev[r] = 0.0; cur[r] = 0.0; k[r] = 0; x[r] = 0.0; x2[r] = 0.0;
    if (valid) {
      const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot[r]];
      RingTrig g{tg.x, tg.y, tg.z, tg.w};
      x[r] = g.cth; x2[r] = g.cth * g.cth;
      if constexpr (SEED) {
        const size_t s = (size_t)im * p.nslots + slot[r];
        const double2 st = reinterpret_cast<const double2 *>(p.ss)[s];
        cur[r] = st.x; prev[r] = st.y; k[r] = p.sk[s];
      } else {
        start_spin0(m, K, g, cur[r], k[r]);
      }
      any = true;
    }
  }
  if (__any_sync(FULL, any) && (!SEED || j0 < J)) {
    const TileS0<NC> *rows = reinterpret_cast<const TileS0<NC> *>(p.trows) + p.tofs[im];
    auto issue_tile = [&](int b, int jt) {     // rows past this m's padded range are never used
      const char *src = reinterpret_cast<const char *>(rows + jt);
      char *dst = reinterpret_cast<char *>(tile[b]);
#pragma unroll
      for (int q = 0; q < (int)(TLN * sizeof(TileS0<NC>)) / 512; ++q) cp_async16(dst + (q * 32 + lane) * 16, src + (q * 32 + lane) * 16);
      cp_async_commit();
    };
    issue_tile(0, j0);
    cp_async_wait_all();
    __syncwarp();
    int buf = 0;
    for (int jt = j0; jt < J; jt += TLN, buf ^= 1) {
      if (jt + TLN < J) issue_tile(buf ^ 1, jt + TLN);
      const int ngroups = min(TLN, J - jt + 3) / 4;
#pragma unroll 1
      for (int g = 0; g < ngroups; ++g) {
        bool all_on = true, none_on = true;
#pragma unroll
        for (int r = 0; r < R; ++r) { all_on &= (k[r] == 0); none_on &= (k[r] < 0); }
        if (__all_sync(FULL, all_on)) synth0_group<2, NC, R>(tile[buf] + 4 * g, x2, cur, prev, acc, k);
        else if (__all_sync(FULL, none_on)) synth0_group<0, NC, R>(tile[buf] + 4 * g, x2, cur, prev, acc, k);
        else synth0_group<1, NC, R>(tile[buf] + 4 * g, x2, cur, prev, acc, k);
      }
      cp_async_wait_all();
      __syncwarp();
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r)
    if (slot[r] < p.nslots) {
      double f = 1.0;
      if constexpr (NC == 2) {
        const double s = reinterpret_cast<const double4 *>(p.trig)[slot[r]].y;
        f = 1.0 / (s * s);
      }
#pragma unroll
      for (int n = 0; n < NC; ++n) {
        const double per = acc[n][0][r], pei = acc[n][1][r], por = acc[n][2][r], poi = acc[n][3][r];
        double4 v = make_double4(fma(x[r], por, per), fma(x[r], poi, pei), fma(-x[r], por, per), fma(-x[r], poi, pei));
        if constexpr (NC == 2) { v.x *= f; v.y *= f; v.z *= f; v.w *= f; }
        *ph_out(p, n, im, slot[r]) = v;
      }
    }
}

// ------------------------------------------------------------------------------------
// Scalar front phase of the spin-2 kernels (legendre_core.cuh, "spin 2 seeded from the scalar recurrence").  While no
// ring of the warp is within FRONT_MARGIN_BITS of the accumulation threshold the warp advances the scalar
// two-l-per-step recurrence (1 FP64 op per l and ring pair) instead of the two spin-2 recurrences (4); the first ring
// to get there switches the whole warp.  Used when every valid ring of the warp starts below the threshold and has
// sin(theta) >= FRONT_MIN_STH (nearer to the poles the smaller of the two spin-2 functions would be seeded with too
// few digits: tests/test_host.py test_spin2_scalar_front_on_host).
// ------------------------------------------------------------------------------------
constexpr double FRONT_MIN_STH = 0.15;
constexpr int FRONT_TR = 8;          // rows (of two l) between the snapshots at which the front phase can hand over

// Rows of two l are advanced GR at a time; the hand-over happens at a multiple of TR rows (= one shared-memory tile of
// the caller's l loop, so that the caller simply starts its tile loop later and nothing else in it changes -- the
// kernels sit at their register limit, and every extra value live across the steady-state loop costs spills there):
// the state at the last tile boundary is kept and restored when a ring triggers inside the tile (those rows are then
// redone by the spin-2 recurrences).  nu / nup: scalar state on entry (start_spin0) and exit; returns the rows done.
template <int R, int GR, int TR>
__device__ __forceinline__ int spin2_front_phase(const KParams &p, int im, int m, unsigned vmask, const double (&x)[R],
                                                 const int (&mg)[R], double (&nu)[R], double (&nup)[R], int (&k)[R]) {
  const double2 *rec = reinterpret_cast<const double2 *>(p.fcoef + p.fcofs[im]);
  const int J = (p.lmax - m) / 2 + 1;
  double x2[R], snu[R], snup[R];
  int sk[R];
#pragma unroll
  for (int r = 0; r < R; ++r) x2[r] = x[r] * x[r];
  int jb = 0;
#pragma unroll 1
  for (;;) {                                    // one tile of TR rows per iteration
#pragma unroll
    for (int r = 0; r < R; ++r) { snu[r] = nu[r]; snup[r] = nup[r]; sk[r] = k[r]; }
    bool stop = jb + TR > J - 1;                // the hand-over row and the one after it must exist
    double2 rc[GR];
#pragma unroll
    for (int q = 0; q < GR; ++q) rc[q] = rec[jb + q];          // (the table is zero padded past the last row)
#pragma unroll 1
    for (int j = jb; !stop && j < jb + TR; j += GR) {
      bool sw = false;
#pragma unroll
      for (int r = 0; r < R; ++r) sw |= ((vmask >> r) & 1) && front_must_switch(nu[r], k[r], mg[r]);
      if (__any_sync(FULL, sw)) { stop = true; break; }
      double2 nx[GR];
#pragma unroll
      for (int q = 0; q < GR; ++q) nx[q] = rec[j + GR + q];
#pragma unroll
      for (int q = 0; q < GR; ++q)
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const double nxt = step0x2(rc[q].x, rc[q].y, x2[r], nu[r], nup[r]);
          nup[r] = nu[r]; nu[r] = nxt;
        }
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (k[r] < 0 && needs_rescale(nu[r])) { nu[r] *= SCALE_DOWN; nup[r] *= SCALE_DOWN; ++k[r]; }
#pragma unroll
      for (int q = 0; q < GR; ++q) rc[q] = nx[q];
    }
    if (stop) {                                 // back to the tile boundary
#pragma unroll
      for (int r = 0; r < R; ++r) { nu[r] = snu[r]; nup[r] = snup[r]; k[r] = sk[r]; }
      return jb;
    }
    jb += TR;
  }
}
// conversion of one ring at row jb (l_b = m + 2 jb): spin-2 state in kernel normalisation
__device__ __forceinline__ void spin2_front_finish(const KParams &p, int im, int m, int jb, double x, double sth, double nu, double nup,
                                                   double &P, double &Pp, double &M, double &Mp) {
  const double4 *mix = reinterpret_cast<const double4 *>(p.fmix + 2 * p.fcofs[im]);
  const double4 mb = mix[jb];
  const double mixb[4] = {mb.x, mb.y, mb.z, mb.w};
  const double hprev = jb > 0 ? mix[jb - 1].z : 0.0;
  const double *c0 = p.coef + p.cofs[im] + 4 * (size_t)(2 * jb);   // l0 = m (m >= 2): row l_b - l0 = 2 jb; the table is zero padded
  const double4 r0 = reinterpret_cast<const double4 *>(c0)[0], r1 = reinterpret_cast<const double4 *>(c0)[1];
  const double cc0[4] = {r0.x, r0.y, r0.z, r0.w}, cc1[4] = {r1.x, r1.y, r1.z, r1.w};
  spin2_front_convert(m + 2 * jb, m, p.lmax, x, sth, nu, nup, mixb, hprev, cc0, cc1, P, Pp, M, Mp);
}

// ------------------------------------------------------------------------------------
// spin-2 synthesis.  cp = -(E+iB) g, cm = -(E-iB) g;  P,M = mu of (+2)lambda, (-2)lambda.
//   a1 = sum cp P, a2 = sum cm M (north);  a3 = sum sg cp M, a4 = sum sg cm P (south)
//   Q = (a1+a2)/2, U = -i (a1-a2)/2
// ------------------------------------------------------------------------------------
template <int MODE, int R>
__device__ __forceinline__ void synth2_group(const TileS2 *t, const double (&x)[R], double (&P)[R],
                                             double (&Pp)[R], double (&M)[R], double (&Mp)[R],
                                             double (&a)[R][8], int (&k)[R], unsigned ron = ~0u) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const double A = t[j].A, C = t[j].C;
    const double cpr = t[j].cpr, cpi = t[j].cpi, cmr = t[j].cmr, cmi = t[j].cmi;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (MODE == 2 || (MODE == 1 && ((ron >> r) & 1))) {
        bool on = (MODE == 2 || k[r] == 0);
        double vp = on ? P[r] : 0.0, vm = on ? M[r] : 0.0;
        a[r][0] = fma(vp, cpr, a[r][0]); a[r][1] = fma(vp, cpi, a[r][1]);
        a[r][2] = fma(vm, cmr, a[r][2]); a[r][3] = fma(vm, cmi, a[r][3]);
        if (j & 1) {
          a[r][4] = fma(-vm, cpr, a[r][4]); a[r][5] = fma(-vm, cpi, a[r][5]);
          a[r][6] = fma(-vp, cmr, a[r][6]); a[r][7] = fma(-vp, cmi, a[r][7]);
        } else {
          a[r][4] = fma(vm, cpr, a[r][4]); a[r][5] = fma(vm, cpi, a[r][5]);
          a[r][6] = fma(vp, cmr, a[r][6]); a[r][7] = fma(vp, cmi, a[r][7]);
        }
      }
      double up = fma(A, x[r], C), um = fma(A, x[r], -C);
      double np_ = fma(up, P[r], -Pp[r]), nm_ = fma(um, M[r], -Mp[r]);
      Pp[r] = P[r]; P[r] = np_; Mp[r] = M[r]; M[r] = nm_;
    }
  }
  if (MODE < 2) {
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (k[r] < 0 && (needs_rescale(P[r]) || needs_rescale(M[r]))) {
        P[r] *= SCALE_DOWN; Pp[r] *= SCALE_DOWN; M[r] *= SCALE_DOWN; Mp[r] *= SCALE_DOWN; ++k[r];
      }
  }
}

__global__ void __launch_bounds__(256) prep_s2_kernel(KParams p) {
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int l0 = max(m, p.spin);
  const int j = blockIdx.x * blockDim.x + threadIdx.x, l = l0 + j;
  const int npad = l0 <= p.lmax ? (p.lmax - l0 + 1 + 7) & ~7 : 0;
  if (j >= npad) return;
  TileS2 e{0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (l <= p.lmax) {
    const double *coef = p.coef + p.cofs[im];
    const double *aE = p.alm0, *aB = p.alm1;
    const long long mvs = p.mvstart[im];
    const double nrm = (p.real_packed && m > 0) ? 0.70710678118654752440 : 1.0;
    double4 c = reinterpret_cast<const double4 *>(coef)[l - l0];   // {A', C', g, 0}
    double gs = c.z * nrm;
    e.A = c.x; e.C = c.y;
    double er, ei = 0.0, br, bi = 0.0;
    if (p.real_packed) {
      if (m == 0) { er = aE[mvs + l]; br = aB[mvs + l]; }
      else {
        er = aE[mvs + 2 * (long long)l]; ei = aE[mvs + 2 * (long long)l + 1];
        br = aB[mvs + 2 * (long long)l]; bi = aB[mvs + 2 * (long long)l + 1];
      }
    } else {
      er = aE[2 * (mvs + l)]; br = aB[2 * (mvs + l)];
      if (m > 0) { ei = aE[2 * (mvs + l) + 1]; bi = aB[2 * (mvs + l) + 1]; }
    }
    if (p.lscale0) { const double f = p.lscale0[l]; er *= f; ei *= f; }
    if (p.lscale1) { const double f = p.lscale1[l]; br *= f; bi *= f; }
    // (+s)a = spinsign (E + iB), (-s)a = spinsign (-1)^s (E - iB) = -(E - iB); spinsign = -1 for even s
    const double sgs = p.spinsign * gs;
    e.cpr = sgs * (er - bi); e.cpi = sgs * (ei + br);
    e.cmr = -gs * (er + bi); e.cmi = -gs * (ei - br);
  }
  reinterpret_cast<TileS2 *>(p.trows)[p.tofs[im] + j] = e;
}

template <int R, int MINB, bool SEED = false>
__global__ void __launch_bounds__(32, MINB) synth2_kernel(KParams p) {
  __shared__ __align__(16) TileS2 tile[2][TL];
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int lane = threadIdx.x;
  const int chunk0 = p.slot_begin + blockIdx.x * (32 * R);
  const int l0 = max(m, p.spin);
  double x[R], P[R], Pp[R], M[R], Mp[R], a[R][8];
  int k[R], slot[R];
  bool any = false;
  const double K = p.Kstart[m];
  // scalar front phase (spin 2, m >= 4): eligible when every valid ring of the warp starts below the threshold and
  // is not too close to a pole; P / Pp hold the scalar state until the conversion
  unsigned vmask = 0;
  int mg[R];
  bool front = !SEED && p.fcoef != nullptr && m >= 4 && l0 <= p.lmax, fok = true;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    slot[r] = chunk0 + lane * R + r;
    bool valid = slot[r] < p.nslots && m <= p.mlim[min(slot[r], p.nslots - 1)] && l0 <= p.lmax;
#pragma unroll
    for (int q = 0; q < 8; ++q) a[r][q] = 0.0;
    P[r] = M[r] = Pp[r] = Mp[r] = 0.0; k[r] = 0; x[r] = 0.0; mg[r] = 0;
    if (valid) {
      const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot[r]];
      RingTrig g{tg.x, tg.y, tg.z, tg.w};
      x[r] = g.cth;
      vmask |= 1u << r;
      if constexpr (SEED) {
        const size_t s = (size_t)im * p.nslots + slot[r];
        const double4 st = reinterpret_cast<const double4 *>(p.ss)[s];
        P[r] = st.x; Pp[r] = st.y; M[r] = st.z; Mp[r] = st.w; k[r] = p.sk[s];
      } else {
        mg[r] = front_margin_bits(g.sth);
        if (front) { start_spin0(m, p.fK0[m], g, P[r], k[r]); fok &= k[r] < 0 && g.sth >= FRONT_MIN_STH; }
      }
      any = true;
    }
  }
  front = front && __all_sync(FULL, fok);
  // l (counted from l0) the front phase has covered (whole tiles), or where the seed table starts the warp
  int lskip = SEED ? p.sl[(size_t)im * gridDim.x + blockIdx.x] : 0;
  if (__any_sync(FULL, any) && (!SEED || l0 + lskip <= p.lmax)) {
    if (front) {
      const int jb = spin2_front_phase<R, 4, FRONT_TR>(p, im, m, vmask, x, mg, P, Pp, k);
      lskip = 2 * jb;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const double nu = P[r], nup = Pp[r];
        P[r] = Pp[r] = 0.0;
        if ((vmask >> r) & 1) {
          const double sth = reinterpret_cast<const double4 *>(p.trig)[slot[r]].y;
          spin2_front_finish(p, im, m, jb, x[r], sth, nu, nup, P[r], Pp[r], M[r], Mp[r]);
        } else k[r] = 0;
      }
    } else if (!SEED) {
#pragma unroll
      for (int r = 0; r < R; ++r)
        if ((vmask >> r) & 1) {
          const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot[r]];
          RingTrig g{tg.x, tg.y, tg.z, tg.w};
          if (p.spin == 2) start_spin2(m, K, g, P[r], M[r], k[r]); else start_spin_s(m, p.spin, K, g, P[r], M[r], k[r]);
        }
    }
    const TileS2 *rows = reinterpret_cast<const TileS2 *>(p.trows) + p.tofs[im];
    auto issue_tile = [&](int b, int lt) {     // rows past this m's padded range are never used
      const char *src = reinterpret_cast<const char *>(rows + (lt - l0));
      char *dst = reinterpret_cast<char *>(tile[b]);
#pragma unroll
      for (int q = 0; q < (int)(TL * sizeof(TileS2)) / 512; ++q) cp_async16(dst + (q * 32 + lane) * 16, src + (q * 32 + lane) * 16);
      cp_async_commit();
    };
    issue_tile(0, l0 + lskip);
    cp_async_wait_all();
    __syncwarp();
    int buf = 0;
    for (int lt = l0 + lskip; lt <= p.lmax; lt += TL, buf ^= 1) {
      if (lt + TL <= p.lmax) issue_tile(buf ^ 1, lt + TL);
      const int ngroups = min(TL, p.lmax - lt + 8) / 8;
#pragma unroll 1
      for (int g = 0; g < ngroups; ++g) {
        bool all_on = true, none_on = true;
#pragma unroll
        for (int r = 0; r < R; ++r) { all_on &= (k[r] == 0); none_on &= (k[r] < 0); }
        if (__all_sync(FULL, all_on)) synth2_group<2, R>(tile[buf] + 8 * g, x, P, Pp, M, Mp, a, k);
        else if (__all_sync(FULL, none_on)) synth2_group<0, R>(tile[buf] + 8 * g, x, P, Pp, M, Mp, a, k);
        else synth2_group<1, R>(tile[buf] + 8 * g, x, P, Pp, M, Mp, a, k);
      }
      cp_async_wait_all();
      __syncwarp();
    }
  }
  // sg_l = (-1)^(l+m+2) = sg0 * (-1)^(l-l0)
  const double sg0 = ((l0 + m) & 1) ? -0.5 : 0.5;
#pragma unroll
  for (int r = 0; r < R; ++r)
    if (slot[r] < p.nslots) {
      double4 q, u;
      q.x = 0.5 * (a[r][0] + a[r][2]);  q.y = 0.5 * (a[r][1] + a[r][3]);
      u.x = 0.5 * (a[r][1] - a[r][3]);  u.y = -0.5 * (a[r][0] - a[r][2]);
      q.z = sg0 * (a[r][4] + a[r][6]);  q.w = sg0 * (a[r][5] + a[r][7]);
      u.z = sg0 * (a[r][5] - a[r][7]);  u.w = -sg0 * (a[r][4] - a[r][6]);
      *ph_out(p, 0, im, slot[r]) = q;
      *ph_out(p, 1, im, slot[r]) = u;
    }
}

// ------------------------------------------------------------------------------------
// SHARP_ALM2MAP_DERIV1: {d_theta T, d_phi T / sin theta} from one spin-0 a_lm column, as the spin-1 synthesis with
// E = -sqrt(l(l+1)) a, B = 0 (cp = c, cm = -c; legendre_core.cuh, d1_accum / d1_combine).  Same structure as
// synth2_kernel with a 32-byte tile row and half the accumulate FMAs.
// ------------------------------------------------------------------------------------
struct __align__(16) TileD1 { double A, C, cr, ci; };

__global__ void __launch_bounds__(256) prep_d1_kernel(KParams p) {
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int l0 = max(m, 1);
  const int j = blockIdx.x * blockDim.x + threadIdx.x, l = l0 + j;
  const int npad = l0 <= p.lmax ? (p.lmax - l0 + 1 + 7) & ~7 : 0;
  if (j >= npad) return;
  TileD1 e{0.0, 0.0, 0.0, 0.0};
  if (l <= p.lmax) {
    const double *a = p.alm0;
    const long long mvs = p.mvstart[im];
    const double nrm = (p.real_packed && m > 0) ? 0.70710678118654752440 : 1.0;
    const double4 c = reinterpret_cast<const double4 *>(p.coef + p.cofs[im])[l - l0];   // {A', C', g, 0}
    double ar, ai = 0.0;
    if (p.real_packed) {
      if (m == 0) ar = a[mvs + l];
      else { ar = a[mvs + 2 * (long long)l]; ai = a[mvs + 2 * (long long)l + 1]; }
    } else {
      ar = a[2 * (mvs + l)];
      if (m > 0) ai = a[2 * (mvs + l) + 1];
    }
    const double f = -sqrt((double)l * (double)(l + 1)) * c.z * nrm;
    e.A = c.x; e.C = c.y; e.cr = f * ar; e.ci = f * ai;
  }
  reinterpret_cast<TileD1 *>(p.trows)[p.tofs[im] + j] = e;
}

template <int MODE, int R>
__device__ __forceinline__ void synth_d1_group(const TileD1 *t, const double (&x)[R], double (&P)[R],
                                               double (&Pp)[R], double (&M)[R], double (&Mp)[R],
                                               double (&s)[R][8], int (&k)[R]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const double A = t[j].A, C = t[j].C, cr = t[j].cr, ci = t[j].ci;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (MODE >= 1) {
        const bool on = (MODE == 2 || k[r] == 0);
        d1_accum(j & 1, on ? P[r] : 0.0, on ? M[r] : 0.0, cr, ci, s[r]);
      }
      double up = fma(A, x[r], C), um = fma(A, x[r], -C);
      double np_ = fma(up, P[r], -Pp[r]), nm_ = fma(um, M[r], -Mp[r]);
      Pp[r] = P[r]; P[r] = np_; Mp[r] = M[r]; M[r] = nm_;
    }
  }
  if (MODE < 2) {
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (k[r] < 0 && (needs_rescale(P[r]) || needs_rescale(M[r]))) {
        P[r] *= SCALE_DOWN; Pp[r] *= SCALE_DOWN; M[r] *= SCALE_DOWN; Mp[r] *= SCALE_DOWN; ++k[r];
      }
  }
}

template <int R, int MINB>
__global__ void __launch_bounds__(32, MINB) synth_d1_kernel(KParams p) {
  __shared__ __align__(16) TileD1 tile[2][TL];
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int lane = threadIdx.x;
  const int chunk0 = p.slot_begin + blockIdx.x * (32 * R);
  const int l0 = max(m, 1);
  double x[R], P[R], Pp[R], M[R], Mp[R], s[R][8];
  int k[R], slot[R];
  bool any = false;
  const double K = p.Kstart[m];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    slot[r] = chunk0 + lane * R + r;
    bool valid = slot[r] < p.nslots && m <= p.mlim[min(slot[r], p.nslots - 1)] && l0 <= p.lmax;
#pragma unroll
    for (int q = 0; q < 8; ++q) s[r][q] = 0.0;
    P[r] = M[r] = Pp[r] = Mp[r] = 0.0; k[r] = 0; x[r] = 0.0;
    if (valid) {
      const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot[r]];
      RingTrig g{tg.x, tg.y, tg.z, tg.w};
      x[r] = g.cth;
      start_spin_s(m, 1, K, g, P[r], M[r], k[r]);
      any = true;
    }
  }
  if (__any_sync(FULL, any)) {
    const TileD1 *rows = reinterpret_cast<const TileD1 *>(p.trows) + p.tofs[im];
    auto issue_tile = [&](int b, int lt) {     // rows past this m's padded range are never used
      const char *src = reinterpret_cast<const char *>(rows + (lt - l0));
      char *dst = reinterpret_cast<char *>(tile[b]);
#pragma unroll
      for (int q = 0; q < (int)(TL * sizeof(TileD1)) / 512; ++q) cp_async16(dst + (q * 32 + lane) * 16, src + (q * 32 + lane) * 16);
      cp_async_commit();
    };
    issue_tile(0, l0);
    cp_async_wait_all();
    __syncwarp();
    int buf = 0;
    for (int lt = l0; lt <= p.lmax; lt += TL, buf ^= 1) {
      if (lt + TL <= p.lmax) issue_tile(buf ^ 1, lt + TL);
      const int ngroups = min(TL, p.lmax - lt + 8) / 8;
#pragma unroll 1
      for (int g = 0; g < ngroups; ++g) {
        bool all_on = true, none_on = true;
#pragma unroll
        for (int r = 0; r < R; ++r) { all_on &= (k[r] == 0); none_on &= (k[r] < 0); }
        if (__all_sync(FULL, all_on)) synth_d1_group<2, R>(tile[buf] + 8 * g, x, P, Pp, M, Mp, s, k);
        else if (__all_sync(FULL, none_on)) synth_d1_group<0, R>(tile[buf] + 8 * g, x, P, Pp, M, Mp, s, k);
        else synth_d1_group<1, R>(tile[buf] + 8 * g, x, P, Pp, M, Mp, s, k);
      }
      cp_async_wait_all();
      __syncwarp();
    }
  }
  const double sg0 = ((l0 + m) & 1) ? -0.5 : 0.5;
#pragma unroll
  for (int r = 0; r < R; ++r)
    if (slot[r] < p.nslots) {
      double q[4], u[4];
      d1_combine(s[r], sg0, q, u);
      *ph_out(p, 0, im, slot[r]) = make_double4(q[0], q[1], q[2], q[3]);
      *ph_out(p, 1, im, slot[r]) = make_double4(u[0], u[1], u[2], u[3]);
    }
}

// ------------------------------------------------------------------------------------
// Ring reduction for analysis.  Each lane holds 16 partial sums per group (the l of the group
// times the real outputs per l); a 5-stage butterfly reduce-scatter over the warp leaves one
// distinct total in every even lane: 16 double shuffles + 16 DADD per 16 outputs.
//
// The stages that split on a bit of the OUTPUT index (re/im; for spin 2 also S1/S2) need no
// per-lane register selection: the lanes with the corresponding lane bit set accumulate with
// their per-ring inputs permuted (re<->im swapped, P<->M roles swapped), so their register
// named "re" holds an imaginary part, etc., and every lane simply keeps the even-named and
// sends the odd-named register.  Only the stages that split on l need selects.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ double shfl_xor_d(double v, int mask) { return __shfl_xor_sync(FULL, v, mask); }


template <int H>
__device__ __forceinline__ void bfly_select(double *v, int lane, int bit) {
  const bool hi = lane & bit;
#pragma unroll
  for (int i = 0; i < H; ++i) {
    double send = hi ? v[i] : v[i + H], keep = hi ? v[i + H] : v[i];
    v[i] = keep + shfl_xor_d(send, bit);
  }
}
template <int H>
__device__ __forceinline__ void bfly_fixed(double *v, int bit) {
#pragma unroll
  for (int i = 0; i < H; ++i) v[i] = v[2 * i] + shfl_xor_d(v[2 * i + 1], bit);
}

// acc[4 j + 2 s + c], j = l (spin 0: row of two l) in group (4), s = S1/S2 (spin 0: T1/T2) as named (lane bit 3 swaps),
// c = re/im as named (lane bit 4 swaps).  Even lanes store l = 2 b2 + b1, s = b3, part = b4.
__device__ __forceinline__ int store_index_s2(int lane) {
  return 4 * (((lane >> 2) & 1) * 2 + ((lane >> 1) & 1)) + 2 * ((lane >> 3) & 1) + ((lane >> 4) & 1);
}
__device__ __forceinline__ void reduce_store_s2(double (&v)[16], double *dst, int lane) {
  bfly_fixed<8>(v, 16);          // v[2 j + s]
  bfly_fixed<4>(v, 8);           // v[j]
  bfly_select<2>(v, lane, 4);
  bfly_select<1>(v, lane, 2);
  v[0] += shfl_xor_d(v[0], 1);
  if (!(lane & 1)) dst[store_index_s2(lane)] = v[0];
}

// Software-pipelined form of the same butterfly for the steady phase.  In the step that runs
// the FMAs of group g, stage 1 is applied to g's sums as they complete, stage 2 to the state
// left by g-1, stage 3 to g-2, stage 4 to g-3 and stage 5 (+ the store) to g-4: five mutually
// independent shuffle rounds per step instead of one dependent chain of five, so no warp ever
// sits in a latency-only phase (with 2-3 resident warps per scheduler such phases line up and
// leave the FP64 pipe idle).  Same 15 live doubles as holding one extra group of sums.
struct ReducePipe { double v1[8], v2[4], v3[2], v4; };

// `sidx`: shared-memory byte address of this lane's slot in group 0 of the tile (16 doubles per group).  Both lanes of a
// pair hold the same total after stage 5 and store it to the same address: no divergence, no predicate.
template <bool SPIN2>
__device__ __forceinline__ void pipe_tail(const ReducePipe &in, ReducePipe &out, unsigned sidx, int gstore, bool store, int lane) {
  {  // stage 5 -> shared memory (group g-4)
    double v5 = in.v4 + shfl_xor_d(in.v4, 1);
    if (store) asm volatile("st.shared.f64 [%0], %1;" ::"r"(sidx + 128u * (unsigned)gstore), "d"(v5) : "memory");
  }
  {  // stage 4 (group g-3)
    const bool hi = lane & 2;
    double send = hi ? in.v3[0] : in.v3[1], keep = hi ? in.v3[1] : in.v3[0];
    out.v4 = keep + shfl_xor_d(send, 2);
  }
  {  // stage 3 (group g-2)
    const bool hi = lane & 4;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      double send = hi ? in.v2[i] : in.v2[i + 2], keep = hi ? in.v2[i + 2] : in.v2[i];
      out.v3[i] = keep + shfl_xor_d(send, 4);
    }
  }
  // stage 2 (group g-1)
  if (SPIN2) {
#pragma unroll
    for (int i = 0; i < 4; ++i) out.v2[i] = in.v1[2 * i] + shfl_xor_d(in.v1[2 * i + 1], 8);
  } else {
    const bool hi = lane & 8;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double send = hi ? in.v1[i] : in.v1[i + 4], keep = hi ? in.v1[i + 4] : in.v1[i];
      out.v2[i] = keep + shfl_xor_d(send, 8);
    }
  }
}

// ------------------------------------------------------------------------------------
// spin-0 analysis, two l per recurrence step (transpose of the synthesis above):
//   T1_j = sum_rings nu_j (qN + qS),  T2_j = sum_rings nu_j x (qN - qS)
//   a_{l_j} = u_j T1_j + v_{j-1} T1_{j-1},  a_{l_j+1} = h_j T2_j        (done in the per-tile flush)
// One group = 4 rows (8 l); acc[4 j + 2 s + c] = {T1.re, T1.im, T2.re, T2.im} (as named) of row j, i.e. the layout of
// the spin-2 kernel, whose reduction is reused: lanes with bit 3 set run with the T1 / T2 inputs swapped, lanes with
// bit 4 set with re / im swapped.  w[r] = {s.re, s.im, d.re, d.im} (before the per-lane permutation),
// s = qN + qS, d = x (qN - qS).
// ------------------------------------------------------------------------------------
template <int MODE, int R>
__device__ __forceinline__ void anal0_fma(const TileA0 *tA, const double (&x2)[R], double (&cur)[R],
                                          double (&prev)[R], const double (&w)[R][4], int (&k)[R],
                                          double (&acc)[16], unsigned ron = ~0u) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double A = tA[j].A, B = tA[j].B;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (MODE == 2 || (MODE == 1 && ((ron >> r) & 1))) {
        double v = (MODE == 2 || k[r] == 0) ? cur[r] : 0.0;
        s0 = fma(v, w[r][0], s0); s1 = fma(v, w[r][1], s1);
        s2 = fma(v, w[r][2], s2); s3 = fma(v, w[r][3], s3);
      }
      double nxt = step0x2(A, B, x2[r], cur[r], prev[r]);
      prev[r] = cur[r]; cur[r] = nxt;
    }
    if (MODE >= 1) { acc[4 * j] = s0; acc[4 * j + 1] = s1; acc[4 * j + 2] = s2; acc[4 * j + 3] = s3; }
  }
  if (MODE < 2) {
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (k[r] < 0 && needs_rescale(cur[r])) { cur[r] *= SCALE_DOWN; prev[r] *= SCALE_DOWN; ++k[r]; }
  }
}

// steady-phase step: FMAs of one group with stage 1 applied per row, stages 2-5 on the older groups
template <int R, bool FMA>
__device__ __forceinline__ void anal0_step(const TileA0 *tA, const double (&x2)[R], double (&cur)[R],
                                           double (&prev)[R], const double (&w)[R][4],
                                           const ReducePipe &in, ReducePipe &out, unsigned sidx, int gstore, bool store, int lane) {
  pipe_tail<true>(in, out, sidx, gstore, store, lane);
  if (FMA) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double A = tA[j].A, B = tA[j].B;
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        s0 = fma(cur[r], w[r][0], s0); s1 = fma(cur[r], w[r][1], s1);
        s2 = fma(cur[r], w[r][2], s2); s3 = fma(cur[r], w[r][3], s3);
        double nxt = step0x2(A, B, x2[r], cur[r], prev[r]);
        prev[r] = cur[r]; cur[r] = nxt;
      }
      out.v1[2 * j] = s0 + shfl_xor_d(s1, 16);
      out.v1[2 * j + 1] = s2 + shfl_xor_d(s3, 16);
    }
  }
}

// Analysis kernels, common structure: ONE WARP PER CTA, no block-level synchronisation at all.
// A thread owns R ADJACENT ring pairs, the warp 32 R adjacent ones (similar colatitude, so they
// cross the accumulation threshold at similar l, and whole warps fall beyond the m cut-off near
// the poles).  The warp stages its own coefficient tiles (TL rows, double buffered, cp.async
// straight from the table) and walks the groups of a tile in two phases: a transient one while
// some of its rings are still below the threshold (warp-uniform choice between "recurrence only"
// and "predicated", reduction done at once) and a steady one (all rings on -- they stay on) in
// which the butterfly of group g-1 sits in the same basic block as the FMAs of group g, so the
// shuffle latency hides behind FP64 work.  After each tile the reduced sums are read back row-major
// from shared memory and added to the a_lm with fully coalesced atomics (other warps hold the
// other rings of the same m).
// DET: the tile flush stores into the partials buffer (det.h) instead of adding to the a_lm; lane 0 records the first l
// the warp stores (DET_EMPTY until the warp knows it stores anything).
template <int R, int MINB, bool SEED = false, bool DET = false>
__global__ void __launch_bounds__(32, MINB) anal0_kernel(KParams p, DetArgs d) {
  __shared__ __align__(16) TileA0 tile[2][TL];
  __shared__ __align__(16) double red[(TL + 1) * 4];   // row 0: T1 of the last row of the previous tile
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int lane = threadIdx.x;
  const int chunk0 = p.slot_begin + blockIdx.x * (32 * R);
  [[maybe_unused]] const int blk = chunk0 / (32 * R);   // warp block of the whole geometry (DET launches start on a block boundary)
  if constexpr (DET) { if (lane == 0) d.drec[d.dl.rec_index(blk, im)] = DET_EMPTY; }
  const int J = p.lmax >= m ? (p.lmax - m) / 2 + 1 : 0;   // rows (steps of two l) of this m
  double x2[R], cur[R], prev[R], w[R][4];
  int k[R];
  bool any = false;
  const double K = p.Kstart[m];
  const bool swapRI = lane & 16, swapT = lane & 8;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    int slot = chunk0 + lane * R + r;
    bool valid = slot < p.nslots && m <= p.mlim[min(slot, p.nslots - 1)];
    prev[r] = cur[r] = x2[r] = 0.0; k[r] = 0;
    w[r][0] = w[r][1] = w[r][2] = w[r][3] = 0.0;
    if (valid) {
      const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot];
      RingTrig g{tg.x, tg.y, tg.z, tg.w};
      x2[r] = g.cth * g.cth;
      if constexpr (SEED) {
        const size_t s = (size_t)im * p.nslots + slot;
        const double2 st = reinterpret_cast<const double2 *>(p.ss)[s];
        cur[r] = st.x; prev[r] = st.y; k[r] = p.sk[s];
      } else {
        start_spin0(m, K, g, cur[r], k[r]);
      }
      double4 q = *ph_in(p, 0, im, slot);
      if (p.s2s_npolar >= 0) {   // spin 2 as scalar sums: phases / sin^2; the polar rings are anal2_kernel's
        const double f = slot < p.s2s_npolar ? 0.0 : 1.0 / (g.sth * g.sth);
        q.x *= f; q.y *= f; q.z *= f; q.w *= f;
      }
      double z[4] = {q.x + q.z, q.y + q.w, g.cth * (q.x - q.z), g.cth * (q.y - q.w)};
      // w[i] = z[i ^ (swapT ? 2 : 0) ^ (swapRI ? 1 : 0)]
#pragma unroll
      for (int i = 0; i < 4; i += 2) {
        double a0 = swapT ? z[i ^ 2] : z[i], a1 = swapT ? z[(i ^ 2) + 1] : z[i + 1];
        w[r][i] = swapRI ? a1 : a0; w[r][i + 1] = swapRI ? a0 : a1;
      }
      any = true;
    }
  }
  if (!__any_sync(FULL, any)) return;
  // first row of the warp's tile loop: the rows before the seeded one add exact zeros (the T1 of row j0 - 1 that the
  // first flush reads from red[0..3] is zero too)
  const int j0 = SEED ? p.sl[(size_t)im * gridDim.x + blockIdx.x] : 0;
  if (SEED && j0 >= J) return;
  if constexpr (DET) { if (lane == 0) d.drec[d.dl.rec_index(blk, im)] = m + 2 * j0; }
  const double *coef = p.coef + p.cofs[im];
  const double4 *mix = reinterpret_cast<const double4 *>(p.coef2 + 2 * p.cofs[im]);   // {u_j, v_j, h_j, v_{j-1}}
  const long long mvs = p.mvstart[im];
  // real-packed: orthonormal real basis (sqrt2 both ways).  complex a_lm: the phases carry the
  // factor 2 of the m>0 terms, so the adjoint needs 1/2 to return sum conj(Y) x as libsharp2 does
  const double nrm = p.s2s_npolar >= 0 ? 1.0 : (m > 0 ? (p.real_packed ? 0.70710678118654752440 : 0.5) : 1.0);
  const long long xofs = 2 * (p.cofs[im] - m);   // s2s scratch: {re, im} of l at 2 (cofs + l - m)
  // rows past the last one belong to the next m (or the table's zero padding): finite, never used
  auto issue_tile = [&](int b, int jt) {
    const char *src = reinterpret_cast<const char *>(coef + 2 * (size_t)jt);
    char *dst = reinterpret_cast<char *>(tile[b]);
#pragma unroll
    for (int q = 0; q < (int)(TL * sizeof(TileA0)) / 512; ++q) cp_async16(dst + (q * 32 + lane) * 16, src + (q * 32 + lane) * 16);
    cp_async_commit();
  };
  issue_tile(0, j0);
  if (lane < 4) red[lane] = 0.0;
  cp_async_wait_all();
  __syncwarp();
  int buf = 0;
  bool steady = false;
  unsigned sidx = (unsigned)__cvta_generic_to_shared(red + 4 + store_index_s2(lane));
  asm volatile("mov.u32 %0, %0;" : "+r"(sidx));   // opaque: kept in a register instead of being recomputed per group
  for (int jt = j0; jt < J; jt += TL, buf ^= 1) {
    if (jt + TL < J) issue_tile(buf ^ 1, jt + TL);
    const int ngroups = min(TL, J - jt + 3) / 4;
    const TileA0 *T = tile[buf];
    double *dst = red + 4;
    int g = 0;
    if (!steady) {
#pragma unroll 1
      for (; g < ngroups; ++g) {
        bool all_on = true, none_on = true;
#pragma unroll
        for (int r = 0; r < R; ++r) { all_on &= (k[r] == 0); none_on &= (k[r] < 0); }
        if (__all_sync(FULL, all_on)) { steady = true; break; }
        double acc[16];
        if (__all_sync(FULL, none_on)) {
          anal0_fma<0, R>(T + 4 * g, x2, cur, prev, w, k, acc);
          if (!(lane & 1)) dst[16 * g + (lane >> 1)] = 0.0;
        } else {
          anal0_fma<1, R>(T + 4 * g, x2, cur, prev, w, k, acc);
          reduce_store_s2(acc, dst + 16 * g, lane);
        }
      }
    }
    if (g < ngroups) {
      const int gs = g;
      ReducePipe st;
#pragma unroll
      for (int i = 0; i < 8; ++i) st.v1[i] = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i) st.v2[i] = 0.0;
      st.v3[0] = st.v3[1] = st.v4 = 0.0;
#pragma unroll 2
      for (; g < ngroups; ++g) {
        ReducePipe nx;
        anal0_step<R, true>(T + 4 * g, x2, cur, prev, w, st, nx, sidx, g - 4, g - 4 >= gs, lane);
        st = nx;
      }
#pragma unroll
      for (int d = 0; d < 4; ++d, ++g) {   // drain
        ReducePipe nx;
        anal0_step<R, false>(T, x2, cur, prev, w, st, nx, sidx, g - 4, g - 4 >= gs, lane);
        st = nx;
      }
    }
    cp_async_wait_all();
    __syncwarp();
    // flush the tile: four consecutive lanes = (re, im) of l_j and of l_j + 1 -> contiguous atomics
    double *a = p.alm0;
#pragma unroll 4
    for (int e = lane; e < 4 * TL; e += 32) {
      const int li = e >> 2, odd = (e >> 1) & 1, part = e & 1, j = jt + li, l = m + 2 * j + odd;
      if (l <= p.lmax && (m > 0 || part == 0)) {
        const double4 mx = mix[j];
        double val = odd ? mx.z * red[4 * (li + 1) + 2 + part]
                         : fma(mx.x, red[4 * (li + 1) + part], mx.w * red[4 * li + part]);
        val *= nrm;
        if (p.lscale0) val *= p.lscale0[l];
        const long long idx = p.s2s_npolar >= 0 ? xofs + 2 * (long long)l + part
                            : p.real_packed ? (m == 0 ? mvs + l : mvs + 2 * (long long)l + part) : 2 * (mvs + l) + part;
        if constexpr (DET) d.det[d.dl.index(0, blk, im, l, part)] = val;
        else atomicAdd(&a[idx], val);
      }
    }
    __syncwarp();
    if (lane < 2) red[lane] = red[4 * TL + lane];   // T1 of the tile's last row, for the first row of the next tile
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------
// spin-2 analysis.  zp = qQ + i qU, zm = qQ - i qU per ring (north, south*sg0);
//   S1_l = sum P zpN + sg M zpS ; S2_l = sum M zmN + sg P zmS
//   E_l = -(S1+S2)/2 ; B_l = (i/2)(S1-S2)
// One group = 4 l; acc[4 j + 2 s + c] = {S1.re, S1.im, S2.re, S2.im} (as named) of l = start + j.
// Pa / Pb are the recurrences in the "P role" (u = A x + Cs) and "M role" (u = A x - Cs); lanes
// with bit 3 set run them swapped (Cs = -C', Pa = M, Pb = P, w permuted) so that their registers
// named S1 hold S2 and vice versa (see the reduction above).
// ------------------------------------------------------------------------------------
__device__ __forceinline__ double flip_sign(double v, int mask) {
  return __hiloint2double(__double2hiint(v) ^ mask, __double2loint(v));
}

template <int MODE, int R>
__device__ __forceinline__ void anal2_fma(const TileA2 *t, const int csign, const double (&x)[R], double (&Pa)[R],
                                          double (&Pap)[R], double (&Pb)[R], double (&Pbp)[R],
                                          const double (&w)[R][8], int (&k)[R], double (&acc)[16], unsigned ron = ~0u) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double A = t[j].A, C = flip_sign(t[j].C, csign);
    double s1r = 0.0, s1i = 0.0, s2r = 0.0, s2i = 0.0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (MODE == 2 || (MODE == 1 && ((ron >> r) & 1))) {
        bool on = (MODE == 2 || k[r] == 0);
        double va = on ? Pa[r] : 0.0, vb = on ? Pb[r] : 0.0;
        // w: 0,1 zpN ; 2,3 zmN ; 4,5 zpS ; 6,7 zmS  (before the per-lane permutation)
        s1r = fma(va, w[r][0], s1r); s1i = fma(va, w[r][1], s1i);
        s2r = fma(vb, w[r][2], s2r); s2i = fma(vb, w[r][3], s2i);
        if (j & 1) {
          s1r = fma(-vb, w[r][4], s1r); s1i = fma(-vb, w[r][5], s1i);
          s2r = fma(-va, w[r][6], s2r); s2i = fma(-va, w[r][7], s2i);
        } else {
          s1r = fma(vb, w[r][4], s1r); s1i = fma(vb, w[r][5], s1i);
          s2r = fma(va, w[r][6], s2r); s2i = fma(va, w[r][7], s2i);
        }
      }
      double ua = fma(A, x[r], C), ub = fma(A, x[r], -C);
      double na = fma(ua, Pa[r], -Pap[r]), nb = fma(ub, Pb[r], -Pbp[r]);
      Pap[r] = Pa[r]; Pa[r] = na; Pbp[r] = Pb[r]; Pb[r] = nb;
    }
    if (MODE >= 1) { acc[4 * j] = s1r; acc[4 * j + 1] = s1i; acc[4 * j + 2] = s2r; acc[4 * j + 3] = s2i; }
  }
  if (MODE < 2) {
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (k[r] < 0 && (needs_rescale(Pa[r]) || needs_rescale(Pb[r]))) {
        Pa[r] *= SCALE_DOWN; Pap[r] *= SCALE_DOWN; Pb[r] *= SCALE_DOWN; Pbp[r] *= SCALE_DOWN; ++k[r];
      }
  }
}

// Loop order: ring outer, l inner.  For a fixed ring the recurrence is a dependent chain over l,
// so the scheduler issues [next value, 4 accumulates] of one lambda back to back -- five DFMAs with
// the same first operand, which then comes from the operand-reuse cache (a DFMA costs
// max(2, #vector operands fetched from the register file) cycles on B200).
template <int R, bool FMA>
__device__ __forceinline__ void anal2_step(const TileA2 *t, const int csign, const double (&x)[R], double (&Pa)[R],
                                           double (&Pap)[R], double (&Pb)[R], double (&Pbp)[R],
                                           const double (&w)[R][8], const ReducePipe &in, ReducePipe &out,
                                           unsigned sidx, int gstore, bool store, int lane) {
  pipe_tail<true>(in, out, sidx, gstore, store, lane);
  if (FMA) {
    double s[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      double ua[4], ub[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double A = t[j].A, C = flip_sign(t[j].C, csign);
        ua[j] = fma(x[r], A, C); ub[j] = fma(x[r], A, -C);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const double va = Pa[r], vb = Pb[r];
        const double na = fma(va, ua[j], -Pap[r]);
        s[j][0] = fma(va, w[r][0], s[j][0]); s[j][1] = fma(va, w[r][1], s[j][1]);
        if (j & 1) { s[j][2] = fma(-va, w[r][6], s[j][2]); s[j][3] = fma(-va, w[r][7], s[j][3]); }
        else       { s[j][2] = fma(va, w[r][6], s[j][2]);  s[j][3] = fma(va, w[r][7], s[j][3]); }
        const double nb = fma(vb, ub[j], -Pbp[r]);
        s[j][2] = fma(vb, w[r][2], s[j][2]); s[j][3] = fma(vb, w[r][3], s[j][3]);
        if (j & 1) { s[j][0] = fma(-vb, w[r][4], s[j][0]); s[j][1] = fma(-vb, w[r][5], s[j][1]); }
        else       { s[j][0] = fma(vb, w[r][4], s[j][0]);  s[j][1] = fma(vb, w[r][5], s[j][1]); }
        Pap[r] = va; Pa[r] = na; Pbp[r] = vb; Pb[r] = nb;
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      out.v1[2 * j] = s[j][0] + shfl_xor_d(s[j][1], 16);
      out.v1[2 * j + 1] = s[j][2] + shfl_xor_d(s[j][3], 16);
    }
  }
}

// DET: as in anal0_kernel, E into component 0 and B into component 1 of the partials buffer
template <int R, int MINB, bool SEED = false, bool DET = false>
__global__ void __launch_bounds__(32, MINB) anal2_kernel(KParams p, DetArgs d) {
  __shared__ __align__(16) TileA2 tile[2][TL];
  __shared__ __align__(16) double red[TL * 4];
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int lane = threadIdx.x;
  const int chunk0 = p.slot_begin + blockIdx.x * (32 * R);
  [[maybe_unused]] const int blk = chunk0 / (32 * R);
  if constexpr (DET) { if (lane == 0) d.drec[d.dl.rec_index(blk, im)] = DET_EMPTY; }
  const int l0 = max(m, p.spin);
  if (l0 > p.lmax) return;
  double x[R], Pa[R], Pap[R], Pb[R], Pbp[R], w[R][8];
  int k[R];
  bool any = false;
  const double K = p.Kstart[m];
  const double sg0 = ((l0 + m) & 1) ? -1.0 : 1.0;
  const bool swapRI = lane & 16, swapPM = lane & 8;
  const int csign = swapPM ? 0x80000000 : 0;   // sign-bit mask applied to C' (an integer op, not a DMUL)
  // scalar front phase (see synth2_kernel): Pa / Pap hold the scalar state until the conversion
  unsigned vmask = 0;
  int mg[R];
  bool front = !SEED && p.fcoef != nullptr && m >= 4, fok = true;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    int slot = chunk0 + r * 32 + lane;
    bool valid = slot < p.nslots && m <= p.mlim[min(slot, p.nslots - 1)];
    Pa[r] = Pb[r] = Pap[r] = Pbp[r] = x[r] = 0.0; k[r] = 0; mg[r] = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) w[r][q] = 0.0;
    if (valid) {
      const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot];
      RingTrig g{tg.x, tg.y, tg.z, tg.w};
      x[r] = g.cth;
      vmask |= 1u << r;
      if constexpr (SEED) {   // the table holds P / M roles (seed2_kernel)
        const size_t s = (size_t)im * p.nslots + slot;
        const double4 st = reinterpret_cast<const double4 *>(p.ss)[s];
        Pa[r] = swapPM ? st.z : st.x; Pb[r] = swapPM ? st.x : st.z;
        Pap[r] = swapPM ? st.w : st.y; Pbp[r] = swapPM ? st.y : st.w;
        k[r] = p.sk[s];
      } else {
        mg[r] = front_margin_bits(g.sth);
        if (front) { start_spin0(m, p.fK0[m], g, Pa[r], k[r]); fok &= k[r] < 0 && g.sth >= FRONT_MIN_STH; }
      }
      any = true;
    }
  }
  if (!__any_sync(FULL, any)) return;
  front = front && __all_sync(FULL, fok);
  // l (counted from l0) the front phase has covered (whole tiles, which contribute nothing to the a_lm), or where the
  // seed table starts the warp
  int lskip = SEED ? p.sl[(size_t)im * gridDim.x + blockIdx.x] : 0;
  if (SEED && l0 + lskip > p.lmax) return;
  if (front) {
    const int jb = spin2_front_phase<R, 2, FRONT_TR>(p, im, m, vmask, x, mg, Pa, Pap, k);
    lskip = 2 * jb;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const double nu = Pa[r], nup = Pap[r];
      Pa[r] = Pap[r] = 0.0;
      if ((vmask >> r) & 1) {
        const double sth = reinterpret_cast<const double4 *>(p.trig)[chunk0 + r * 32 + lane].y;
        double P0, Pp0, M0, Mp0;
        spin2_front_finish(p, im, m, jb, x[r], sth, nu, nup, P0, Pp0, M0, Mp0);
        Pa[r] = swapPM ? M0 : P0; Pb[r] = swapPM ? P0 : M0;
        Pap[r] = swapPM ? Mp0 : Pp0; Pbp[r] = swapPM ? Pp0 : Mp0;
      } else k[r] = 0;
    }
  } else if (!SEED) {
#pragma unroll
    for (int r = 0; r < R; ++r)
      if ((vmask >> r) & 1) {
        const double4 tg = reinterpret_cast<const double4 *>(p.trig)[chunk0 + r * 32 + lane];
        RingTrig g{tg.x, tg.y, tg.z, tg.w};
        double P0, M0;
        if (p.spin == 2) start_spin2(m, K, g, P0, M0, k[r]); else start_spin_s(m, p.spin, K, g, P0, M0, k[r]);
        Pa[r] = swapPM ? M0 : P0; Pb[r] = swapPM ? P0 : M0;
      }
  }
  // ring data (loaded after the front phase, which needs the registers)
#pragma unroll
  for (int r = 0; r < R; ++r)
    if ((vmask >> r) & 1) {
      const int slot = chunk0 + r * 32 + lane;
      double4 q = *ph_in(p, 0, im, slot), u = *ph_in(p, 1, im, slot);
      double z[8];
      z[0] = q.x - u.y; z[1] = q.y + u.x;            // zpN = qQ + i qU
      z[2] = q.x + u.y; z[3] = q.y - u.x;            // zmN = qQ - i qU
      z[4] = sg0 * (q.z - u.w); z[5] = sg0 * (q.w + u.z);
      z[6] = sg0 * (q.z + u.w); z[7] = sg0 * (q.w - u.z);
      // w[i] = z[i ^ (swapPM ? 2 : 0) ^ (swapRI ? 1 : 0)]
#pragma unroll
      for (int i = 0; i < 8; i += 2) {
        double a0 = swapPM ? z[i ^ 2] : z[i], a1 = swapPM ? z[(i ^ 2) + 1] : z[i + 1];
        w[r][i] = swapRI ? a1 : a0; w[r][i + 1] = swapRI ? a0 : a1;
      }
    }
  const double *coef = p.coef + p.cofs[im];
  const long long mvs = p.mvstart[im];
  // real-packed: orthonormal real basis (sqrt2 both ways).  complex a_lm: the phases carry the
  // factor 2 of the m>0 terms, so the adjoint needs 1/2 to return sum conj(Y) x as libsharp2 does
  const double nrm = m > 0 ? (p.real_packed ? 0.70710678118654752440 : 0.5) : 1.0;
  // rows past lmax belong to the next m (or the table's zero padding): finite, never used
  auto issue_tile = [&](int b, int lt) {
    const char *src = reinterpret_cast<const char *>(coef + 4 * (size_t)(lt - l0));
    char *dst = reinterpret_cast<char *>(tile[b]);
#pragma unroll
    for (int q = 0; q < (int)(TL * sizeof(TileA2)) / 512; ++q) cp_async16(dst + (q * 32 + lane) * 16, src + (q * 32 + lane) * 16);
    cp_async_commit();
  };
  if constexpr (DET) { if (lane == 0) d.drec[d.dl.rec_index(blk, im)] = l0 + lskip; }
  issue_tile(0, l0 + lskip);
  cp_async_wait_all();
  __syncwarp();
  int buf = 0;
  bool steady = false;
  unsigned sidx = (unsigned)__cvta_generic_to_shared(red + store_index_s2(lane));
  asm volatile("mov.u32 %0, %0;" : "+r"(sidx));   // opaque: kept in a register instead of being recomputed per group
  for (int lt = l0 + lskip; lt <= p.lmax; lt += TL, buf ^= 1) {
    if (lt + TL <= p.lmax) issue_tile(buf ^ 1, lt + TL);
    const int ngroups = min(TL, p.lmax - lt + 4) / 4;
    const TileA2 *T = tile[buf];
    double *dst = red;
    int g = 0;
    if (!steady) {
#pragma unroll 1
      for (; g < ngroups; ++g) {
        bool all_on = true, none_on = true;
#pragma unroll
        for (int r = 0; r < R; ++r) { all_on &= (k[r] == 0); none_on &= (k[r] < 0); }
        if (__all_sync(FULL, all_on)) { steady = true; break; }
        double acc[16];
        if (__all_sync(FULL, none_on)) {
          anal2_fma<0, R>(T + 4 * g, csign, x, Pa, Pap, Pb, Pbp, w, k, acc);
          if (!(lane & 1)) dst[16 * g + (lane >> 1)] = 0.0;
        } else {
          anal2_fma<1, R>(T + 4 * g, csign, x, Pa, Pap, Pb, Pbp, w, k, acc, slices_on(k));
          reduce_store_s2(acc, dst + 16 * g, lane);
        }
      }
    }
    if (g < ngroups) {
      const int gs = g;
      ReducePipe st;
#pragma unroll
      for (int i = 0; i < 8; ++i) st.v1[i] = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i) st.v2[i] = 0.0;
      st.v3[0] = st.v3[1] = st.v4 = 0.0;
#pragma unroll 2
      for (; g < ngroups; ++g) {
        ReducePipe nx;
        anal2_step<R, true>(T + 4 * g, csign, x, Pa, Pap, Pb, Pbp, w, st, nx, sidx, g - 4, g - 4 >= gs, lane);
        st = nx;
      }
#pragma unroll
      for (int d = 0; d < 4; ++d, ++g) {   // drain
        ReducePipe nx;
        anal2_step<R, false>(T, csign, x, Pa, Pap, Pb, Pbp, w, st, nx, sidx, g - 4, g - 4 >= gs, lane);
        st = nx;
      }
    }
    cp_async_wait_all();
    __syncwarp();
    // flush the tile: lane pair (2i, 2i+1) = (re, im) of one l -> contiguous atomics
    double *aE = p.alm0, *aB = p.alm1;
#pragma unroll 4
    for (int e = lane; e < 2 * TL; e += 32) {
      const int li = e >> 1, part = e & 1, l = lt + li;
      if (l <= p.lmax && (m > 0 || part == 0)) {
        const double4 v = reinterpret_cast<const double4 *>(red)[li];   // S1.re, S1.im, S2.re, S2.im
        // adjoint of the synthesis combination: E = (sp S1 - S2)/2, B = -(i/2)(sp S1 + S2), sp = spinsign
        const double gs = 0.5 * T[li].g * nrm, sp = p.spinsign;
        double E = part ? gs * (sp * v.y - v.w) : gs * (sp * v.x - v.z);
        double B = part ? -gs * (sp * v.x + v.z) : gs * (sp * v.y + v.w);
        if (p.lscale0) E *= p.lscale0[l];
        if (p.lscale1) B *= p.lscale1[l];
        const long long idx = p.real_packed ? (m == 0 ? mvs + l : mvs + 2 * (long long)l + part) : 2 * (mvs + l) + part;
        if constexpr (DET) {
          d.det[d.dl.index(0, blk, im, l, part)] = E;
          d.det[d.dl.index(1, blk, im, l, part)] = B;
        } else {
          atomicAdd(&aE[idx], E);
          atomicAdd(&aB[idx], B);
        }
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------
// Seed tables.  Before the first ring of a warp reaches the accumulation threshold, a Legendre kernel only advances the
// recurrence (and, for spin 2, the scalar front phase); nothing it adds to the phases or the a_lm there is non-zero.
// That part depends on the geometry, lmax, the m set, the spin and the kernel's slot-to-warp mapping only, so it is run
// once per plan by the seed kernels below and the Legendre kernels start from where it ends.  A seed kernel repeats
// its Legendre kernel's prologue and its group loop without the accumulation, on the same slots per lane, with the same
// start values, steps, rescaling points and front-phase hand-over, and stops at the first group at which a valid ring
// of the warp is on (k == 0).  It records that group's first row (spin 0) or l - l0 (spin 2) per (m, warp) and the
// state of every ring there, per (m, slot).  The groups it skips add exact zeros in the Legendre kernel (nothing while
// no ring is on; products with 0.0 when only invalid slots of the warp are "on"), so a seeded synthesis is bit-for-bit
// the unseeded one and a seeded analysis only loses atomic additions of zeros.
// ------------------------------------------------------------------------------------
// spin 0: synth0 (R = 4) and anal0 (R = 8), ring pair r of lane `lane` = slot chunk0 + lane R + r, groups of 4 rows
template <int R>
__global__ void __launch_bounds__(32) seed0_kernel(KParams p) {
  const int im = blockIdx.y, m = p.mval[im];
  const int lane = threadIdx.x;
  const int chunk0 = blockIdx.x * (32 * R);
  const int J = p.lmax >= m ? (p.lmax - m) / 2 + 1 : 0;
  double x2[R], cur[R], prev[R];
  int k[R];
  unsigned vmask = 0;
  const double K = p.Kstart[m];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int slot = chunk0 + lane * R + r;
    const bool valid = slot < p.nslots && m <= p.mlim[min(slot, p.nslots - 1)];
    prev[r] = cur[r] = x2[r] = 0.0; k[r] = 0;
    if (valid) {
      const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot];
      RingTrig g{tg.x, tg.y, tg.z, tg.w};
      x2[r] = g.cth * g.cth;
      start_spin0(m, K, g, cur[r], k[r]);
      vmask |= 1u << r;
    }
  }
  const double2 *rec = reinterpret_cast<const double2 *>(p.coef + p.cofs[im]);   // {A_j, B_j}, the tiles' rows
  int j = 0;
  if (__any_sync(FULL, vmask != 0)) {
#pragma unroll 1
    for (; j < J; j += 4) {
      bool on = false;
#pragma unroll
      for (int r = 0; r < R; ++r) on |= ((vmask >> r) & 1) && k[r] == 0;
      if (__any_sync(FULL, on)) break;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const double2 ab = rec[j + q];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const double nxt = step0x2(ab.x, ab.y, x2[r], cur[r], prev[r]);
          prev[r] = cur[r]; cur[r] = nxt;
        }
      }
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (k[r] < 0 && needs_rescale(cur[r])) { cur[r] *= SCALE_DOWN; prev[r] *= SCALE_DOWN; ++k[r]; }
    }
  }
  if (lane == 0) const_cast<int *>(p.sl)[(size_t)im * gridDim.x + blockIdx.x] = j;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int slot = chunk0 + lane * R + r;
    if (slot < p.nslots) {
      const size_t s = (size_t)im * p.nslots + slot;
      reinterpret_cast<double2 *>(const_cast<double *>(p.ss))[s] = make_double2(cur[r], prev[r]);
      const_cast<int *>(p.sk)[s] = k[r];
    }
  }
}

// spin 2: synth2 (lane-major slots, front phase rows GR = 4 at a time, groups of GL = 8 l) and anal2 (slots 32 apart,
// GR = 2, GL = 4).  The state is stored in the P / M roles {P, P_prev, M, M_prev}.
template <int R, int GR, int GL, bool STRIDED>
__global__ void __launch_bounds__(32) seed2_kernel(KParams p) {
  const int im = blockIdx.y, m = p.mval[im];
  const int lane = threadIdx.x;
  const int chunk0 = blockIdx.x * (32 * R);
  const int l0 = max(m, p.spin);
  auto slot_of = [&](int r) { return STRIDED ? chunk0 + r * 32 + lane : chunk0 + lane * R + r; };
  double x[R], P[R], Pp[R], M[R], Mp[R];
  int k[R], mg[R];
  unsigned vmask = 0;
  bool front = p.fcoef != nullptr && m >= 4 && l0 <= p.lmax, fok = true;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int slot = slot_of(r);
    const bool valid = slot < p.nslots && m <= p.mlim[min(slot, p.nslots - 1)] && l0 <= p.lmax;
    P[r] = M[r] = Pp[r] = Mp[r] = 0.0; k[r] = 0; x[r] = 0.0; mg[r] = 0;
    if (valid) {
      const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot];
      RingTrig g{tg.x, tg.y, tg.z, tg.w};
      x[r] = g.cth;
      vmask |= 1u << r;
      mg[r] = front_margin_bits(g.sth);
      if (front) { start_spin0(m, p.fK0[m], g, P[r], k[r]); fok &= k[r] < 0 && g.sth >= FRONT_MIN_STH; }
    }
  }
  int lt = 0;   // l - l0
  if (__any_sync(FULL, vmask != 0)) {
    if (__all_sync(FULL, fok) && front) {
      const int jb = spin2_front_phase<R, GR, FRONT_TR>(p, im, m, vmask, x, mg, P, Pp, k);
      lt = 2 * jb;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const double nu = P[r], nup = Pp[r];
        P[r] = Pp[r] = 0.0;
        if ((vmask >> r) & 1) {
          const double sth = reinterpret_cast<const double4 *>(p.trig)[slot_of(r)].y;
          spin2_front_finish(p, im, m, jb, x[r], sth, nu, nup, P[r], Pp[r], M[r], Mp[r]);
        } else k[r] = 0;
      }
    } else {
#pragma unroll
      for (int r = 0; r < R; ++r)
        if ((vmask >> r) & 1) {
          const double4 tg = reinterpret_cast<const double4 *>(p.trig)[slot_of(r)];
          RingTrig g{tg.x, tg.y, tg.z, tg.w};
          start_spin2(m, p.Kstart[m], g, P[r], M[r], k[r]);
        }
    }
    const double4 *coef = reinterpret_cast<const double4 *>(p.coef + p.cofs[im]);   // {A', C', g, 0} from l0
#pragma unroll 1
    for (; l0 + lt <= p.lmax; lt += GL) {
      bool on = false;
#pragma unroll
      for (int r = 0; r < R; ++r) on |= ((vmask >> r) & 1) && k[r] == 0;
      if (__any_sync(FULL, on)) break;
#pragma unroll
      for (int j = 0; j < GL; ++j) {
        const double4 c = coef[lt + j];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const double up = fma(c.x, x[r], c.y), um = fma(c.x, x[r], -c.y);
          const double np_ = fma(up, P[r], -Pp[r]), nm_ = fma(um, M[r], -Mp[r]);
          Pp[r] = P[r]; P[r] = np_; Mp[r] = M[r]; M[r] = nm_;
        }
      }
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (k[r] < 0 && (needs_rescale(P[r]) || needs_rescale(M[r]))) {
          P[r] *= SCALE_DOWN; Pp[r] *= SCALE_DOWN; M[r] *= SCALE_DOWN; Mp[r] *= SCALE_DOWN; ++k[r];
        }
    }
  }
  if (lane == 0) const_cast<int *>(p.sl)[(size_t)im * gridDim.x + blockIdx.x] = lt;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int slot = slot_of(r);
    if (slot < p.nslots) {
      const size_t s = (size_t)im * p.nslots + slot;
      reinterpret_cast<double4 *>(const_cast<double *>(p.ss))[s] = make_double4(P[r], Pp[r], M[r], Mp[r]);
      const_cast<int *>(p.sk)[s] = k[r];
    }
  }
}

// ------------------------------------------------------------------------------------
// Spin 2 as scalar sums (legendre_core.cuh, s2s_coefs): sum_l c_l (+-2)lam_l = (1 / sin^2) sum_{l'} d_l' lam_l' with d a
// banded map of the a_lm up to l' = lmax + 2, so a spin-2 synthesis is a prep kernel that forms the scalar sequences of
// the two map components plus two spin-0 syntheses (phases scaled by 1 / sin^2 on store), and an analysis is two spin-0
// analyses (phases scaled on load) into a scratch buffer plus the transposed map.  1 + 2 FP64 ops per (l, ring pair)
// and component instead of 4 + 8 for both; the synthesis runs the recurrence once for both components (synth0_kernel<2>),
// so 1 + 4 for Q and U together.  `p` is the spin-0 view (lmax + 2 and the two-l-per-step tables of that range).
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) prep_s2s_kernel(KParams p) {
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int lmax = p.lmax - 2, l0 = max(m, 2);
  const int j = blockIdx.x * blockDim.x + threadIdx.x, lj = m + 2 * j;
  const int J = (p.lmax - m) / 2 + 1;
  const int npad = (J + 7) & ~7;
  if (j >= npad) return;
  TileS0<2> e{0.0, 0.0, {{0.0, 0.0, 0.0, 0.0}, {0.0, 0.0, 0.0, 0.0}}};
  if (j < J) {
    const double *aE = p.alm0, *aB = p.alm1;
    const long long mvs = p.mvstart[im];
    const double nrm = (p.real_packed && m > 0) ? 0.70710678118654752440 : 1.0;
    double d[2][3][2] = {};   // [component][l_j + t][re, im]
#pragma unroll
    for (int dl = -2; dl <= 4; ++dl) {   // sources l_j - 2 .. l_j + 4 reach l_j .. l_j + 2
      const int l = lj + dl;
      if (l < l0 || l > lmax) continue;
      double er, ei = 0.0, br, bi = 0.0;
      if (p.real_packed) {
        if (m == 0) { er = aE[mvs + l]; br = aB[mvs + l]; }
        else {
          er = aE[mvs + 2 * (long long)l]; ei = aE[mvs + 2 * (long long)l + 1];
          br = aB[mvs + 2 * (long long)l]; bi = aB[mvs + 2 * (long long)l + 1];
        }
      } else {
        er = aE[2 * (mvs + l)]; br = aB[2 * (mvs + l)];
        if (m > 0) { ei = aE[2 * (mvs + l) + 1]; bi = aB[2 * (mvs + l) + 1]; }
      }
      const double fE = p.lscale0 ? nrm * p.lscale0[l] : nrm, fB = p.lscale1 ? nrm * p.lscale1[l] : nrm;
      double s[2][5][2] = {};
      s2s_scatter(l, m, fE * er, fE * ei, fB * br, fB * bi, s);
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        const int i = t - dl + 2;
#pragma unroll
        for (int c = 0; c < 2; ++c)
          if (i >= 0 && i < 5) { d[c][t][0] += s[c][i][0]; d[c][t][1] += s[c][i][1]; }
      }
    }
    const double2 rc = reinterpret_cast<const double2 *>(p.coef + p.cofs[im])[j];        // {A_j, B_j}
    const double4 mx = reinterpret_cast<const double4 *>(p.coef2 + 2 * p.cofs[im])[j];   // {u_j, v_j, h_j, v_{j-1}}
    e.A = rc.x; e.B = rc.y;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      e.c[c][0] = fma(mx.x, d[c][0][0], mx.y * d[c][2][0]); e.c[c][1] = fma(mx.x, d[c][0][1], mx.y * d[c][2][1]);
      e.c[c][2] = mx.z * d[c][1][0]; e.c[c][3] = mx.z * d[c][1][1];
    }
  }
  reinterpret_cast<TileS0<2> *>(p.trows)[p.tofs[im] + j] = e;
}

// E, B from the scalar sums T (component c at T + c * ctot, {re, im} of (m, l) at 2 (xcofs[im] + l - m)), added to the
// a_lm after the real-packed norm and the per-l factors of the spin-2 analysis kernel.  `p` is the spin-2 view.
__global__ void __launch_bounds__(256) post_s2s_kernel(KParams p, const double *T, const long long *xcofs, long long ctot) {
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < max(m, 2) || l > p.lmax) return;
  const double *tq = T + 2 * (xcofs[im] - m), *tu = tq + ctot;
  double q[5][2], u[5][2];
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const int t = l - 2 + i;
    const bool ok = t >= m;
    q[i][0] = ok ? tq[2 * t] : 0.0; q[i][1] = ok ? tq[2 * t + 1] : 0.0;
    u[i][0] = ok ? tu[2 * t] : 0.0; u[i][1] = ok ? tu[2 * t + 1] : 0.0;
  }
  double er, ei, br, bi;
  s2s_gather(l, m, q, u, er, ei, br, bi);
  // real-packed: orthonormal real basis (sqrt2 both ways); complex a_lm: 1/2 as in anal2_kernel
  const double nrm = m > 0 ? (p.real_packed ? 0.70710678118654752440 : 0.5) : 1.0;
  const double fE = p.lscale0 ? nrm * p.lscale0[l] : nrm, fB = p.lscale1 ? nrm * p.lscale1[l] : nrm;
  double *aE = p.alm0, *aB = p.alm1;
  const long long mvs = p.mvstart[im];
  const long long i0 = p.real_packed ? (m == 0 ? mvs + l : mvs + 2 * (long long)l) : 2 * (mvs + l);
  aE[i0] += fE * er; aB[i0] += fB * br;
  if (m > 0) { aE[i0 + 1] += fE * ei; aB[i0 + 1] += fB * bi; }
}

// Ordered reduce of a deterministic analysis (det.h): for each (l, part) of the local m's of `p`, a = a + (the sum of the
// partials of every warp block in ascending block order), component c of the partials into alm0 (c = 0) / alm1 (c = 1).
// The a_lm slots and the destination index are those of the kernels' tile flush.
__global__ void __launch_bounds__(256) det_reduce_kernel(KParams p, DetArgs d, int ncomp) {
  const int im = p.im0 + blockIdx.y, m = p.mval[im];
  const int e = blockIdx.x * blockDim.x + threadIdx.x, l = e >> 1, part = e & 1;
  if (l < max(m, p.spin) || l > p.lmax || (m == 0 && part)) return;
  const long long idx = det_dst_index(p.s2s_npolar >= 0, p.real_packed, m, p.mvstart[im], 2 * (p.cofs[im] - m), l, part);
  const int *rec = d.drec + d.dl.rec_index(0, im);
  const size_t bstride = (size_t)d.dl.nm * d.dl.row();
  for (int c = 0; c < ncomp; ++c) {
    const double *src = d.det + d.dl.index(c, 0, im, l, part);
    const double s = det_sum(rec, 1, d.dl.nb, l, [&](int b) { return src[(size_t)b * bstride]; });
    double *a = c ? p.alm1 : p.alm0;
    a[idx] = a[idx] + s;
  }
}

// ------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------
// Ring pairs per thread (register blocking).  Defaults were picked from the sweep recorded in
// profiles/; CMDR_SHT_R_S0 / _S2 / _D1 / _A0 / _A2 (with _MINB_) override them for tuning runs.
static int env_int(const char *name, int dflt) {
  const char *e = getenv(name);
  return (e && *e) ? atoi(e) : dflt;
}

static KParams make_params(const LegGeom &g, const LegAlm &a, double *alm0, double *alm1, double4 *ph) {
  KParams p;
  p.lmax = a.lmax; p.nm = a.nm; p.real_packed = a.real_packed;
  p.spin = a.spin; p.spinsign = (a.spin & 1) ? 1.0 : -1.0;
  p.slot_begin = g.slot_begin; p.nslots = g.slot_end >= 0 ? g.slot_end : g.nslots; p.NPL = g.NPL; p.NML = g.NML; p.ncomp_tot = g.ncomp_tot; p.comp0 = g.comp0;
  p.ring_major = phase_ring_major() ? 1 : 0;
  p.mval = a.mval; p.mvstart = a.mvstart; p.coef = a.coef; p.coef2 = a.coef2; p.cofs = a.cofs; p.Kstart = a.Kstart;
  p.fcoef = a.front_coef; p.fmix = a.front_mix; p.fcofs = a.front_cofs; p.fK0 = a.front_K0;
  p.tofs = nullptr; p.trows = nullptr;
  p.sl = nullptr; p.ss = nullptr; p.sk = nullptr;
  p.s2s_npolar = -1;
  p.im0 = a.im_begin;
  p.trig = g.trig; p.mlim = g.mlim; p.wslot = g.wslot;
  p.alm0 = alm0; p.alm1 = alm1; p.ph = ph;
  p.lscale0 = a.lscale[0]; p.lscale1 = a.lscale[1];
  p.src_rank = g.npeer ? g.src_rank : -1;
  for (int i = 0; i < CMDR_MAX_PEERS; ++i) p.peer[i] = g.npeer ? g.peer[i] : ph;
  return p;
}

template <int R, typename K, typename... A>
static void launch_w(K kernel, const KParams &p, int nm, cudaStream_t st, A... args) {   // one warp per CTA
  const int n = p.nslots - p.slot_begin;
  if (n <= 0) return;
  dim3 grid((n + 32 * R - 1) / (32 * R), nm);
  kernel<<<grid, 32, 0, st>>>(p, args...);
}

// ---- seed tables: one per (geometry handle, alm handle, kernel), built on first use ----
enum SeedKind { SEED_S0, SEED_A0, SEED_S2, SEED_A2, SEED_S0X, SEED_A0X };   // ..X: spin-0 kernels of the s2s route
struct SeedTab { int *sl = nullptr; double *ss = nullptr; int *sk = nullptr; size_t bytes = 0; };
static std::map<std::tuple<const void *, const void *, int>, SeedTab> g_seeds;
static bool g_seeds_on = true;
static size_t g_seed_bytes = 0;

static void seed_free(SeedTab &t) {
  cudaFree(t.sl); cudaFree(t.ss); cudaFree(t.sk);
  g_seed_bytes -= t.bytes;
}
void seed_forget(const void *h) {
  for (auto it = g_seeds.begin(); it != g_seeds.end();) {
    if (std::get<0>(it->first) == h || std::get<1>(it->first) == h) {
      CMDR_CUDA_CHECK(cudaDeviceSynchronize());   // queued kernels may still read the table
      seed_free(it->second);
      it = g_seeds.erase(it);
    } else {
      ++it;
    }
  }
}
void seed_release() {
  if (g_seeds.empty()) return;
  CMDR_CUDA_CHECK(cudaDeviceSynchronize());
  for (auto &kv : g_seeds) seed_free(kv.second);
  g_seeds.clear();
}

// The seed table of `kind` for a launch with parameters `p` (nullptr: start from the closed-form values).  Used when
// the launch covers every slot of a single-GPU geometry (the tables follow the warps of a launch from slot 0) and the
// table takes at most 1/32 of the device memory: at nside 2048 / lmax 4000, 20 B (spin 0) or 36 B (spin 2) per
// (m, ring pair) = 0.33 / 0.59 GB per kernel.
static const SeedTab *seed_table(const LegGeom &g, SeedKind kind, int R, const KParams &p, int nm, cudaStream_t st) {
  if (!g_seeds_on || !g.seed_geom || p.slot_begin != 0 || p.nslots != g.nslots || g.wslot) return nullptr;
  const auto key = std::make_tuple(g.seed_geom, g.seed_alm, (int)kind);
  auto it = g_seeds.find(key);
  if (it != g_seeds.end()) return &it->second;
  const int nwarps = (g.nslots + 32 * R - 1) / (32 * R);
  const size_t nst = (size_t)nm * g.nslots, nsl = (size_t)nm * nwarps;
  const size_t sbytes = (kind == SEED_S2 || kind == SEED_A2 ? 4 : 2) * sizeof(double);
  const size_t bytes = nst * (sbytes + sizeof(int)) + nsl * sizeof(int);
  static size_t cap = 0;
  if (!cap) { size_t fr, tot; CMDR_CUDA_CHECK(cudaMemGetInfo(&fr, &tot)); cap = tot / 32; }
  if (bytes > cap) return nullptr;
  SeedTab t;
  t.bytes = bytes;
  CMDR_CUDA_CHECK(cudaMalloc(&t.sl, nsl * sizeof(int)));
  CMDR_CUDA_CHECK(cudaMalloc(&t.ss, nst * sbytes));
  CMDR_CUDA_CHECK(cudaMalloc(&t.sk, nst * sizeof(int)));
  KParams q = p;   // all local m's, from slot 0
  q.im0 = 0; q.sl = t.sl; q.ss = t.ss; q.sk = t.sk;
  const dim3 grid(nwarps, nm);
  switch (kind) {
    case SEED_S0: case SEED_S0X: seed0_kernel<4><<<grid, 32, 0, st>>>(q); break;
    case SEED_A0: case SEED_A0X: seed0_kernel<8><<<grid, 32, 0, st>>>(q); break;
    case SEED_S2: seed2_kernel<4, 4, 8, false><<<grid, 32, 0, st>>>(q); break;
    case SEED_A2: seed2_kernel<4, 2, 4, true><<<grid, 32, 0, st>>>(q); break;
  }
  count_launch();
  CMDR_CUDA_CHECK(cudaGetLastError());
  CMDR_CUDA_CHECK(cudaStreamSynchronize(st));   // once per plan: other streams may use the table next
  g_seed_bytes += bytes;
  return &(g_seeds[key] = t);
}
static void use_seed(KParams &p, const SeedTab *t) { p.sl = t->sl; p.ss = t->ss; p.sk = t->sk; }

// ---- deterministic analysis (det.h): on with cmdr_sht_set_deterministic or CMDR_SHT_DETERMINISTIC=1 at load ----
static bool g_det = getenv("CMDR_SHT_DETERMINISTIC") && atoi(getenv("CMDR_SHT_DETERMINISTIC")) != 0;
bool deterministic() { return g_det; }
// slots per warp block of the deterministic kernels: anal0_kernel<8, ...>, anal2_kernel<4, ...> (the defaults; the
// CMDR_SHT_R_A0 / _A2 tuning overrides do not apply in this mode)
int det_block_slots(int spin) { return spin == 0 ? 32 * 8 : 32 * 4; }

// Partials of a launch whose blocks cover work slots [0, nslots) and local m's [im0, im0 + nm), ncomp components, in
// the library's scratch arena (one buffer: the kernels and the reduce of a transform run in stream order)
static DetArgs det_use(const KParams &p, int nslots, int im0, int nm, int ncomp) {
  DetArgs d;
  d.dl.nb = (nslots + det_block_slots(p.spin) - 1) / det_block_slots(p.spin);
  d.dl.nm = nm; d.dl.im0 = im0; d.dl.lmax = p.lmax;
  d.det = static_cast<double *>(scratch_get("det_part", sizeof(double) * d.dl.comp_stride() * ncomp));
  d.drec = static_cast<int *>(scratch_get("det_rec", sizeof(int) * (size_t)d.dl.nb * nm));
  return d;
}
// local m's per launch so that the partials take at most 1/16 of the device memory (decided once, as seed_table does);
// a launch over more m's runs as several launches over m ranges
static int det_m_per_launch(int nslots, int spin, int lmax, int ncomp) {
  static size_t cap = 0;
  if (!cap) { size_t fr, tot; CMDR_CUDA_CHECK(cudaMemGetInfo(&fr, &tot)); cap = tot / 16; }
  const size_t nb = (nslots + det_block_slots(spin) - 1) / det_block_slots(spin);
  const size_t per_m = nb * (sizeof(double) * 2 * (size_t)(lmax + 1) * ncomp + sizeof(int));
  return (int)std::max<size_t>(1, std::min<size_t>(cap / per_m, 1 << 30));
}
static void det_reduce(const KParams &p, const DetArgs &d, int nmr, int ncomp, cudaStream_t st) {
  det_reduce_kernel<<<dim3((unsigned)((d.dl.row() + 255) / 256), nmr), 256, 0, st>>>(p, d, ncomp);
  count_launch();
}
// the deterministic Legendre analysis kernel of `p` (partials set), seeded where the plain launch would be
static void det_anal_kernel(const LegGeom &g, const LegAlm &a, KParams p, const DetArgs &d, SeedKind kind, int nmr,
                            cudaStream_t st) {
  if (p.spin == 0) {
    if (const SeedTab *t = seed_table(g, kind, 8, p, a.nm, st)) { use_seed(p, t); launch_w<8>(anal0_kernel<8, 12, true, true>, p, nmr, st, d); }
    else launch_w<8>(anal0_kernel<8, 12, false, true>, p, nmr, st, d);
  } else {
    if (const SeedTab *t = p.spin == 2 ? seed_table(g, SEED_A2, 4, p, a.nm, st) : nullptr) {
      use_seed(p, t); launch_w<4>(anal2_kernel<4, 12, true, true>, p, nmr, st, d);
    } else {
      launch_w<4>(anal2_kernel<4, 12, false, true>, p, nmr, st, d);
    }
  }
  count_launch();
}

// ---- spin 2 as scalar sums (prep_s2s_kernel / post_s2s_kernel above) ----
static bool g_s2s_on = true;
bool spin2_scalar_on() { return g_s2s_on; }

static bool s2s_route(const LegGeom &g, const LegAlm &a) { return a.spin == 2 && !a.deriv1 && a.s2s_coef && g.s2s_npolar >= 0; }

// spin-0 view of a spin-2 launch: lmax + 2 and the two-l-per-step tables of that range, spin-2 m cut-off and slots
static KParams s2s_params(const LegGeom &g, const LegAlm &a, const KParams &p) {
  KParams q = p;
  q.lmax = a.lmax + 2; q.spin = 0;
  q.coef = a.s2s_coef; q.coef2 = a.s2s_mix; q.cofs = a.s2s_cofs; q.Kstart = a.s2s_K0; q.tofs = a.s2s_tofs;
  q.fcoef = nullptr;
  q.s2s_npolar = g.s2s_npolar;
  return q;
}

// Every slot runs the spin-0 kernels (so that their seed tables apply); the spin-2 kernel then overwrites the polar
// slots' phases.  `p`: the spin-2 parameters with the spin-2 tile rows.
static void launch_s2s_synth(const LegGeom &g, const LegAlm &a, const KParams &p, int nmr, cudaStream_t st, bool prep) {
  KParams q = s2s_params(g, a, p);
  q.trows = static_cast<double *>(scratch_get("synth_rows_s2s", sizeof(TileS0<2>) * (size_t)(a.s2s_trows + TL_S2S)));
  if (prep) {
    prep_s2s_kernel<<<dim3((a.lmax + 2 + 8 + 255) / 256, nmr), 256, 0, st>>>(q);
    count_launch();
  }
  if (const SeedTab *t = seed_table(g, SEED_S0X, 4, q, a.nm, st)) { use_seed(q, t); launch_w<4>(synth0_kernel<2, 4, 12, true>, q, nmr, st); }
  else launch_w<4>(synth0_kernel<2, 4, 12>, q, nmr, st);
  count_launch();
  if (g.s2s_npolar > 0) {
    KParams pp = p;
    pp.nslots = min(p.nslots, g.s2s_npolar);
    if (prep) {
      prep_s2_kernel<<<dim3((a.lmax + 8 + 255) / 256, nmr), 256, 0, st>>>(pp);
      count_launch();
    }
    launch_w<4>(synth2_kernel<4, 8>, pp, nmr, st);
    count_launch();
  }
  CMDR_CUDA_CHECK(cudaGetLastError());
}

// Polar rings contribute to the scalar sums with weight 0 and go through the spin-2 kernel instead; the post kernel
// then adds the transposed map of the sums to the a_lm.
static void launch_s2s_anal(const LegGeom &g, const LegAlm &a, const KParams &p, int nmr, cudaStream_t st) {
  KParams q = s2s_params(g, a, p);
  q.lscale0 = q.lscale1 = nullptr;   // applied by the post kernel
  const long long ctot = 2 * a.s2s_nl;   // doubles per component
  double *T = static_cast<double *>(scratch_get("anal_s2s", sizeof(double) * 2 * (size_t)ctot));
  CMDR_CUDA_CHECK(cudaMemsetAsync(T, 0, sizeof(double) * 2 * (size_t)ctot, st));
  if (g_det) {   // both scalar sums through the partials and the reduce into T, then the polar rings into the a_lm
    const DetArgs d = det_use(q, q.nslots, q.im0, nmr, 2);
    for (int c = 0; c < 2; ++c) {   // the two launches store the same records
      KParams qc = q;
      qc.comp0 = p.comp0 + c;
      DetArgs dc = d;
      dc.det = d.det + (size_t)c * d.dl.comp_stride();
      det_anal_kernel(g, a, qc, dc, SEED_A0X, nmr, st);
    }
    q.alm0 = T; q.alm1 = T + ctot;
    det_reduce(q, d, nmr, 2, st);
    if (g.s2s_npolar > 0) {
      KParams pp = p;
      pp.nslots = min(p.nslots, g.s2s_npolar);
      const DetArgs dp = det_use(pp, pp.nslots, pp.im0, nmr, 2);
      det_anal_kernel(g, a, pp, dp, SEED_A2, nmr, st);
      det_reduce(pp, dp, nmr, 2, st);
    }
  } else {
    const SeedTab *t = seed_table(g, SEED_A0X, 8, q, a.nm, st);
    if (t) use_seed(q, t);
    for (int c = 0; c < 2; ++c) {
      KParams qc = q;
      qc.comp0 = p.comp0 + c;
      qc.alm0 = T + (size_t)c * ctot;
      if (t) launch_w<8>(anal0_kernel<8, 12, true>, qc, nmr, st, DetArgs{});
      else launch_w<8>(anal0_kernel<8, 12>, qc, nmr, st, DetArgs{});
      count_launch();
    }
    if (g.s2s_npolar > 0) {
      KParams pp = p;
      pp.nslots = min(p.nslots, g.s2s_npolar);
      launch_w<4>(anal2_kernel<4, 12>, pp, nmr, st, DetArgs{});
      count_launch();
    }
  }
  post_s2s_kernel<<<dim3((a.lmax + 1 + 255) / 256, nmr), 256, 0, st>>>(p, T, a.s2s_cofs, ctot);
  count_launch();
  CMDR_CUDA_CHECK(cudaGetLastError());
}

void launch_legendre_synth(const LegGeom &g, const LegAlm &a, const double *const *alm, double4 *ph, cudaStream_t st,
                           bool prep) {
  if (a.nm == 0 || g.nslots == 0) return;
  const int nmr = (a.im_end >= 0 ? a.im_end : a.nm) - a.im_begin;   // local m's of this launch
  if (nmr <= 0) return;
  const int spin = a.spin;
  // DERIV1 reads one a_lm column: never touch alm[1]
  KParams p = make_params(g, a, const_cast<double *>(alm[0]), (spin && !a.deriv1) ? const_cast<double *>(alm[1]) : nullptr, ph);
  // tile rows {A', [C',] g a_lm} for all local (m, l): written once per transform (`prep`), then
  // streamed by every warp of the Legendre kernel
  const size_t rowbytes = spin == 0 ? sizeof(TileS0<1>) : (a.deriv1 ? sizeof(TileD1) : sizeof(TileS2));
  p.tofs = a.tofs;
  p.trows = static_cast<double *>(scratch_get(spin == 0 ? "synth_rows0" : "synth_rows2", rowbytes * (size_t)(a.trows + TL)));
  if (s2s_route(g, a)) { launch_s2s_synth(g, a, p, nmr, st, prep); return; }
  if (prep) {
    dim3 pg((a.lmax + 8 + 255) / 256, nmr);
    if (spin == 0) prep_s0_kernel<<<pg, 256, 0, st>>>(p);
    else if (a.deriv1) prep_d1_kernel<<<pg, 256, 0, st>>>(p);
    else prep_s2_kernel<<<pg, 256, 0, st>>>(p);
    count_launch();
  }
  static const int r0 = env_int("CMDR_SHT_R_S0", 4), r2 = env_int("CMDR_SHT_R_S2", 4);
  static const int b0 = env_int("CMDR_SHT_MINB_S0", 16), b2 = env_int("CMDR_SHT_MINB_S2", 8);
  static const int rd = env_int("CMDR_SHT_R_D1", 2), bd = env_int("CMDR_SHT_MINB_D1", 16);
  if (a.deriv1) {
    switch (rd * 100 + bd) {
      case 312: launch_w<3>(synth_d1_kernel<3, 12>, p, nmr, st); break;
      case 412: launch_w<4>(synth_d1_kernel<4, 12>, p, nmr, st); break;
      case 408: launch_w<4>(synth_d1_kernel<4, 8>, p, nmr, st); break;
      default: launch_w<2>(synth_d1_kernel<2, 16>, p, nmr, st); break;
    }
  } else if (spin == 0) {
    switch (r0 * 100 + b0) {
      case 216: launch_w<2>(synth0_kernel<1, 2, 16>, p, nmr, st); break;
      case 412: launch_w<4>(synth0_kernel<1, 4, 12>, p, nmr, st); break;
      case 612: launch_w<6>(synth0_kernel<1, 6, 12>, p, nmr, st); break;
      case 812: launch_w<8>(synth0_kernel<1, 8, 12>, p, nmr, st); break;
      case 808: launch_w<8>(synth0_kernel<1, 8, 8>, p, nmr, st); break;
      default:
        if (const SeedTab *t = seed_table(g, SEED_S0, 4, p, a.nm, st)) { use_seed(p, t); launch_w<4>(synth0_kernel<1, 4, 16, true>, p, nmr, st); }
        else launch_w<4>(synth0_kernel<1, 4, 16>, p, nmr, st);
        break;
    }
  } else {
    switch (r2 * 100 + b2) {
      case 116: launch_w<1>(synth2_kernel<1, 16>, p, nmr, st); break;
      case 212: launch_w<2>(synth2_kernel<2, 12>, p, nmr, st); break;
      case 312: launch_w<3>(synth2_kernel<3, 12>, p, nmr, st); break;
      case 308: launch_w<3>(synth2_kernel<3, 8>, p, nmr, st); break;
      case 412: launch_w<4>(synth2_kernel<4, 12>, p, nmr, st); break;
      case 408:
        if (const SeedTab *t = spin == 2 ? seed_table(g, SEED_S2, 4, p, a.nm, st) : nullptr) {
          use_seed(p, t); launch_w<4>(synth2_kernel<4, 12, true>, p, nmr, st);   // 12: the 8 of the unseeded kernel lets the seeded one take 170 registers, one warp per SM fewer
        } else {
          launch_w<4>(synth2_kernel<4, 8>, p, nmr, st);
        }
        break;
      default: launch_w<2>(synth2_kernel<2, 16>, p, nmr, st); break;
    }
  }
  count_launch();
  CMDR_CUDA_CHECK(cudaGetLastError());
}

void launch_legendre_anal(const LegGeom &g, const LegAlm &a, double *const *alm, const double4 *ph, cudaStream_t st,
                          bool reduce) {
  if (a.nm == 0 || g.nslots == 0) return;
  const int nmr = (a.im_end >= 0 ? a.im_end : a.nm) - a.im_begin;   // local m's of this launch
  if (nmr <= 0) return;
  const int spin = a.spin;
  KParams p = make_params(g, a, alm[0], spin ? alm[1] : nullptr, const_cast<double4 *>(ph));
  if (g_det) {
    if (p.slot_begin % det_block_slots(spin) != 0 || (!reduce && s2s_route(g, a)) || (reduce && p.slot_begin != 0)) {
      fprintf(stderr, "cmdr_sht: deterministic analysis launched over slots [%d, %d), not a cut on warp blocks\n", p.slot_begin, p.nslots);
      abort();
    }
    if (!reduce) {   // one piece of a pipelined analysis: partials of the whole geometry and every local m
      det_anal_kernel(g, a, p, det_use(p, g.nslots, 0, a.nm, spin ? 2 : 1), SEED_A0, nmr, st);
      CMDR_CUDA_CHECK(cudaGetLastError());
      return;
    }
    const int s2s = s2s_route(g, a);
    const int mpl = det_m_per_launch(p.nslots, s2s ? 0 : spin, s2s ? a.lmax + 2 : a.lmax, spin ? 2 : 1);
    for (int i0 = a.im_begin; i0 < a.im_begin + nmr; i0 += mpl) {
      const int n = std::min(mpl, a.im_begin + nmr - i0);
      KParams pi = p;
      pi.im0 = i0;
      if (s2s) { launch_s2s_anal(g, a, pi, n, st); continue; }
      const DetArgs d = det_use(pi, pi.nslots, i0, n, spin ? 2 : 1);
      det_anal_kernel(g, a, pi, d, SEED_A0, n, st);
      det_reduce(pi, d, n, spin ? 2 : 1, st);
    }
    CMDR_CUDA_CHECK(cudaGetLastError());
    return;
  }
  if (s2s_route(g, a)) { launch_s2s_anal(g, a, p, nmr, st); return; }
  // spin 0: 8 ring pairs per thread since the two-l-per-step kernels (fewer registers per ring pair; the butterfly and the
  // per-tile flush are per warp, so their share halves): 8.71 -> 8.31 ms at nside 2048 / lmax 4000
  static const int r0 = env_int("CMDR_SHT_R_A0", 8), r2 = env_int("CMDR_SHT_R_A2", 4);
  // resident warps per SM the register allocation is capped for (tuning: CMDR_SHT_MINB_A0 / _A2)
  static const int b0 = env_int("CMDR_SHT_MINB_A0", 12), b2 = env_int("CMDR_SHT_MINB_A2", 12);
  if (spin == 0) {
    switch (r0 * 100 + b0) {
      case 416: launch_w<4>(anal0_kernel<4, 16>, p, nmr, st, DetArgs{}); break;
      case 408: launch_w<4>(anal0_kernel<4, 8>, p, nmr, st, DetArgs{}); break;
      case 612: launch_w<6>(anal0_kernel<6, 12>, p, nmr, st, DetArgs{}); break;
      case 608: launch_w<6>(anal0_kernel<6, 8>, p, nmr, st, DetArgs{}); break;
      case 812:
        if (const SeedTab *t = seed_table(g, SEED_A0, 8, p, a.nm, st)) { use_seed(p, t); launch_w<8>(anal0_kernel<8, 12, true>, p, nmr, st, DetArgs{}); }
        else launch_w<8>(anal0_kernel<8, 12>, p, nmr, st, DetArgs{});
        break;
      case 808: launch_w<8>(anal0_kernel<8, 8>, p, nmr, st, DetArgs{}); break;
      default: launch_w<4>(anal0_kernel<4, 12>, p, nmr, st, DetArgs{}); break;
    }
  } else {
    switch (r2 * 100 + b2) {
      case 312: launch_w<3>(anal2_kernel<3, 12>, p, nmr, st, DetArgs{}); break;
      case 308: launch_w<3>(anal2_kernel<3, 8>, p, nmr, st, DetArgs{}); break;
      case 216: launch_w<2>(anal2_kernel<2, 16>, p, nmr, st, DetArgs{}); break;
      case 212: launch_w<2>(anal2_kernel<2, 12>, p, nmr, st, DetArgs{}); break;
      case 412:
        if (const SeedTab *t = spin == 2 ? seed_table(g, SEED_A2, 4, p, a.nm, st) : nullptr) {
          use_seed(p, t); launch_w<4>(anal2_kernel<4, 12, true>, p, nmr, st, DetArgs{});
        } else {
          launch_w<4>(anal2_kernel<4, 12>, p, nmr, st, DetArgs{});
        }
        break;
      case 410: launch_w<4>(anal2_kernel<4, 10>, p, nmr, st, DetArgs{}); break;
      default: launch_w<4>(anal2_kernel<4, 8>, p, nmr, st, DetArgs{}); break;
    }
  }
  count_launch();
  CMDR_CUDA_CHECK(cudaGetLastError());
}

void legendre_anal_reduce(const LegGeom &g, const LegAlm &a, double *const *alm, cudaStream_t st) {
  if (!g_det || a.nm == 0 || g.nslots == 0) return;
  const int nmr = (a.im_end >= 0 ? a.im_end : a.nm) - a.im_begin;
  if (nmr <= 0) return;
  KParams p = make_params(g, a, alm[0], a.spin ? alm[1] : nullptr, nullptr);
  det_reduce(p, det_use(p, g.nslots, 0, a.nm, a.spin ? 2 : 1), nmr, a.spin ? 2 : 1, st);
  CMDR_CUDA_CHECK(cudaGetLastError());
}

}  // namespace cmdr

extern "C" {
void cmdr_sht_set_legendre_seeds(int on) { cmdr::g_seeds_on = on != 0; }
void cmdr_sht_set_spin2_scalar(int on) { cmdr::g_s2s_on = on != 0; }
void cmdr_sht_set_deterministic(int on) { cmdr::g_det = on != 0; }
int cmdr_sht_deterministic(void) { return cmdr::g_det ? 1 : 0; }
size_t cmdr_sht_legendre_seed_bytes(void) { return cmdr::g_seed_bytes; }
}
