// qd_kernels.cuh -- the per-pixel charge-stability kernels (Path A), hand-written for sm_100a.
//
// Work decomposition
//   item  = (scan, block of rows).  One WARP owns one item at a time and is fully independent of the other warps of
//           its CTA (no __syncthreads anywhere): it stages the env's model record and the scan descriptor into its own
//           shared-memory slot with two TMA bulk copies on one mbarrier, derives the affine coefficients
//           g(ix,iy) = g0 + ix*gx + iy*gy of the dot potentials (the voltage grid itself is never materialised), then
//           walks its rows.  Within a row the 32 lanes take 32 consecutive pixels (fast axis x), so the fp32 sensor
//           image and the uint8 charge map are written with fully coalesced 128 B / 32*N B warp stores.
//   pixel = one thread: exact continuous relaxation (only when some dot potential is negative), floor, 2^N candidate
//           search, then -- cooperatively across the warp, sequential along x -- hysteresis latching and the
//           telegraph-noise chain, then the sensor Lorentzians and the noise terms.
//
// Candidate search without the O(N^2) quadratic form per candidate.  With r = floor(n_c) - g and h = Cinv r,
//     E(delta) = (r+delta)^T Cinv (r+delta) = r.h + sum_j delta_j 2 h_j + Q[delta],   Q[delta] = delta^T Cinv delta.
//   Q depends on the env only: 2^N doubles precomputed at qd_set_models and staged with the record.  Exact dominance
//   bounds fix most dots first (ground_state_box, step 2); the 0-3 undecided ones are walked in Gray-code order (one
//   term of the linear part and one Q look-up per step, step 3a).  Wide cases and kT > 0 use the block enumeration
//   (3b): the linear part splits over the low/high halves of the bit string, L(delta) = Lhi[H] + Llo[b], Llo (<= 16
//   values) in registers, one broadcast LDS per two candidates.  Either way the winner is the first minimum of the
//   ascending enumeration (dot 0 most significant), as in oracle/path_a.py.
#pragma once
#include <math.h>

#include "qd_device.cuh"
#include "qd_layout.h"

namespace qd {

struct KArgs {
  qd_layout L;
  const double* __restrict__ records;
  const qd_scan* __restrict__ scans;
  const double* __restrict__ points;   // [pixels, n_volt] or nullptr (affine scans)
  float* __restrict__ z_out;
  void* __restrict__ n_out;
  double* __restrict__ nbar;           // tunnel path: <n> per pixel, [pixels, N] (written by qd_tunnel_gs_kernel)
  unsigned* status;                    // sticky QD_STATUS_* word (host-mapped): written only when something is wrong
  // tunnel path, split pipeline (qd_tunnel_relax / select / eigen kernels): per-pixel scratch of the current chunk of
  // scans, addressed by (scan index inside the chunk) * tstride + pixel
  unsigned char* tfloor;               // [slots][8]   floor of the relaxed continuous occupations
  unsigned long long* tkeys;           // [slots][32]  the 32 kept basis states, 8 bits per dot
  double* tpot;                        // [slots][16]  dot potentials g[0..8), tunnel couplings |t|[8..15), cdd scale s_c [15]
  long long tstride;                   // pixels per scan slot (largest scan of the upload)
  int topt;                            // tunnel path: optimisation switches (QDSIM_TUNNEL_OPT, default all on; A/B and bisection)
  // tunnel path, select / eigen kernels: a fix-up launch redoes only the pixels the marking kernel (select2 / eigen2)
  // marked; its items are shorter than the marking kernel's, whose item length (pixels) locates the item-level marks
  int fixup;
  int mark_ppi;
  float e2_kappa, e2_qsafe, e2_tol;    // qd_tunnel_eigen2_kernel: shift aggressiveness, contraction safety factor, stopping tolerance
  // single-scan fast path (one do2d_open): the descriptor travels in the kernel parameters instead of through a
  // host-to-device copy; `scans` is then unused
  int use_one;
  qd_scan one;
  int n_scan;
  int n_type;
  unsigned flags;
  int rows_per_item;
  int items_per_scan;
  int slot_bytes;
  int col_parts;                       // items per row block along x (> 1 only when nothing is carried along a row: no
                                       // latching, telegraph or 1/f chain) -- small launches spread over more SMs
};

constexpr int QD_DER_DOUBLES = 48;  // derived per-item block: g0[8] gx[8] gy[8] us0 usx usy pad[5] carry[8] + spare
constexpr int QD_PC_DOUBLES = 8 * 64 + 8 * 16 + 8 + 8 * 32 + 8 * 24;   // projection cache: 8 matrices, inversion scratch, keys + meta; per-lane lin[8]; affine forms

constexpr int QD_BF_DOUBLES = 8 + 64 + 8;   // brute force, per item: d[8], U[64] of the PERMUTED cdd_inv, perm / inverse perm (16 ints)

__host__ __device__ inline int qd_slot_bytes(const qd_layout& L) {
  int b = L.rec_doubles * 8 + (int)sizeof(qd_scan) + QD_DER_DOUBLES * 8 + 16;
  if (L.algorithm == QD_ALG_DEFAULT || L.algorithm == QD_ALG_THRESHOLDED) b += QD_PC_DOUBLES * 8;
  if (L.algorithm == QD_ALG_BRUTE_FORCE) b += QD_BF_DOUBLES * 8;
  return (b + 127) & ~127;
}

// ---------------------------------------------------------------------------------------------------------------
// Exact continuous relaxation: min (n-g)^T cdd^{-1} (n-g), n >= 0  (monotone active set on the M-matrix cdd;
// oracle/path_a.py: continuous_relaxation).
//
// For an active (clamped) set S the solution is LINEAR in g:  w = P_S g,  P_S = I - cdd[:,S] (cdd_SS)^{-1} E_S^T, and P_S
// depends on the env and on S only -- not on the pixel.  A scan meets a handful of distinct S (the swept dots cross
// zero, the others are clamped or free throughout), so each warp keeps a small cache of P_S matrices in its shared
// memory slot, built cooperatively by the 32 lanes (Gauss-Jordan on the masked matrix) on a miss.  Per pixel a round
// of the active-set iteration is then one N x N mat-vec with broadcast shared-memory operands.
// ---------------------------------------------------------------------------------------------------------------
#ifndef QD_MIN_BLOCKS
#define QD_MIN_BLOCKS 3
#endif
#ifndef QD_CTA_WARPS
#define QD_CTA_WARPS 4          // warps per CTA of qd_scan_kernel (the warps are independent: any value works)
#endif
constexpr int QD_PC_WAYS = 8;

// y = M x for a row-major N x N fp64 matrix in shared memory (16-byte aligned), all lanes reading the same elements:
// broadcast LDS.128 fetches two matrix entries per load when N is even.
template <int N>
__device__ __forceinline__ void matvec_smem(const double* __restrict__ M, const double (&x)[N], double (&y)[N]) {
  if constexpr (N % 2 == 0) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      double s0 = 0.0, s1 = 0.0;
#pragma unroll
      for (int j = 0; j < N; j += 2) {
        const double2 m = *reinterpret_cast<const double2*>(M + i * N + j);
        s0 = fma(m.x, x[j], s0);
        s1 = fma(m.y, x[j + 1], s1);
      }
      y[i] = s0 + s1;
    }
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      double s0 = 0.0;
#pragma unroll
      for (int j = 0; j < N; ++j) s0 = fma(M[i * N + j], x[j], s0);
      y[i] = s0;
    }
  }
}
struct ProjCache {
  double* aff;      // [QD_PC_WAYS][3][8]: P_S g0, P_S gx, P_S gy -- the relaxed occupations are affine in the pixel indices
  const double* gsrc;  // g0[8] gx[8] gy[8] of the current item (nullptr: explicit voltage list, no affine form)
  double* lin_s;    // [8][32]: per-lane copy of the linear coefficients, indexed by BIT position (free-bit enumeration)
  uint32_t* keys;   // [QD_PC_WAYS]
  uint32_t* meta;   // [0] = entries in use, [1] = next victim
  double* mats;     // [QD_PC_WAYS][64]  (mat_stride = 64), or one scratch matrix (mat_stride = 0: affine forms only)
  double* aug;      // [8][16] scratch of the cooperative inversion
  int mat_stride;
};

template <int N>
__device__ __noinline__ int proj_cache_build(const ProjCache& pc, const double* __restrict__ cdd, unsigned S, int lane) {
  constexpr int W = 2 * N;
  double* A = pc.aug;
  for (int e = lane; e < N * W; e += 32) {
    const int r = e / W, c = e - r * W;
    double v;
    if (c < N) v = (((S >> r) & 1u) && ((S >> c) & 1u)) ? cdd[r * N + c] : (r == c ? 1.0 : 0.0);
    else v = (r == c - N) ? 1.0 : 0.0;
    A[e] = v;
  }
  __syncwarp();
  for (int k = 0; k < N; ++k) {
    if (!((S >> k) & 1u)) continue;                      // identity pivot
    const double inv = 1.0 / A[k * W + k];
    double rowk[(N * W + 31) / 32], fr[(N * W + 31) / 32];
#pragma unroll
    for (int t = 0; t < (N * W + 31) / 32; ++t) {
      const int e = lane + 32 * t;
      if (e < N * W) {
        const int r = e / W, c = e - r * W;
        rowk[t] = A[k * W + c] * inv;
        fr[t] = A[r * W + k];
      }
    }
    __syncwarp();
#pragma unroll
    for (int t = 0; t < (N * W + 31) / 32; ++t) {
      const int e = lane + 32 * t;
      if (e < N * W) {
        const int r = e / W;
        A[e] = (r == k) ? rowk[t] : A[e] - fr[t] * rowk[t];
      }
    }
    __syncwarp();
  }
  // victim slot (round robin) and P_S = I - cdd[:,S] K[S,:] restricted to columns in S; rows in S are zero
  const int slot = (int)pc.meta[1];
  double* P = pc.mats + slot * pc.mat_stride;
  for (int e = lane; e < N * N; e += 32) {
    const int i = e / N, j = e - i * N;
    double v = (i == j) ? 1.0 : 0.0;
    if ((S >> j) & 1u) {
      for (int q = 0; q < N; ++q)
        if ((S >> q) & 1u) v -= cdd[i * N + q] * A[q * W + N + j];
    }
    if ((S >> i) & 1u) v = 0.0;
    P[e] = v;
  }
  __syncwarp();
  if (pc.gsrc != nullptr && lane < 24) {
    // g = g0 + ix gx + iy gy on an affine scan, so w = P_S g = (P_S g0) + ix (P_S gx) + iy (P_S gy): three small
    // mat-vecs per (item, S) replace one per pixel and round
    const int t = lane >> 3, i = lane & 7;
    double acc = 0.0;
    if (i < N) {
      const double* src = pc.gsrc + 8 * t;
      for (int j = 0; j < N; ++j) acc = fma(P[i * N + j], src[j], acc);
    }
    pc.aff[slot * 24 + lane] = acc;
  }
  if (lane == 0) {
    pc.keys[slot] = S;
    pc.meta[1] = (uint32_t)((slot + 1) % QD_PC_WAYS);
    if (pc.meta[0] < QD_PC_WAYS) pc.meta[0] += 1;
  }
  __syncwarp();
  return slot;
}

template <int N, bool AFFINE>
__device__ __forceinline__ void relax_lcp(const double (&g)[N], const double* __restrict__ cdd, const ProjCache& pc,
                                          int lane, double fx, double fy, double (&nc)[N]) {
  unsigned act = 0;
#pragma unroll
  for (int j = 0; j < N; ++j) act |= ((unsigned)__double2hiint(g[j]) >> 31) << j;     // sign bits (a -0.0 clamps to 0 too)
  bool need = act != 0;
#pragma unroll
  for (int j = 0; j < N; ++j) nc[j] = g[j];
#pragma unroll 1
  for (int round = 0; round <= N; ++round) {
    unsigned pend = __ballot_sync(0xffffffffu, need);
    if (!pend) break;
    bool changed = false;
    while (pend) {
      const int leader = __ffs(pend) - 1;
      const unsigned S = __shfl_sync(0xffffffffu, act, leader);
      const bool member = need && act == S;
      pend &= ~__ballot_sync(0xffffffffu, member);
      const unsigned hit = __ballot_sync(0xffffffffu, lane < (int)pc.meta[0] && pc.keys[lane & (QD_PC_WAYS - 1)] == S &&
                                                          lane < QD_PC_WAYS);
      const int slot = hit ? __ffs(hit) - 1 : proj_cache_build<N>(pc, cdd, S, lane);
      if (member) {
        const double* __restrict__ P = pc.mats + slot * pc.mat_stride;
        unsigned neu = act;
        double wv[N];
        if constexpr (AFFINE) {
          const double* __restrict__ A = pc.aff + slot * 24;
          if constexpr (N % 2 == 0) {
#pragma unroll
            for (int i = 0; i < N; i += 2) {
              const double2 a0 = *reinterpret_cast<const double2*>(A + i);
              const double2 ax = *reinterpret_cast<const double2*>(A + 8 + i);
              const double2 ay = *reinterpret_cast<const double2*>(A + 16 + i);
              wv[i] = fma(fy, ay.x, fma(fx, ax.x, a0.x));
              wv[i + 1] = fma(fy, ay.y, fma(fx, ax.y, a0.y));
            }
          } else {
#pragma unroll
            for (int i = 0; i < N; ++i) wv[i] = fma(fy, A[16 + i], fma(fx, A[8 + i], A[i]));
          }
        } else {
          matvec_smem<N>(P, g, wv);
        }
#pragma unroll
        for (int i = 0; i < N; ++i) {
          const double sacc = ((act >> i) & 1u) ? 0.0 : wv[i];
          nc[i] = sacc;
          neu |= ((unsigned)__double2hiint(sacc) >> 31) << i;
        }
        changed = neu != act;
        act = neu;
      }
      __syncwarp();
    }
    need = changed;
  }
  // (a lane leaves the loop only after a round that produced no negative entry, so nc >= 0 here)
}

// ---------------------------------------------------------------------------------------------------------------
// default / thresholded ground state of one pixel.  nd[] <- occupations (integers when kT == 0).
// ---------------------------------------------------------------------------------------------------------------
template <int N, bool THERMAL, bool AFFINE>
__device__ __forceinline__ void ground_state_box(const double (&g)[N], const double* __restrict__ rec,
                                                 const qd_layout& L, const ProjCache& pc, int lane, bool thresholded,
                                                 double kT, double fx, double fy, double (&nd)[N]) {
  constexpr int NLO = N < 4 ? N : 4;
  constexpr int NHI = N - NLO;
  constexpr int LOC = 1 << NLO;
  const double* __restrict__ cinv = rec + L.o_cinv;
  const double* __restrict__ Q = rec + L.o_q;

  // any g_j < 0?  OR of the sign words (a -0.0 only costs a relax_lcp call that returns at once)
  int sgn = 0;
#pragma unroll
  for (int j = 0; j < N; ++j) sgn |= __double2hiint(g[j]);
  const bool neg = sgn < 0;
  double nc[N];
#pragma unroll
  for (int j = 0; j < N; ++j) nc[j] = g[j];
  if (__any_sync(0xffffffffu, neg)) relax_lcp<N, AFFINE>(g, rec + L.o_cdd, pc, lane, fx, fy, nc);

  double f[N], r[N], lin[N];
#pragma unroll
  for (int j = 0; j < N; ++j) {
    f[j] = floor(nc[j]);
    r[j] = f[j] - g[j];
  }
  matvec_smem<N>(cinv, r, lin);
#pragma unroll
  for (int i = 0; i < N; ++i) lin[i] *= 2.0;
  // Restrictions on the candidate box.  bit (N-1-j) <-> dot j;  fixmask: bit is fixed, fixval: its value.
  // (1) thresholded: dots that keep only round(n_c).
  unsigned fixmask = 0, fixval = 0;
  if (thresholded) {
    const double half_thr = 0.5 * rec[L.o_par + QD_PAR_THRESHOLD];
#pragma unroll
    for (int j = 0; j < N; ++j) {
      const double frac = nc[j] - f[j];
      if (!(fabs(frac - 0.5) < half_thr)) {
        fixmask |= 1u << (N - 1 - j);
        if (floor(nc[j] + 0.5) - f[j] == 1.0) fixval |= 1u << (N - 1 - j);
      }
    }
  }
  const unsigned thr_mask = fixmask, thr_val = fixval;
  // (2) exact dominance: raising dot j from 0 to 1 changes E by  a_j + 2 sum_{k != j} Cinv_jk delta_k, which lies in
  //     [a_j + sneg_j, a_j + spos_j] whatever the other dots do (a_j = 2 h_j + Cinv_jj).  If that interval is strictly
  //     positive the minimiser has delta_j = 0, if strictly negative delta_j = 1.  Only the undecided dots are
  //     enumerated; the 1e-9 guard keeps every near-tie inside the enumeration, so the argmin is unchanged.
  {
    const double* __restrict__ spos = rec + L.o_spos;
    const double* __restrict__ sneg = rec + L.o_sneg;
    unsigned zmask = 0, omask = 0;
#pragma unroll
    for (int j = 0; j < N; ++j) {
      const unsigned bit = 1u << (N - 1 - j);
      const double aj = lin[j] + cinv[j * N + j];
      zmask |= (aj + sneg[j] > 1e-9) ? bit : 0u;
      omask |= (aj + spos[j] < -1e-9) ? bit : 0u;
    }
    const unsigned add = (zmask | omask) & ~fixmask;       // thresholded bits keep their own value
    fixval |= omask & add;
    fixmask |= add;
  }
  const double INF = __longlong_as_double(0x7ff0000000000000LL);
  double llo[LOC];
  double best = INF;
  int bidx = 0;
  // ---- (3a) few undecided dots everywhere in the warp: enumerate only those, Gray-code order ----
  // After (1) and (2) a pixel typically has 0-3 free dots.  E(delta) = sum_j delta_j lin_j + Q[delta] (+ const): walking
  // the 2^k settings of the free bits in Gray-code order changes one term of the linear part per step and costs one
  // table look-up.  The winner is the lexicographic (energy, index) minimum = the first minimum of the ascending
  // enumeration below.  The warp runs 2^kmax steps; wide cases (kmax > 4) take the block enumeration (3b).
  const unsigned freeb = ~fixmask & ((1u << N) - 1u);
  const int kfree = __popc(freeb);
  const int kmax = __reduce_max_sync(0xffffffffu, kfree);
  if (kmax <= 4) {
    double* __restrict__ ls = pc.lin_s + lane;
    unsigned idx = fixval, pos = 0;
    double Lsum = 0.0;
    {
      int nfree = 0;
#pragma unroll
      for (int p = 0; p < N; ++p) {
        const double lp = lin[N - 1 - p];
        ls[p * 32] = lp;
        if ((fixval >> p) & 1u) Lsum += lp;
        if ((freeb >> p) & 1u) { pos |= (unsigned)p << (4 * nfree); ++nfree; }
      }
    }
    best = Lsum + Q[idx];
    bidx = (int)idx;
    const unsigned steps = 1u << kmax, mine = 1u << kfree;
#pragma unroll 1
    for (unsigned c = 1; c < steps; ++c) {
      if (c < mine) {
        const unsigned p = (pos >> (4 * (__ffs(c) - 1))) & 15u;
        idx ^= 1u << p;
        const double lp = ls[p * 32];
        Lsum += ((idx >> p) & 1u) ? lp : -lp;
        const double e = Lsum + Q[idx];
        if (e < best || (e == best && (int)idx < bidx)) { best = e; bidx = (int)idx; }
      }
    }
  } else {
  // ---- (3b) block enumeration: low half in registers, high halves on demand ----
  llo[0] = 0.0;
#pragma unroll
  for (int p = 0; p < NLO; ++p)
#pragma unroll
    for (int b = 0; b < (1 << p); ++b) llo[b + (1 << p)] = llo[b] + lin[N - 1 - p];
#pragma unroll
  for (int b = 0; b < LOC; ++b)
    if (((unsigned)b ^ fixval) & fixmask & (LOC - 1)) llo[b] = INF;

  double best_m = INF;
  int best_h = 0;
  // high halves H still allowed for this pixel, as a bit set over H; one warp-wide OR gives the H values the warp has
  // to visit at all (a single REDUX instead of a vote per H)
  unsigned okset = (NHI == 0) ? 1u : ((NHI >= 5) ? 0xffffffffu : ((1u << (1 << NHI)) - 1u));
#pragma unroll
  for (int p = 0; p < NHI; ++p) {
    // H values whose bit p is set: 0xAAAAAAAA, 0xCCCCCCCC, 0xF0F0F0F0, 0xFF00FF00, 0xFFFF0000
    const unsigned ones = (p == 0) ? 0xAAAAAAAAu : (p == 1) ? 0xCCCCCCCCu : (p == 2) ? 0xF0F0F0F0u : (p == 3) ? 0xFF00FF00u : 0xFFFF0000u;
    const unsigned bit = 1u << (NLO + p);
    if (fixmask & bit) okset &= (fixval & bit) ? ones : ~ones;
  }
  unsigned visit = __reduce_or_sync(0xffffffffu, okset);
#pragma unroll 1
  while (visit) {
    const int H = __ffs(visit) - 1;
    visit &= visit - 1u;
    const bool ok = (okset >> H) & 1u;
    double lh = 0.0;
#pragma unroll
    for (int p = 0; p < NHI; ++p) lh += ((H >> p) & 1) ? lin[N - 1 - NLO - p] : 0.0;
    if (!ok) lh = INF;
    const double* __restrict__ q = Q + (H << NLO);
    double m0 = INF, m1 = INF;                            // two independent min chains
    if constexpr (LOC >= 2) {
#pragma unroll
      for (int b = 0; b < LOC; b += 2) {
        const double2 qq = *reinterpret_cast<const double2*>(q + b);
        const double e0 = llo[b] + qq.x;
        const double e1 = llo[b + 1] + qq.y;
        m0 = min_lt(e0, m0);
        m1 = min_lt(e1, m1);
      }
    } else {
      m0 = llo[0] + q[0];
    }
    const double m = min_lt(m1, m0);
    const double e = m + lh;
    if (e < best) { best = e; best_m = m; best_h = H; }
  }
  // index of the first candidate of the winning high half that attains the minimum (ascending order, ties -> lowest)
  bidx = best_h << NLO;
  {
    const double* __restrict__ q = Q + (best_h << NLO);
    int mb = 0;
#pragma unroll
    for (int b = LOC - 1; b >= 0; --b)
      if (llo[b] + q[b] == best_m) mb = b;
    bidx |= mb;
  }
  }

  if (THERMAL && kT > 0.0) {
    // Boltzmann average over the same candidates, weights exp(-(E - Emin)/kT)
    const double inv_kT = 1.0 / kT;
    double Z = 0.0;
    double acc[N];
#pragma unroll
    for (int j = 0; j < N; ++j) acc[j] = 0.0;
    // Every candidate the algorithm allows carries weight exp(-(E - Emin)/kT), cut at 40 kT (4e-18).  A dot whose flip
    // costs more than that cut-off whatever the others do (the dominance bounds of step 2 with margin 40 kT) has one
    // value in every candidate that survives the cut, so only the remaining dots are walked (Gray code, as in 3a).
    const double cut = 40.0 * kT;
    unsigned tmask = thr_mask, tval = thr_val;
    {
      const double* __restrict__ spos = rec + L.o_spos;
      const double* __restrict__ sneg = rec + L.o_sneg;
      unsigned zt = 0, ot = 0;
#pragma unroll
      for (int j = 0; j < N; ++j) {
        const unsigned bit = 1u << (N - 1 - j);
        const double aj = lin[j] + cinv[j * N + j];
        zt |= (aj + sneg[j] > cut) ? bit : 0u;
        ot |= (aj + spos[j] < -cut) ? bit : 0u;
      }
      const unsigned add = (zt | ot) & ~tmask;
      tval |= ot & add;
      tmask |= add;
    }
    const unsigned freet = ~tmask & ((1u << N) - 1u);
    const int kft = __popc(freet);
    const int kmt = __reduce_max_sync(0xffffffffu, kft);
    if (kmt <= 6) {
      double* __restrict__ ls = pc.lin_s + lane;
      unsigned idx = tval, pos = 0;
      double Lsum = 0.0, Z = 0.0;
      {
        int nfree = 0;
#pragma unroll
        for (int p = 0; p < N; ++p) {
          const double lp = lin[N - 1 - p];
          ls[p * 32] = lp;
          if ((tval >> p) & 1u) Lsum += lp;
          if ((freet >> p) & 1u) { pos |= (unsigned)p << (4 * nfree); ++nfree; }
        }
      }
      const unsigned steps = 1u << kmt, mine = 1u << kft;
#pragma unroll 1
      for (unsigned c = 0; c < steps; ++c) {
        if (c < mine) {
          if (c > 0) {
            const unsigned p = (pos >> (4 * (__ffs(c) - 1))) & 15u;
            idx ^= 1u << p;
            const double lp = ls[p * 32];
            Lsum += ((idx >> p) & 1u) ? lp : -lp;
          }
          const double d = ((Lsum + Q[idx]) - best) * inv_kT;
          if (d < 40.0) {
            const double wgt = exp(-d);
            Z += wgt;
#pragma unroll
            for (int j = 0; j < N; ++j)
              if ((idx >> (N - 1 - j)) & 1u) acc[j] += wgt;
          }
        }
      }
      const double invZ = 1.0 / Z;
#pragma unroll
      for (int j = 0; j < N; ++j) nd[j] = f[j] + acc[j] * invZ;
      return;
    }
    llo[0] = 0.0;
#pragma unroll
    for (int p = 0; p < NLO; ++p)
#pragma unroll
      for (int b = 0; b < (1 << p); ++b) llo[b + (1 << p)] = llo[b] + lin[N - 1 - p];
#pragma unroll
    for (int b = 0; b < LOC; ++b)
      if (((unsigned)b ^ thr_val) & thr_mask & (LOC - 1)) llo[b] = INF;
#pragma unroll 1
    for (int H = 0; H < (1 << NHI); ++H) {
      double lh = 0.0;
#pragma unroll
      for (int p = 0; p < NHI; ++p) lh += ((H >> p) & 1) ? lin[N - 1 - NLO - p] : 0.0;
      if ((((unsigned)H << NLO) ^ thr_val) & thr_mask & ~(unsigned)(LOC - 1)) continue;
      const double* __restrict__ q = Q + (H << NLO);
      double wh = 0.0;
#pragma unroll
      for (int b = 0; b < LOC; ++b) {
        const double d = ((llo[b] + q[b]) + lh - best) * inv_kT;
        if (d < 40.0) {
          const double wgt = exp(-d);
          wh += wgt;
#pragma unroll
          for (int p = 0; p < NLO; ++p)
            if ((b >> p) & 1) acc[N - 1 - p] += wgt;
        }
      }
      Z += wh;
#pragma unroll
      for (int p = 0; p < NHI; ++p)
        if ((H >> p) & 1) acc[N - 1 - NLO - p] += wh;
    }
    const double invZ = 1.0 / Z;
#pragma unroll
    for (int j = 0; j < N; ++j) nd[j] = f[j] + acc[j] * invZ;
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j) nd[j] = f[j] + (double)((bidx >> (N - 1 - j)) & 1);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// brute_force ground state: the minimum over ALL n in {0..maxc}^N (dot 0 slowest, first minimum wins), found by exact
// branch and bound instead of visiting the (maxc+1)^N candidates (15 625 at N = 6, 390 625 at N = 8).
//   cdd_inv = U D U^T (U unit upper triangular, D > 0; factored once per env on the host), so with z = n - g
//       E(n) = sum_k d_k (z_k + sum_{j<k} U_jk z_j)^2 :
//   term k depends on dots 0..k only and every term is >= 0, hence the partial sum over the fixed leading dots is a LOWER
//   BOUND of every completion (Schnorr-Euchner enumeration).  A subtree is entered only if its partial sum is strictly
//   below the best energy found so far; the walk starts from the rounded, clipped potentials (+1e-9, so that candidate is
//   itself re-found in enumeration order and ties resolve to the first minimum, as in the exhaustive loop).
//   kT > 0: second walk over the candidates within 40 kT of the minimum (the exhaustive loop's own cut-off).
// ---------------------------------------------------------------------------------------------------------------
template <int N, int LVL>
struct BruteLevel {
  // PASS 0: argmin.  PASS 1: Boltzmann accumulation over candidates with E < cut = Emin + 40 kT.
  template <int PASS>
  static __device__ __forceinline__ void run(const double* __restrict__ ud, const double (&g)[N], int maxc, double p_prev,
                                             const double (&s)[N], unsigned code, double& best, unsigned& bcode,
                                             double emin, double inv_kT, double& Z, double (&acc)[N]) {
    const double dl = ud[LVL];
    const double ctr = g[LVL] - s[LVL];                     // continuous minimiser of this level's term
    // children in order of increasing distance from the centre (Schnorr-Euchner zig-zag): the first leaf reached is the
    // sequentially rounded point -- a strong incumbent -- and a level is left at its FIRST child that fails the bound,
    // since every later child is farther from the centre
    int up = (int)fmin(fmax(ceil(ctr), 0.0), (double)(maxc + 1));
    int dn = up - 1;
#pragma unroll 1
    while (dn >= 0 || up <= maxc) {
      const bool take_up = dn < 0 || (up <= maxc && ((double)up - ctr) < (ctr - (double)dn));
      const int v = take_up ? up : dn;
      if (take_up) ++up; else --dn;
      const double y = (double)v - ctr;
      const double p = fma(dl * y, y, p_prev);
      if (!(p < best)) break;                               // best: running minimum (PASS 0) / the 40 kT cut (PASS 1)
      const unsigned c2 = code * 16u + (unsigned)v;
      if constexpr (LVL == N - 1) {
        if constexpr (PASS == 0) {
          best = p;
          bcode = c2;
        } else {
          const double wgt = exp(-(p - emin) * inv_kT);
          Z += wgt;
#pragma unroll
          for (int j = 0; j < N; ++j) acc[j] += wgt * (double)((c2 >> (4 * (N - 1 - j))) & 15u);
        }
      } else {
        const double zl = (double)v - g[LVL];
        double s2[N];
#pragma unroll
        for (int k = 0; k < N; ++k) s2[k] = (k > LVL) ? fma(ud[8 + LVL * N + k], zl, s[k]) : 0.0;
        BruteLevel<N, LVL + 1>::template run<PASS>(ud, g, maxc, p, s2, c2, best, bcode, emin, inv_kT, Z, acc);
      }
    }
  }
};
template <int N>
struct BruteLevel<N, N> {
  template <int PASS>
  static __device__ __forceinline__ void run(const double*, const double (&)[N], int, double, const double (&)[N], unsigned,
                                             double&, unsigned&, double, double, double&, double (&)[N]) {}
};

// `ud`: d[8] | U[64] of cdd_inv with rows / columns permuted by `pm` (pm[l] = dot at tree level l, pm[8 + j] = level of dot
// j); `gp`: the potentials in that order.  The order is chosen per work item (most negative potential first): a dot far below
// its first transition is pinned to 0 carriers, and with it at the TOP of the tree its unavoidable cost sits in every
// partial sum and conditions the centres of the levels below -- the bound bites (likewise a dot far above max_charge_carriers,
// pinned to the upper face).  (With such dots at the bottom the
// unconstrained completion the bound assumes is far below anything the box allows, and the walk degenerates.)
// Exact energy ties (measure zero; the parity tests skip margins <= 1e-9) resolve in tree order.
template <int N, bool THERMAL>
__device__ __forceinline__ void ground_state_brute(const double (&gp)[N], const double* __restrict__ rec,
                                                   const qd_layout& L, const double* __restrict__ ud,
                                                   const int* __restrict__ pm, double kT, double (&nd)[N]) {
  const double (&g)[N] = gp;
  const int maxc = (int)rec[L.o_par + QD_PAR_MAXC];
  double Z = 0.0;
  double s[N], acc[N];
#pragma unroll
  for (int j = 0; j < N; ++j) { s[j] = 0.0; acc[j] = 0.0; }
  // starting incumbent: the potentials rounded and clipped to the box
  unsigned bcode = 0;
  double best = 0.0;
  {
    double sk[N];
#pragma unroll
    for (int k = 0; k < N; ++k) sk[k] = 0.0;
#pragma unroll
    for (int l = 0; l < N; ++l) {
      const double v = fmin(fmax(rint(g[l]), 0.0), (double)maxc);
      const double zl = v - g[l];
      const double y = zl + sk[l];
      best = fma(ud[l] * y, y, best);
      bcode = bcode * 16u + (unsigned)(int)v;
#pragma unroll
      for (int k = 0; k < N; ++k)
        if (k > l) sk[k] = fma(ud[8 + l * N + k], zl, sk[k]);
    }
    best += 1e-9;
  }
  BruteLevel<N, 0>::template run<0>(ud, g, maxc, 0.0, s, 0u, best, bcode, 0.0, 0.0, Z, acc);
  if (THERMAL && kT > 0.0) {
    double cut = best + 40.0 * kT;
    unsigned dummy = 0;
    BruteLevel<N, 0>::template run<1>(ud, g, maxc, 0.0, s, 0u, cut, dummy, best, 1.0 / kT, Z, acc);
    const double invZ = 1.0 / Z;
    double np_[N];
#pragma unroll
    for (int l = 0; l < N; ++l) np_[l] = acc[l] * invZ;
    // level l -> dot pm[l]
#pragma unroll
    for (int j = 0; j < N; ++j) {
      const int lv = pm[8 + j];
      double v = np_[0];
#pragma unroll
      for (int l = 1; l < N; ++l) v = (lv == l) ? np_[l] : v;
      nd[j] = v;
    }
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j) nd[j] = (double)((bcode >> (4 * (N - 1 - pm[8 + j]))) & 15u);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The scan kernel.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t compose2(uint32_t later, uint32_t earlier) {
  // functions {0,1}->{0,1} encoded as bit s = f(s); returns later o earlier
  return ((later >> (earlier & 1u)) & 1u) | (((later >> ((earlier >> 1) & 1u)) & 1u) << 1);
}

template <int N>
__device__ __forceinline__ uint64_t pack_key(const double (&nd)[N], bool integral) {
  uint64_t k = 0;
  if (integral) {                                  // hard argmin (kT == 0): the occupations are exact integers
#pragma unroll
    for (int j = 0; j < N; ++j) k |= (uint64_t)((unsigned)__double2int_rz(nd[j]) & 0xffu) << (8 * j);
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j) k |= (uint64_t)((unsigned)(int)floor(nd[j] + 0.5) & 0xffu) << (8 * j);
  }
  return k;
}

// ---------------------------------------------------------------------------------------------------------------
// Stages shared by the scan kernels (qd_scan_kernel, qd_scan_fast_kernel; the staging also by the tunnel kernels).
// ---------------------------------------------------------------------------------------------------------------

// Stage the head of the env record (`rec_bytes`) and the scan descriptor into the warp's slot: lane 0 issues two TMA bulk
// copies on one mbarrier, the warp waits and flips the phase.  use_one: the one descriptor of a single-scan call sits in
// the kernel parameters -- the lanes copy it and TMA brings the record alone.
__device__ __forceinline__ void stage_item(const KArgs& a, const qd_scan* gscan, uint32_t rec_bytes, double* rec, qd_scan* sc,
                                           uint64_t* bar, uint32_t& phase, int lane, bool use_one = false) {
  if (use_one) {
    if (lane == 0) {
      fence_proxy_async();
      mbar_expect_tx(bar, rec_bytes);
      tma_bulk_g2s(rec, a.records + (size_t)a.one.env_id * a.L.rec_doubles, rec_bytes, bar);
    }
    const double* src = reinterpret_cast<const double*>(&a.one);
    double* dst = reinterpret_cast<double*>(sc);
    for (int i = lane; i < (int)(sizeof(qd_scan) / 8); i += 32) dst[i] = src[i];
    __syncwarp();
  } else if (lane == 0) {
    const int env = gscan->env_id;
    fence_proxy_async();
    mbar_expect_tx(bar, rec_bytes + (uint32_t)sizeof(qd_scan));
    tma_bulk_g2s(rec, a.records + (size_t)env * a.L.rec_doubles, rec_bytes, bar);
    tma_bulk_g2s(sc, gscan, (uint32_t)sizeof(qd_scan), bar);
  }
  mbar_wait(bar, phase);
  phase ^= 1u;
}

// Rows [row0, row1) and columns [cx0, cx1) of item `part` of an nx x ny scan: a block of rows_per_item rows, split along x
// into col_parts ranges of whole 32-pixel chunks.
struct ItemWindow {
  int row0, row1, cx0, cx1;
  bool empty;
};
__device__ __forceinline__ ItemWindow item_window(const KArgs& a, int part, int nx, int ny) {
  const int cparts = a.col_parts > 1 ? a.col_parts : 1;
  const int rpart = part / cparts, cpart = part - rpart * cparts;
  ItemWindow w;
  w.row0 = rpart * a.rows_per_item;
  w.row1 = min(ny, w.row0 + a.rows_per_item);
  const int n_chunk_x = (nx + 31) >> 5;
  w.cx0 = ((n_chunk_x * cpart) / cparts) << 5;
  w.cx1 = min(nx, ((n_chunk_x * (cpart + 1)) / cparts) << 5);
  w.empty = w.row0 >= ny || w.cx0 >= w.cx1;
  return w;
}

// Per-item affine forms of the dot potentials (der[0..8) g0, [8..16) gx, [16..24) gy) and of the sensor potential
// (der[24..27) us0, usx, usy) on an affine scan window, one lane per row of cgd (lanes 0..N).
// Occupations are bounded by the largest dot potential of the window (+1 for the ceil candidate, +2 on the tunnel path;
// the relaxed occupations never exceed max(g, 0) on an M-matrix).  uint8 charge maps and the packed latching keys hold
// 0..255: windows that could leave that range are flagged instead of saturating silently.  check_overflow = false for
// brute force, whose occupations are bounded by max_charge_carriers instead.
template <int N>
__device__ __forceinline__ void item_affine_forms(const KArgs& a, const double* rec, const qd_scan* sc, double* der, int lane,
                                                  bool check_overflow = true) {
  const qd_layout& L = a.L;
  const int NV = L.n_volt;
  if (lane <= N) {
    const double* arow = (lane < N) ? rec + L.o_a + lane * NV : rec + L.o_sa;
    double s0 = 0.0, sx = 0.0, sy = 0.0;
    for (int k = 0; k < NV; ++k) {
      const double c = arow[k];
      s0 = fma(c, sc->v0[k], s0);
      sx = fma(c, sc->dx[k], sx);
      sy = fma(c, sc->dy[k], sy);
    }
    if (lane < N) {
      der[lane] = s0; der[8 + lane] = sx; der[16 + lane] = sy;
      const double gmax = s0 + fmax(sx * (double)(sc->nx - 1), 0.0) + fmax(sy * (double)(sc->ny - 1), 0.0);
      const bool replaced = (a.flags & QD_FLAG_RADIAL) && sc->rad_mode == 2;      // no occupations are computed there
      if (check_overflow && !replaced && !(gmax < 252.0) && a.status)
        *reinterpret_cast<volatile unsigned*>(a.status) = QD_STATUS_OCC_OVERFLOW;
    } else { der[24] = s0; der[25] = sx; der[26] = sy; }
  }
}

// The random draws of a pixel: one Philox4x32-10 block (purpose 0, counter = pixel index) -> Box-Muller pair (white,
// radial), latching uniform, telegraph uniform.  All zero when nothing random is on.
struct PixelDraws {
  float z_white, z_rad, u_latch, u_tele;
};
__device__ __forceinline__ PixelDraws pixel_draws(bool need_rng, uint64_t seed, long long pix) {
  PixelDraws d = {0.f, 0.f, 0.f, 0.f};
  if (need_rng) {
    const Philox4 w = philox4x32_10(seed, (uint64_t)pix, 0u);
    box_muller(w.w0, w.w1, d.z_white, d.z_rad);
    d.u_latch = u24(w.w2);
    d.u_tele = u24(w.w3);
  }
  return d;
}

// Hysteresis latching of one 32-pixel chunk along x, on packed keys (8 bits per dot), from the held configuration
// `held_key`; `todo` = the lanes still to resolve.  Loops over events only: the first lane whose key differs from the
// held one, the differing dots classified by a byte-nonzero mask, p_leads / p_inter looked up.  The lanes from there on
// that want the same new configuration form a run; every one of them faces the same (held -> new) transition, so the
// first of them whose uniform is below p accepts and the ones before it stay latched to the held configuration.
// take_held(i, rejected, acc) runs on every lane once per event, while held_key is still the configuration held so far
// (i: first differing lane, rejected: lanes that keep the held configuration, acc: accepting lane, 32 if none): it moves
// whatever else travels with the configuration.
template <typename TakeHeld>
__device__ __forceinline__ void latch_chunk(uint64_t& key, uint64_t& held_key, unsigned todo, float u_latch, const double* rec,
                                            const qd_layout& L, int lane, TakeHeld&& take_held) {
  while (true) {
    const unsigned diff = __ballot_sync(0xffffffffu, key != held_key) & todo;
    if (!diff) break;
    const int i = __ffs(diff) - 1;
    const uint64_t ck = shfl_u64(key, i);
    const uint64_t x = ck ^ held_key;
    const uint64_t nz = (((x & 0x7f7f7f7f7f7f7f7fULL) + 0x7f7f7f7f7f7f7f7fULL) | x) & 0x8080808080808080ULL;
    const int ndiff = __popcll(nz);
    double p_acc = 2.0;                            // > every uniform: accept
    if (ndiff == 1) {
      p_acc = rec[L.o_pleads + ((__ffsll((long long)nz) - 1) >> 3)];
    } else if (ndiff == 2) {
      const int d0 = (__ffsll((long long)nz) - 1) >> 3;
      const int d1 = (63 - __clzll((long long)nz)) >> 3;
      p_acc = rec[L.o_pinter + d0 * 8 + d1];
    }
    const unsigned from_i = ~((1u << i) - 1u);
    const unsigned same = __ballot_sync(0xffffffffu, key == ck) & todo & from_i;
    const unsigned brk = ~same & from_i & todo;
    const unsigned run = same & ~(brk ? (~0u << (__ffs(brk) - 1)) : 0u);
    const unsigned acc = __ballot_sync(0xffffffffu, (double)u_latch < p_acc) & run;
    const int acl = acc ? __ffs(acc) - 1 : 32;
    const unsigned rejected = run & ((acl >= 32) ? ~0u : ((1u << acl) - 1u));
    if ((rejected >> lane) & 1u) key = held_key;
    take_held(i, rejected, acl);
    if (acl < 32) held_key = ck;
    const int done_to = (acl < 32) ? acl : (31 - __clz(run));
    todo &= ~((2u << done_to) - 1u);
  }
}

// Telegraph state at the start of row iy: the stationary draw (Philox purpose 1), or state 0 on a flat pass, where the
// chain runs on from row to row.
__device__ __forceinline__ uint32_t tele_start(bool f_carry, uint64_t seed, int iy, const double* par) {
  if (f_carry) return 0u;
  const Philox4 wr = philox4x32_10(seed, (uint64_t)iy, 1u);
  return ((double)u24(wr.w0) < par[QD_PAR_TELE_STAT]) ? 1u : 0u;
}

// Sensor: ten fp32 Lorentzians of the first differences of the free energy, x_k = x0 + k xs for k = -5..4.
__device__ __forceinline__ float sensor_lorentz10(double x0, double xs) {
  float zs = 0.f;
#pragma unroll
  for (int k = -5; k < 5; ++k) {
    const float xk = (float)fma((double)k, xs, x0);
    zs += rcp_approx(fmaf(xk, xk, 1.0f));
  }
  return zs;
}

// Amplitude of the radial noise at pixel (fx, fy) (rad_mode 1): rad_alpha * (|v| - rad_zero_radius) clamped to
// [0, rad_max_amp], v = the pixel's voltage offset rad_x0 + fx rad_dx, rad_y0 + fy rad_dy.
__device__ __forceinline__ float radial_amp(const qd_scan* sc, double fx, double fy) {
  const float vx = (float)fma(fx, sc->rad_dx, sc->rad_x0);
  const float vy = (float)fma(fy, sc->rad_dy, sc->rad_y0);
  const float dist = sqrtf(fmaf(vx, vx, vy * vy));
  return fminf(fmaxf((float)sc->rad_alpha * (dist - (float)sc->rad_zero_radius), 0.0f), (float)sc->rad_max_amp);
}

// THERMAL = false instantiations carry no Boltzmann-average code at all (the hard-argmin kernels are the hot ones; the
// launch picks THERMAL = true only when QD_FLAG_THERMAL is set).
// POINTS = true: explicit voltage list (a.points) instead of the affine descriptor -- the single-device entry points.
template <int N, int ALG, bool THERMAL, bool POINTS>
__global__ void __launch_bounds__(QD_CTA_WARPS * 32, QD_MIN_BLOCKS) qd_scan_kernel(const KArgs a) {
  extern __shared__ __align__(128) unsigned char qd_smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const qd_layout& L = a.L;
  const int NV = L.n_volt;

  unsigned char* slot = qd_smem + (size_t)warp * a.slot_bytes;
  double* rec = reinterpret_cast<double*>(slot);
  qd_scan* sc = reinterpret_cast<qd_scan*>(slot + (size_t)L.rec_doubles * 8);
  double* der = reinterpret_cast<double*>(slot + (size_t)L.rec_doubles * 8 + sizeof(qd_scan));
  uint64_t* bar = reinterpret_cast<uint64_t*>(der + QD_DER_DOUBLES);
  double* d_g0 = der;
  double* d_gx = der + 8;
  double* d_gy = der + 16;
  double* d_us = der + 24;      // us0, usx, usy
  double* d_carry = der + 32;   // latched configuration of the last pixel of the previous chunk
  ProjCache pc;
  double* bf_ud = reinterpret_cast<double*>(bar + 2);            // brute force: per-item factor of the permuted cdd_inv
  int* bf_pm = reinterpret_cast<int*>(bf_ud + 72);
  pc.mats = reinterpret_cast<double*>(bar + 2);
  pc.aug = pc.mats + 8 * 64;
  pc.keys = reinterpret_cast<uint32_t*>(pc.aug + 8 * 16);
  pc.meta = pc.keys + QD_PC_WAYS;
  pc.lin_s = pc.aug + 8 * 16 + 8;
  pc.aff = pc.lin_s + 8 * 32;
  pc.gsrc = POINTS ? nullptr : der;
  pc.mat_stride = 64;

  if (lane == 0) mbar_init(bar, 1);
  __syncwarp();
  uint32_t phase = 0;

  const bool f_latch = a.flags & QD_FLAG_LATCH;
  const bool f_noise = a.flags & QD_FLAG_NOISE;
  const bool f_radial = a.flags & QD_FLAG_RADIAL;
  const bool f_thermal = a.flags & QD_FLAG_THERMAL;
  const bool f_carry = a.flags & QD_FLAG_CARRY_ROWS;
  const bool f_white_out = a.flags & QD_FLAG_WHITE_ON_OUTPUT;
  const bool f_pink = a.flags & QD_FLAG_PINK;
  double* d_pink = der + 40;    // state of the four 1/f chains at the last pixel processed (warp-uniform, in shared memory)
  const uint32_t rec_bytes = (uint32_t)L.rec_doubles * 8u;

  const long long total_items = (long long)a.n_scan * a.items_per_scan;
  for (long long item = (long long)blockIdx.x * warps_per_cta + warp; item < total_items;
       item += (long long)gridDim.x * warps_per_cta) {
    const int scan_id = (int)(item / a.items_per_scan);
    const int part = (int)(item - (long long)scan_id * a.items_per_scan);
    const qd_scan* gscan = a.scans + scan_id;

    stage_item(a, gscan, rec_bytes, rec, sc, bar, phase, lane, a.use_one);
    if constexpr (ALG == QD_ALG_DEFAULT) {
      if (lane == 0) { pc.meta[0] = 0u; pc.meta[1] = 0u; }    // the projection cache belongs to one env
    }

    const int nx = sc->nx, ny = sc->ny;
    const ItemWindow w = item_window(a, part, nx, ny);
    if (w.empty) { __syncwarp(); continue; }
    const int row0 = w.row0, row1 = w.row1, cx0 = w.cx0, cx1 = w.cx1;

    if constexpr (!POINTS) item_affine_forms<N>(a, rec, sc, der, lane, ALG != QD_ALG_BRUTE_FORCE);
    __syncwarp();
    if constexpr (ALG == QD_ALG_BRUTE_FORCE) {
      // ---- tree order of this item (most negative potential at the item's centre first) and cdd_inv = U D U^T in it ----
      if (lane == 0) {
        int ord[N];
        double gc[N];
        const double maxc_d = rec[L.o_par + QD_PAR_MAXC];
        for (int j = 0; j < N; ++j) {
          ord[j] = j;
          // sort key: how far INSIDE the box [0, maxc] the potential at the item's centre lies (negative: outside, pinned to
          // a face -- those dots go to the top of the tree, the most firmly pinned first)
          const double gcj = POINTS ? 0.0 : fma(0.5 * (double)(row0 + row1 - 1), d_gy[j], fma(0.5 * (double)(nx - 1), d_gx[j], d_g0[j]));
          gc[j] = fmin(gcj, maxc_d - gcj);
        }
        if (!POINTS) {
          for (int i = 1; i < N; ++i) {                    // insertion sort by potential, ascending
            const int o = ord[i];
            int j = i - 1;
            while (j >= 0 && gc[ord[j]] > gc[o]) { ord[j + 1] = ord[j]; --j; }
            ord[j + 1] = o;
          }
        }
        for (int l = 0; l < N; ++l) { bf_pm[l] = ord[l]; bf_pm[8 + ord[l]] = l; }
        const double* __restrict__ Cm = rec + L.o_cinv;
        double* d = bf_ud;
        double* U = bf_ud + 8;
        for (int k = N - 1; k >= 0; --k) {
          double dk = Cm[ord[k] * N + ord[k]];
          for (int j = k + 1; j < N; ++j) dk -= U[k * N + j] * U[k * N + j] * d[j];
          d[k] = dk;
          U[k * N + k] = 1.0;
          const double idk = 1.0 / dk;
          for (int i = 0; i < k; ++i) {
            double u = Cm[ord[i] * N + ord[k]];
            for (int j = k + 1; j < N; ++j) u -= U[i * N + j] * U[k * N + j] * d[j];
            U[i * N + k] = u * idk;
          }
        }
      }
      __syncwarp();
    }

    const double* par = rec + L.o_par;
    const double kT = (THERMAL && f_thermal) ? par[QD_PAR_KT] : 0.0;
    const bool latch_on = f_latch && par[QD_PAR_LATCH] != 0.0;
    const bool replace = f_radial && sc->rad_mode == 2;
    const uint64_t seed = sc->seed;
    const long long pix0 = sc->pix_offset;
    const double inv_gamma = 1.0 / sc->peak_width;
    const double css = rec[L.o_css];
    const bool need_rng = f_noise || latch_on || (f_radial && sc->rad_mode != 0);

    uint64_t held_key = 0;
    bool have_held = false;
    uint32_t tele_state = 0;
    bool tele_init = false;
    bool pink_init = false;

    for (int iy = row0; iy < row1; ++iy) {
      if (!f_carry) { have_held = false; tele_init = false; pink_init = false; }
      for (int c0 = cx0; c0 < cx1; c0 += 32) {
        const int ix = c0 + lane;
        const bool valid = ix < nx;
        const int ixc = valid ? ix : nx - 1;
        const long long pix = (long long)iy * nx + ixc;
        const unsigned vmask = __ballot_sync(0xffffffffu, valid);
        const PixelDraws rnd = pixel_draws(need_rng, seed, pix);

        double nd[N];
        double g[N];
        double us;
        float zf;
        if (!replace) {
          // ---- dot potentials g = cgd . v ----
          if constexpr (!POINTS) {
            const double fx = (double)ixc, fy = (double)iy;
#pragma unroll
            for (int j = 0; j < N; ++j) g[j] = fma(fy, d_gy[j], fma(fx, d_gx[j], d_g0[j]));
            us = fma(fy, d_us[2], fma(fx, d_us[1], d_us[0]));
          } else {
            const double* __restrict__ v = a.points + (size_t)pix * NV;
#pragma unroll
            for (int j = 0; j < N; ++j) g[j] = 0.0;
            us = 0.0;
            for (int k = 0; k < NV; ++k) {
              const double vk = v[k];
#pragma unroll
              for (int j = 0; j < N; ++j) g[j] = fma(rec[L.o_a + j * NV + k], vk, g[j]);
              us = fma(rec[L.o_sa + k], vk, us);
            }
            if constexpr (ALG != QD_ALG_BRUTE_FORCE) {
              bool big = false;
#pragma unroll
              for (int j = 0; j < N; ++j) big |= !(g[j] < 252.0);
              if (big && a.status) *reinterpret_cast<volatile unsigned*>(a.status) = QD_STATUS_OCC_OVERFLOW;
            }
          }

          // ---- ground state ----
          if constexpr (ALG == QD_ALG_TUNNEL) {
            // the tunnel-coupled ground state was computed by qd_tunnel_gs_kernel (one warp per pixel)
            const double* __restrict__ src = a.nbar + (size_t)(pix0 + pix) * N;
#pragma unroll
            for (int j = 0; j < N; ++j) nd[j] = src[j];
          } else if constexpr (ALG == QD_ALG_BRUTE_FORCE) {
            double gp[N];                            // potentials in tree order
            if constexpr (!POINTS) {
              const double fx = (double)ixc, fy = (double)iy;
#pragma unroll
              for (int l = 0; l < N; ++l) { const int j = bf_pm[l]; gp[l] = fma(fy, d_gy[j], fma(fx, d_gx[j], d_g0[j])); }
            } else {
#pragma unroll
              for (int l = 0; l < N; ++l) gp[l] = g[l];           // explicit voltage lists keep the identity order
            }
            ground_state_brute<N, THERMAL>(gp, rec, L, bf_ud, bf_pm, kT, nd);
          }
          else ground_state_box<N, THERMAL, !POINTS>(g, rec, L, pc, lane, L.algorithm == QD_ALG_THRESHOLDED, kT, (double)ixc, (double)iy, nd);

          // ---- hysteresis latching along x ----
          if (latch_on) {
            // integral: hard argmin, the occupations ARE the key bytes -- the event loop then works on keys alone
            // and the occupations of the latched pixels are unpacked once at the end
            const bool integral = ALG != QD_ALG_TUNNEL && kT <= 0.0;
            uint64_t key = pack_key<N>(nd, integral);
            const uint64_t key_free = key;
            unsigned todo = vmask;
            if (!have_held) {                       // first pixel of the row (or of the scan): accepted as is
              held_key = shfl_u64(key, 0);
              todo &= ~1u;
              have_held = true;
            }
            // a rejected pixel takes the occupations of lane i - 1 (the held configuration), or the carry of the last chunk
            latch_chunk(key, held_key, todo, rnd.u_latch, rec, L, lane, [&](int i, unsigned rejected, int) {
              if (rejected && !integral) {
                const int src = (i > 0) ? i - 1 : 0;
#pragma unroll
                for (int j = 0; j < N; ++j) {
                  const double prev = shfl_f64(nd[j], src);
                  const double held = (i > 0) ? prev : d_carry[j];
                  if ((rejected >> lane) & 1u) nd[j] = held;
                }
              }
            });
            if (integral) {
              if (key != key_free) {
#pragma unroll
                for (int j = 0; j < N; ++j) nd[j] = (double)(int)((unsigned)(key >> (8 * j)) & 0xffu);
              }
            } else {
              // configuration after the last valid pixel -> carry for the next chunk
              const int last = 31 - __clz(vmask);
              if (lane == last) {
#pragma unroll
                for (int j = 0; j < N; ++j) d_carry[j] = nd[j];
              }
              __syncwarp();
            }
          }

          // ---- sensor input noise: white + telegraph ----
          double noise_in = 0.0, noise_out = 0.0;
          if (f_noise) {
            const double wn = par[QD_PAR_WHITE] * (double)rnd.z_white;
            if (f_white_out) noise_out = wn; else noise_in = wn;
            const double tamp = par[QD_PAR_TELE_AMP];
            if (tamp != 0.0) {
              if (!tele_init) {
                tele_state = tele_start(f_carry, seed, iy, par);
                tele_init = true;
              }
              const uint32_t flip0 = ((double)rnd.u_tele < par[QD_PAR_P01]) ? 1u : 0u;
              const uint32_t flip1 = ((double)rnd.u_tele < par[QD_PAR_P10]) ? 1u : 0u;
              uint32_t fn = valid ? ((0u ^ flip0) | ((1u ^ flip1) << 1)) : 2u;   // invalid lanes: identity
#pragma unroll
              for (int d = 1; d < 32; d <<= 1) {
                const uint32_t other = __shfl_up_sync(0xffffffffu, fn, d);
                if (lane >= d) fn = compose2(fn, other);
              }
              const uint32_t st = (fn >> tele_state) & 1u;
              tele_state = __shfl_sync(0xffffffffu, st, 31);
              noise_in += tamp * (double)st;
            }
          }
          // ---- 1/f input noise: four Ornstein-Uhlenbeck chains x_k[i] = a_k x_k[i-1] + sqrt(1 - a_k^2) xi_k[i] along x,
          // a_k = exp(-1 / tau_k), tau_k = 2, 8, 32, 128 pixels, unit stationary variance each; the term is
          // pink_amp * (x_0 + x_1 + x_2 + x_3) / 2.  Draws: Philox purpose 2 (per pixel), 3 (stationary start of a row / of
          // a flat pass).  A chain is a prefix scan of affine maps with a constant slope: five shuffle steps per chain.
          if (f_pink && par[QD_PAR_PINK] != 0.0) {
            if (!pink_init) {
              const Philox4 ws = philox4x32_10(seed, (uint64_t)iy, 3u);
              float s0, s1, s2, s3;
              box_muller(ws.w0, ws.w1, s0, s1);
              box_muller(ws.w2, ws.w3, s2, s3);
              __syncwarp();
              if (lane == 0) { d_pink[0] = (double)s0; d_pink[1] = (double)s1; d_pink[2] = (double)s2; d_pink[3] = (double)s3; }
              __syncwarp();
              pink_init = true;
            }
            const Philox4 wp = philox4x32_10(seed, (uint64_t)pix, 2u);
            float e4[4];
            box_muller(wp.w0, wp.w1, e4[0], e4[1]);
            box_muller(wp.w2, wp.w3, e4[2], e4[3]);
            const int last = 31 - __clz(vmask);
            double psum = 0.0;
            double xs_new[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const double ak = (k == 0) ? 0.60653065971263342 : (k == 1) ? 0.88249690258459546
                              : (k == 2) ? 0.96923323447634413 : 0.99221793826024351;      // exp(-1/2), exp(-1/8), exp(-1/32), exp(-1/128)
              double Bk = sqrt(1.0 - ak * ak) * (double)e4[k];
              double ad = ak, apow = 1.0;
#pragma unroll
              for (int d = 1; d < 32; d <<= 1) {
                const double tb = __hiloint2double(__shfl_up_sync(0xffffffffu, __double2hiint(Bk), d),
                                                   __shfl_up_sync(0xffffffffu, __double2loint(Bk), d));
                if (lane >= d) Bk = fma(ad, tb, Bk);
                if ((lane + 1) & d) apow *= ad;
                ad *= ad;
              }
              if ((lane + 1) & 32) apow *= ad;
              const double xk = fma(apow, d_pink[k], Bk);
              xs_new[k] = shfl_f64(xk, last);
              psum += xk;
            }
            __syncwarp();
            if (lane == 0) {
#pragma unroll
              for (int k = 0; k < 4; ++k) d_pink[k] = xs_new[k];
            }
            __syncwarp();
            noise_in += par[QD_PAR_PINK] * 0.5 * psum;
          }

          // ---- sensor: ten Lorentzians of the first differences of the full-system free energy ----
          double base = 0.0;
#pragma unroll
          for (int j = 0; j < N; ++j) base = fma(rec[L.o_sw + j], nd[j] - g[j], base);
          base *= 2.0;
          const double t = (rint(us) + noise_in) - us;
          // dPhi_k = css (2 (t + k) + 1) + base is affine in k: x_k = dPhi_k / gamma = x0 + k * xs
          const double xs = 2.0 * css * inv_gamma;
          const double x0 = fma(css, fma(2.0, t, 1.0), base) * inv_gamma;
          double z;
          if constexpr (ALG == QD_ALG_TUNNEL) {
            // tunnel path: fp64 Lorentzians.  <n> carries the eigen-solver's own error (1e-6 budget), so the sensor adds
            // none of its own; the cost is nothing next to the per-pixel eigen-solve.
            double zs = 0.0;
#pragma unroll
            for (int k = -5; k < 5; ++k) {
              const double xk = fma((double)k, xs, x0);
              zs += 1.0 / fma(xk, xk, 1.0);
            }
            z = zs + noise_out;
          } else {
            z = (double)sensor_lorentz10(x0, xs) + noise_out;
          }
          if (f_radial && sc->rad_mode == 1) z = fma((double)rnd.z_rad, (double)radial_amp(sc, (double)ixc, (double)iy), z);
          zf = (float)z;
        } else {
          zf = rnd.z_rad;
#pragma unroll
          for (int j = 0; j < N; ++j) nd[j] = 0.0;
        }

        // ---- coalesced stores ----
        if (valid) {
          const long long o = pix0 + (long long)iy * nx + ix;
          if (a.z_out) a.z_out[o] = zf;
          if (a.n_type == QD_N_U8) {
            unsigned char* p = reinterpret_cast<unsigned char*>(a.n_out) + o * N;
            if constexpr (N == 8) {
              uint64_t k = 0;
#pragma unroll
              for (int j = 0; j < N; ++j) k |= (uint64_t)(unsigned char)min(255, (int)nd[j]) << (8 * j);
              *reinterpret_cast<uint64_t*>(p) = k;
            } else if constexpr (N == 4) {
              uint32_t k = 0;
#pragma unroll
              for (int j = 0; j < N; ++j) k |= (uint32_t)(unsigned char)min(255, (int)nd[j]) << (8 * j);
              *reinterpret_cast<uint32_t*>(p) = k;
            } else if constexpr (N == 2) {
              const uint16_t k = (uint16_t)((unsigned char)min(255, (int)nd[0]) | ((unsigned char)min(255, (int)nd[1]) << 8));
              *reinterpret_cast<uint16_t*>(p) = k;
            } else {
#pragma unroll
              for (int j = 0; j < N; ++j) p[j] = (unsigned char)min(255, (int)nd[j]);
            }
          } else if (a.n_type == QD_N_F32) {
            float* p = reinterpret_cast<float*>(a.n_out) + o * N;
#pragma unroll
            for (int j = 0; j < N; ++j) p[j] = (float)nd[j];
          } else if (a.n_type == QD_N_F64) {
            double* p = reinterpret_cast<double*>(a.n_out) + o * N;
#pragma unroll
            for (int j = 0; j < N; ++j) p[j] = nd[j];
          }
        }
      }
    }
    __syncwarp();
  }
}


// ---------------------------------------------------------------------------------------------------------------
// The HOT instantiation: default / thresholded search, hard argmin (kT = 0), affine scan windows -- config 4's kernel.
// Same arithmetic as qd_scan_kernel<N, QD_ALG_DEFAULT, false, false> (the parity tests run both; the stages above are
// shared), restructured so that a pixel never holds its occupations as doubles:
//   * floor(n_c) is packed straight into the 8-bit-per-dot key the latching pass works on; the argmin adds its bits with
//     one multiply (bit N-1-j -> byte j), and for N = 8 the uint8 charge map IS that key, stored with one STG.64;
//   * the sensor's dot term sum_j w_j (n_j - g_j) splits into SN = sum_j w_j n_j, which travels with the key through the
//     latching pass (a rejected pixel takes the held configuration's SN), and sum_j w_j g_j, affine in the pixel indices
//     (three coefficients per item);
//   * the Gray-code walk serves every width (2^kmax steps), so there is no block enumeration and no 16-entry register table;
//   * the telegraph chain is resolved on two ballots (lanes that would flip 0->1 / 1->0) by a warp-uniform loop over the
//     actual toggles (usually none) instead of a 5-step shuffle scan;
//   * the projection cache keeps only the affine forms P_S g0, P_S gx, P_S gy (one scratch matrix while building).
// Fewer live registers (128, four CTAs per SM instead of three) and a shared-memory slot of 10.6 KB per warp.
// ---------------------------------------------------------------------------------------------------------------
#ifndef QD_FAST_MIN_BLOCKS
#define QD_FAST_MIN_BLOCKS 4
#endif
constexpr int QD_FAST_DER = 32;     // g0[8] gx[8] gy[8] us[3] sg[3] pad[2]
constexpr int QD_FAST_PC = 64 + 8 * 16 + 8 + 8 * 32 + QD_PC_WAYS * 24;   // scratch P, inversion scratch, keys/meta, lin, affine forms

__host__ __device__ inline int qd_fast_slot_bytes(const qd_layout& L) {
  const int b = L.rec_doubles * 8 + (int)sizeof(qd_scan) + (QD_FAST_DER + 32 + QD_FAST_PC) * 8 + 16;
  return (b + 127) & ~127;
}

template <int N>
__global__ void __launch_bounds__(QD_CTA_WARPS * 32, QD_FAST_MIN_BLOCKS) qd_scan_fast_kernel(const KArgs a) {
  extern __shared__ __align__(128) unsigned char qd_smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const qd_layout& L = a.L;

  unsigned char* slot = qd_smem + (size_t)warp * a.slot_bytes;
  double* rec = reinterpret_cast<double*>(slot);
  qd_scan* sc = reinterpret_cast<qd_scan*>(slot + (size_t)L.rec_doubles * 8);
  double* der = reinterpret_cast<double*>(slot + (size_t)L.rec_doubles * 8 + sizeof(qd_scan));
  double* d_g0 = der;
  double* d_gx = der + 8;
  double* d_gy = der + 16;
  double* d_us = der + 24;      // us0, usx, usy
  double* d_sg = der + 27;      // sum_j w_j g_j: sg0, sgx, sgy
  double* swt = der + QD_FAST_DER;     // [0..15]: sum of w over the set LOW bits (dots N-1 .. N-4); [16..31]: HIGH bits
  ProjCache pc;
  pc.mats = swt + 32;
  pc.aug = pc.mats + 64;
  pc.keys = reinterpret_cast<uint32_t*>(pc.aug + 8 * 16);
  pc.meta = pc.keys + QD_PC_WAYS;
  pc.lin_s = pc.aug + 8 * 16 + 8;
  pc.aff = pc.lin_s + 8 * 32;
  pc.gsrc = der;
  pc.mat_stride = 0;
  uint64_t* bar = reinterpret_cast<uint64_t*>(pc.aff + QD_PC_WAYS * 24);

  if (lane == 0) mbar_init(bar, 1);
  __syncwarp();
  uint32_t phase = 0;

  const bool f_latch = a.flags & QD_FLAG_LATCH;
  const bool f_noise = a.flags & QD_FLAG_NOISE;
  const bool f_radial = a.flags & QD_FLAG_RADIAL;
  const bool f_carry = a.flags & QD_FLAG_CARRY_ROWS;
  const bool f_white_out = a.flags & QD_FLAG_WHITE_ON_OUTPUT;
  const bool thresholded = L.algorithm == QD_ALG_THRESHOLDED;
  const uint32_t rec_bytes = (uint32_t)L.rec_doubles * 8u;
  const double* __restrict__ cinv = rec + L.o_cinv;
  const double* __restrict__ Q = rec + L.o_q;
  const double* __restrict__ spos = rec + L.o_spos;
  const double* __restrict__ sneg = rec + L.o_sneg;
  const double* __restrict__ sw = rec + L.o_sw;
  const double* par = rec + L.o_par;

  const long long total_items = (long long)a.n_scan * a.items_per_scan;
  for (long long item = (long long)blockIdx.x * warps_per_cta + warp; item < total_items;
       item += (long long)gridDim.x * warps_per_cta) {
    const int scan_id = (int)(item / a.items_per_scan);
    const int part = (int)(item - (long long)scan_id * a.items_per_scan);
    const qd_scan* gscan = a.scans + scan_id;

    stage_item(a, gscan, rec_bytes, rec, sc, bar, phase, lane, a.use_one);
    if (lane == 0) { pc.meta[0] = 0u; pc.meta[1] = 0u; }      // the projection cache belongs to one (env, window)

    const int nx = sc->nx, ny = sc->ny;
    const ItemWindow w = item_window(a, part, nx, ny);
    if (w.empty) { __syncwarp(); continue; }
    const int row0 = w.row0, row1 = w.row1, cx0 = w.cx0, cx1 = w.cx1;

    // ---- per-item affine forms: dot potentials, sensor potential, sum_j w_j g_j; the two nibble tables of w ----
    item_affine_forms<N>(a, rec, sc, der, lane);
    {
      double t = 0.0;
      const int h = lane & 15;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int p = (lane < 16) ? q : q + 4;               // bit position inside the candidate index
        if (p < N && ((h >> q) & 1)) t += sw[N - 1 - p];
      }
      swt[lane] = t;
    }
    __syncwarp();
    if (lane < 3) {
      double t = 0.0;
      for (int j = 0; j < N; ++j) t = fma(sw[j], der[8 * lane + j], t);
      d_sg[lane] = t;
    }
    __syncwarp();

    const bool latch_on = f_latch && par[QD_PAR_LATCH] != 0.0;
    const bool replace = f_radial && sc->rad_mode == 2;
    const uint64_t seed = sc->seed;
    const long long pix0 = sc->pix_offset;
    const double inv_gamma = 1.0 / sc->peak_width;
    const double css = rec[L.o_css];
    const bool need_rng = f_noise || latch_on || (f_radial && sc->rad_mode != 0);

    uint64_t held_key = 0;
    double held_sn = 0.0;
    bool have_held = false;
    uint32_t tele_state = 0;
    bool tele_init = false;

    for (int iy = row0; iy < row1; ++iy) {
      if (!f_carry) { have_held = false; tele_init = false; }
      for (int c0 = cx0; c0 < cx1; c0 += 32) {
        const int ix = c0 + lane;
        const bool valid = ix < nx;
        const int ixc = valid ? ix : nx - 1;
        const long long pix = (long long)iy * nx + ixc;
        const unsigned vmask = __ballot_sync(0xffffffffu, valid);
        const double fx = (double)ixc, fy = (double)iy;
        const PixelDraws rnd = pixel_draws(need_rng, seed, pix);

        uint64_t key = 0;
        float zf;
        if (!replace) {
          double sn;          // sum_j w_j n_j of the configuration this pixel ends up with
          {
            // ---- dot potentials, relaxation, floor ----
            double g[N], nc[N];
            int sgn = 0;
#pragma unroll
            for (int j = 0; j < N; ++j) {
              g[j] = fma(fy, d_gy[j], fma(fx, d_gx[j], d_g0[j]));
              nc[j] = g[j];
              sgn |= __double2hiint(g[j]);
            }
            if (__any_sync(0xffffffffu, sgn < 0)) relax_lcp<N, true>(g, rec + L.o_cdd, pc, lane, fx, fy, nc);
            double r[N], lin[N];
            unsigned fixmask = 0, fixval = 0;
            uint32_t klo = 0, khi = 0;
            sn = 0.0;
#pragma unroll
            for (int j = 0; j < N; ++j) {
              const double fj = floor(nc[j]);
              r[j] = fj - g[j];
              sn = fma(sw[j], fj, sn);
              const uint32_t fi = (uint32_t)__double2int_rz(fj) & 0xffu;
              if (j < 4) klo |= fi << (8 * j); else khi |= fi << (8 * (j - 4));
              if (thresholded) {
                const double frac = nc[j] - fj;
                if (!(fabs(frac - 0.5) < 0.5 * par[QD_PAR_THRESHOLD])) {
                  fixmask |= 1u << (N - 1 - j);
                  if (floor(nc[j] + 0.5) - fj == 1.0) fixval |= 1u << (N - 1 - j);
                }
              }
            }
            key = ((uint64_t)khi << 32) | klo;
            matvec_smem<N>(cinv, r, lin);
            // ---- exact dominance (see ground_state_box) + the linear coefficients by BIT position to shared memory ----
            double* __restrict__ ls = pc.lin_s + lane;
            unsigned zmask = 0, omask = 0;
#pragma unroll
            for (int j = 0; j < N; ++j) {
              const unsigned bit = 1u << (N - 1 - j);
              const double l2 = lin[j] + lin[j];
              ls[(N - 1 - j) * 32] = l2;
              const double aj = l2 + cinv[j * N + j];
              zmask |= (aj + sneg[j] > 1e-9) ? bit : 0u;
              omask |= (aj + spos[j] < -1e-9) ? bit : 0u;
            }
            const unsigned add = (zmask | omask) & ~fixmask;       // thresholded bits keep their own value
            fixval |= omask & add;
            fixmask |= add;
            // ---- Gray-code walk over the undecided dots ----
            const unsigned freeb = ~fixmask & ((1u << N) - 1u);
            const int kfree = __popc(freeb);
            const int kmax = __reduce_max_sync(0xffffffffu, kfree);
            unsigned idx = fixval;
            double Lsum = 0.0;
#pragma unroll
            for (int p = 0; p < N; ++p)
              if ((fixval >> p) & 1u) Lsum += ls[p * 32];
            double best = Lsum + Q[idx];
            unsigned bidx = idx;
            if (kmax > 0) {
              // nibble list of the free bit positions, lowest first
              unsigned pos = 0;
              {
                int nfree = 0;
#pragma unroll
                for (int p = 0; p < N; ++p)
                  if ((freeb >> p) & 1u) { pos |= (unsigned)p << (4 * nfree); ++nfree; }
              }
              const unsigned steps = 1u << kmax, mine = 1u << kfree;
#pragma unroll 1
              for (unsigned c = 1; c < steps; ++c) {
                if (c < mine) {
                  const unsigned p = (pos >> (4 * (__ffs(c) - 1))) & 15u;
                  idx ^= 1u << p;
                  const double lp = ls[p * 32];
                  Lsum += ((idx >> p) & 1u) ? lp : -lp;
                  const double e = Lsum + Q[idx];
                  if (e < best || (e == best && idx < bidx)) { best = e; bidx = idx; }
                }
              }
            }
            // bit (N-1-j) of the winner -> byte j of the key
            key += ((((uint64_t)(bidx << (8 - N))) * 0x8040201008040201ULL) & 0x8080808080808080ULL) >> 7;
            sn += swt[bidx & 15u] + swt[16 + (bidx >> 4)];
          }

          // ---- hysteresis latching along x, on keys; SN travels with the configuration ----
          if (latch_on) {
            unsigned todo = vmask;
            if (!have_held) {                       // first pixel of the row (or of the scan): accepted as is
              held_key = shfl_u64(key, 0);
              held_sn = shfl_f64(sn, 0);
              todo &= ~1u;
              have_held = true;
            }
            latch_chunk(key, held_key, todo, rnd.u_latch, rec, L, lane, [&](int, unsigned rejected, int acl) {
              if ((rejected >> lane) & 1u) sn = held_sn;
              if (acl < 32) held_sn = shfl_f64(sn, acl);
            });
          }

          // ---- sensor input noise: white + telegraph ----
          double noise_in = 0.0, noise_out = 0.0;
          if (f_noise) {
            const double wn = par[QD_PAR_WHITE] * (double)rnd.z_white;
            if (f_white_out) noise_out = wn; else noise_in = wn;
            const double tamp = par[QD_PAR_TELE_AMP];
            if (tamp != 0.0) {
              if (!tele_init) {
                tele_state = tele_start(f_carry, seed, iy, par);
                tele_init = true;
              }
              // lanes that flip when they are reached in state 0 / in state 1
              const unsigned f0 = __ballot_sync(0xffffffffu, valid && (double)rnd.u_tele < par[QD_PAR_P01]);
              const unsigned f1 = __ballot_sync(0xffffffffu, valid && (double)rnd.u_tele < par[QD_PAR_P10]);
              unsigned st_mask = 0u, rem = 0xffffffffu, cur = tele_state;
              while (true) {
                const unsigned m = (cur ? f1 : f0) & rem;
                if (!m) { if (cur) st_mask |= rem; break; }
                const int t = __ffs(m) - 1;                       // next toggle: lanes before it keep `cur`
                if (cur) st_mask |= rem & ((1u << t) - 1u);
                cur ^= 1u;
                if (cur) st_mask |= 1u << t;
                rem &= ~((2u << t) - 1u);
                if (!rem) break;
              }
              tele_state = cur;
              noise_in += tamp * (double)((st_mask >> lane) & 1u);
            }
          }

          // ---- sensor: ten Lorentzians of the first differences of the full-system free energy ----
          const double us = fma(fy, d_us[2], fma(fx, d_us[1], d_us[0]));
          const double sg = fma(fy, d_sg[2], fma(fx, d_sg[1], d_sg[0]));
          const double base = 2.0 * (sn - sg);
          const double t = (rint(us) + noise_in) - us;
          const double xs = 2.0 * css * inv_gamma;
          const double x0 = fma(css, fma(2.0, t, 1.0), base) * inv_gamma;
          double z = (double)sensor_lorentz10(x0, xs) + noise_out;
          if (f_radial && sc->rad_mode == 1) z = fma((double)rnd.z_rad, (double)radial_amp(sc, fx, fy), z);
          zf = (float)z;
        } else {
          zf = rnd.z_rad;
        }

        // ---- coalesced stores: the key IS the uint8 charge map ----
        if (valid) {
          const long long o = pix0 + (long long)iy * nx + ix;
          if (a.z_out) a.z_out[o] = zf;
          if (a.n_type == QD_N_U8) {
            unsigned char* p = reinterpret_cast<unsigned char*>(a.n_out) + o * N;
            if constexpr (N == 8) *reinterpret_cast<uint64_t*>(p) = key;
            else if constexpr (N == 4) *reinterpret_cast<uint32_t*>(p) = (uint32_t)key;
            else if constexpr (N == 2) *reinterpret_cast<uint16_t*>(p) = (uint16_t)key;
            else {
#pragma unroll
              for (int j = 0; j < N; ++j) p[j] = (unsigned char)(key >> (8 * j));
            }
          } else if (a.n_type == QD_N_F32) {
            float* p = reinterpret_cast<float*>(a.n_out) + o * N;
#pragma unroll
            for (int j = 0; j < N; ++j) p[j] = (float)(unsigned)((key >> (8 * j)) & 0xffu);
          } else if (a.n_type == QD_N_F64) {
            double* p = reinterpret_cast<double*>(a.n_out) + o * N;
#pragma unroll
            for (int j = 0; j < N; ++j) p[j] = (double)(unsigned)((key >> (8 * j)) & 0xffu);
          }
        }
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Setup kernel: Q[delta] = delta^T Cinv delta for every env (once per qd_set_models).
// ---------------------------------------------------------------------------------------------------------------
__global__ void qd_build_q_kernel(qd_layout L, double* __restrict__ records, int n_env) {
  const int n = L.n_dot;
  const int per = 1 << n;
  const long long total = (long long)n_env * per;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int env = (int)(t / per);
    const unsigned idx = (unsigned)(t - (long long)env * per);
    double* rec = records + (size_t)env * L.rec_doubles;
    const double* cinv = rec + L.o_cinv;
    double s = 0.0;
    for (int i = 0; i < n; ++i) {
      if (!((idx >> (n - 1 - i)) & 1u)) continue;
      for (int j = 0; j < n; ++j)
        if ((idx >> (n - 1 - j)) & 1u) s += cinv[i * n + j];
    }
    rec[L.o_q + idx] = s;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// FMA micro-benchmarks: the roofline denominators of this FP-pipe-bound path (MEASURED_PEAKS.json has no CUDA-core
// figure).  8 independent chains per thread.
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) qd_fma_peak_kernel(T* out, int iters, T a, T b) {
  T x0 = (T)threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      x0 = x0 * a + b; x1 = x1 * a + b; x2 = x2 * a + b; x3 = x3 * a + b;
      x4 = x4 * a + b; x5 = x5 * a + b; x6 = x6 * a + b; x7 = x7 * a + b;
    }
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

}  // namespace qd
