// qd_tunnel_noda.cuh -- E2: the eigen stage of the tunnel-coupled path without a tridiagonalisation.
//
// Same contract as qd_tunnel_eigen_kernel (32 kept basis states per pixel in, <n> out; reference:
// src/qarray_latched/DotArrays/ground_state.py:120-160, hamiltonian_build.py:75-137, 460-483), different algorithm.
//
// H = diag(F) + hopping is block diagonal in the total charge, and every hopping element is -t sqrt(..) with t > 0 (or all
// of one sign, which a diagonal +-1 gauge turns into the same thing; |psi|^2 does not see the gauge).  Each sector is
// therefore a symmetric Z-matrix (non-positive off-diagonal), and three facts replace the dense eigen-solver:
//   * Perron-Frobenius: the ground vector of a sector is positive; A - sigma I is a nonsingular M-matrix for every
//     sigma < lambda_0, so LDL^T WITHOUT pivoting is stable, all pivots are positive, (A - sigma I)^-1 x stays positive.
//   * Sylvester: "all pivots of A - sigma I positive" <=> sigma < lambda_0.  One factorisation at the best upper bound U of
//     the global ground energy proves that a sector cannot hold the ground state (and is the certificate that an
//     aggressively chosen shift was still below the spectrum).
//   * Noda's iteration (inverse iteration whose shift is a rigorous lower bound, sigma + min_i x_i / y_i) converges
//     quadratically from any positive start.
// Per pixel: warm start every sector from the previous pixel's vectors (hash look-up by basis state), Rayleigh quotients,
// the sector with the lowest quotient is the candidate; shift it at rho - min(1.5 ||r||, 4 ||r||^2 / gap estimate), test
// the others at U = rho_candidate -- ONE warp-wide factorisation (row per lane, the row lives in registers, the pivot
// column goes through shared memory) -- then one or two triangular solves.  Everything that does not fit (a sector of
// more than 16 states, no convergence in 12 rounds) is marked with a NaN and redone by qd_tunnel_eigen_kernel in fix-up
// mode.  Prototype and iteration statistics: tools/proto_noda2.py (1.7 factorisations + 2.9 solves per pixel on the
// bench workload, |d<n>| < 2e-9 against LAPACK).
#pragma once
#include "qd_tunnel.cuh"

namespace qd {

constexpr int QD_E2_LS = 17;                         // row stride of the sector-local matrices (odd: conflict free)
constexpr int QD_E2_MAXIT = 12;

// Slot of qd_tunnel_eigen2_kernel for n_dot dots (qd_kernels.cuh: slot layouts).  Only cdd_inv is staged (by the lanes,
// from the record): the per-pixel potentials come from the relax kernel, the four scalars of the scan descriptor are
// read from global memory.  The offsets count from the start of the slot.  10.1 KB at 8 dots -> five CTAs of four warps
// per SM.
// Lm comes BEFORE H: the loops of the factorisation run to a warp-uniform bound and read up to 271 doubles past a short
// sector's rows -- with this order they land in H (finite numbers), and no padding is needed.  Small per-pixel vectors
// alias the head of Lm (dead before the first factorisation).
struct Eigen2Slot {
  int cinv;           // [n_dot^2], rounded up to an even count
  int Lm;             // [32][QD_E2_LS] the factorisation, in place
  int gs, ts;         // [8] each, at Lm + 16 and Lm + 24 doubles (aliases)
  int perm;           // int[32] the sort permutation, at Lm + 32 doubles (alias)
  int colbuf;         // [48] start vector of the first mat-vec, at Lm + 64 doubles (alias)
  int H;              // [32][QD_E2_LS] row `lane`, columns of the lane's own sector
  int hkey;           // u64 [64] hash keys
  int hx;             // [64] hash values
  int bytes;
};
__host__ __device__ constexpr Eigen2Slot qd_tunnel_eigen2_slot(int n_dot) {
  Eigen2Slot S{};
  int o = 0;
  S.cinv = o;     o += ((n_dot * n_dot + 1) & ~1) * 8;
  S.Lm = o;       o += 32 * QD_E2_LS * 8;
  S.gs = S.Lm + 16 * 8;
  S.ts = S.Lm + 24 * 8;
  S.perm = S.Lm + 32 * 8;
  S.colbuf = S.Lm + 64 * 8;
  S.H = o;        o += 32 * QD_E2_LS * 8;
  S.hkey = o;     o += 64 * 8;
  S.hx = o;       o += 64 * 8;
  S.bytes = qd_slot_round(o);
  return S;
}

// 1 / x for a positive normal x: MUFU.RCP64H seed (20 bits) + two Newton steps
__device__ __forceinline__ double rcp_nr(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
}
// 1 / sqrt(x), ~1e-12 relative (callers track the norm they actually produced)
__device__ __forceinline__ double rsqrt_nr(double x) {
  double r;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double h = 0.5 * x;
  r = r * fma(-h * r, r, 1.5);
  return r * fma(-h * r, r, 1.5);
}
// segment reductions for segments of at most 16 lanes; every lane gets its segment's value
__device__ __forceinline__ double seg_sum16(double v, int lane, int s0, int s1) {
#pragma unroll
  for (int d = 1; d < 16; d <<= 1) {
    const double t = __hiloint2double(__shfl_up_sync(0xffffffffu, __double2hiint(v), d),
                                      __shfl_up_sync(0xffffffffu, __double2loint(v), d));
    if (lane - d >= s0) v += t;
  }
  return shfl_f64(v, s1);
}
__device__ __forceinline__ double seg_min16(double v, int lane, int s0, int s1) {
#pragma unroll
  for (int d = 1; d < 16; d <<= 1) {
    const double t = __hiloint2double(__shfl_up_sync(0xffffffffu, __double2hiint(v), d),
                                      __shfl_up_sync(0xffffffffu, __double2loint(v), d));
    if (lane - d >= s0) v = min_lt(t, v);
  }
  return shfl_f64(v, s1);
}
// Sums of 8 values over the warp at once: total j ends up in the lanes with (lane >> 2) == j.  9 double shuffles instead of 40.
__device__ __forceinline__ double warp_sum8(const double (&v)[8], int lane) {
  double a[4], b[2];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool hi = lane & 16;
    const double send = hi ? v[i] : v[i + 4], keep = hi ? v[i + 4] : v[i];
    a[i] = keep + shfl_f64(send, lane ^ 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool hi = lane & 8;
    const double send = hi ? a[i] : a[i + 2], keep = hi ? a[i + 2] : a[i];
    b[i] = keep + shfl_f64(send, lane ^ 8);
  }
  const bool hi = lane & 4;
  double c = (hi ? b[1] : b[0]) + shfl_f64(hi ? b[0] : b[1], lane ^ 4);
  c += shfl_f64(c, lane ^ 2);
  c += shfl_f64(c, lane ^ 1);
  return c;
}

// minimum / maximum over the warp of a non-NaN double through two 32-bit REDUX on an order-preserving integer image
__device__ __forceinline__ unsigned long long ord_key(double v) {
  const long long b = __double_as_longlong(v);
  return (unsigned long long)b ^ ((unsigned long long)(b >> 63) | 0x8000000000000000ULL);
}
__device__ __forceinline__ double ord_val(unsigned long long k) {
  return __longlong_as_double((k >> 63) ? (long long)(k ^ 0x8000000000000000ULL) : (long long)~k);
}
__device__ __forceinline__ double warp_min_rx(double v) {
  const unsigned long long k = ord_key(v);
  const unsigned hi = (unsigned)(k >> 32);
  const unsigned mh = __reduce_min_sync(0xffffffffu, hi);
  const unsigned ml = __reduce_min_sync(0xffffffffu, hi == mh ? (unsigned)k : 0xffffffffu);
  return ord_val(((unsigned long long)mh << 32) | ml);
}
__device__ __forceinline__ double warp_max_rx(double v) {
  const unsigned long long k = ord_key(v);
  const unsigned hi = (unsigned)(k >> 32);
  const unsigned mh = __reduce_max_sync(0xffffffffu, hi);
  const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? (unsigned)k : 0u);
  return ord_val(((unsigned long long)mh << 32) | ml);
}

// LDL^T of (A - sig I) for every sector at once, in place in shared memory, rolled loops: lane = row.  W[i][k] (i > k)
// keeps l_ik d_k; the substitutions scale by 1 / d_k on the fly.  (A form with the rows in registers needs static
// indexing, i.e. full unrolling for every size: ~15 % fewer instructions per factorisation, ten times the code -- the
// kernel was then bound by instruction fetch, DESIGN.md section 4.2.)  `mact` (warp uniform) = size of the largest
// sector that matters.  Returns "my own pivot was not positive"; 1 / d_i goes to dinv.
__device__ __forceinline__ bool e2_factor_sm(const double* __restrict__ hrow, double* W, int lane, int s0, int ri, double d,
                                             double pfloor, double& dinv, int mact) {
  // Loops run to the warp-uniform mact without clamps: a sector shorter than mact reads rows past its end (other
  // sectors' rows, or -- past lane 31 -- the H17 matrix that follows W in shared memory) into columns at or beyond its
  // own size, which nothing reads back.
  double* wrow = W + lane * QD_E2_LS;
#pragma unroll 4
  for (int c = 0; c < mact; ++c) wrow[c] = hrow[c];
  wrow[min(ri, 15)] = d;
  bool fail = false;
  const double* __restrict__ diag = W + s0 * (QD_E2_LS) ;
#pragma unroll 1
  for (int k = 0; k < mact; ++k) {
    __syncwarp();
    double piv = diag[k * (QD_E2_LS + 1)];
    const bool ok = piv > pfloor;
    if (ri == k) fail = !ok;
    piv = ok ? piv : pfloor;
    const double inv = rcp_nr(piv);
    if (ri == k) dinv = inv;
    const double l = (ri > k) ? wrow[k] * inv : 0.0;
    const double* __restrict__ tp = diag + (k + 1) * QD_E2_LS + k;         // column k, rows k+1.. of the sector
    double* __restrict__ wp = wrow + k + 1;
    // two columns per trip and NO remainder code (trip counts are 0..7: remainder handling cost more than the loop); the
    // odd column past mact is the pad column of the stride-17 rows at worst
    for (int n2 = (mact - k) >> 1; n2 > 0; --n2, tp += 2 * QD_E2_LS, wp += 2) {
      const double t0 = tp[0], t1 = tp[QD_E2_LS];
      const double w0 = wp[0], w1 = wp[1];
      wp[0] = fma(-l, t0, w0);
      wp[1] = fma(-l, t1, w1);
    }
  }
  __syncwarp();
  return fail;
}
__device__ __forceinline__ double e2_solve_sm(const double* __restrict__ W, int lane, int s0, int ri, int m, double dinv, double x,
                                              int mact) {
  const double* __restrict__ wrow = W + lane * QD_E2_LS;
  double y = x;
#pragma unroll 4
  for (int k = 0; k + 1 < mact; ++k) {
    const double zk = shfl_f64(y * dinv, min(s0 + k, 31));
    const double w = wrow[k];
    if (ri > k) y = fma(-w, zk, y);
  }
  const double* __restrict__ wcol = W + s0 * QD_E2_LS + ri;      // + k * LS: W[s0 + k][ri]
#pragma unroll 4
  for (int k = mact - 1; k >= 1; --k) {
    const double zk = shfl_f64(y * dinv, min(s0 + k, 31));
    const double w = wcol[k * QD_E2_LS];
    if (ri < k && k < m) y = fma(-w, zk, y);
  }
  return y * dinv;
}

#ifndef QD_E2_MIN_BLOCKS
#define QD_E2_MIN_BLOCKS 5
#endif
template <int N>
__global__ void __launch_bounds__(128, QD_E2_MIN_BLOCKS) qd_tunnel_eigen2_kernel(const KArgs a) {
  constexpr int B = N - 1;
  constexpr unsigned FULL = 0xffffffffu;
  constexpr double INF = 1e300;
  extern __shared__ __align__(128) unsigned char qd_smem[];
  __shared__ double sq_tab[258];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const qd_layout& L = a.L;
  for (int k = threadIdx.x; k < 258; k += blockDim.x) sq_tab[k] = sqrt((double)k);
  __syncthreads();

  constexpr Eigen2Slot S = qd_tunnel_eigen2_slot(N);
  unsigned char* slot = qd_smem + (size_t)warp * a.slot_bytes;
  double* Csm = reinterpret_cast<double*>(slot + S.cinv);
  double* Lm = reinterpret_cast<double*>(slot + S.Lm);
  double* H = reinterpret_cast<double*>(slot + S.H);
  double* gs = reinterpret_cast<double*>(slot + S.gs);
  double* ts = reinterpret_cast<double*>(slot + S.ts);
  int* perm = reinterpret_cast<int*>(slot + S.perm);
  double* colbuf = reinterpret_cast<double*>(slot + S.colbuf);
  uint64_t* hkey = reinterpret_cast<uint64_t*>(slot + S.hkey);
  double* hx = reinterpret_cast<double*>(slot + S.hx);
  const double* __restrict__ C = Csm;

  const long long total_items = (long long)a.n_scan * a.items_per_scan;
  for (long long item = (long long)blockIdx.x * warps_per_cta + warp; item < total_items;
       item += (long long)gridDim.x * warps_per_cta) {
    const int scan_id = (int)(item / a.items_per_scan);
    const int part = (int)(item - (long long)scan_id * a.items_per_scan);
    const qd_scan* gscan = a.scans + scan_id;
    const int nx = gscan->nx, ny = gscan->ny;
    const long long npix = (long long)nx * ny;
    const long long p_begin = (long long)part * a.rows_per_item;
    const long long p_end = min(npix, p_begin + (long long)a.rows_per_item);
    if (p_begin >= npix) continue;
    const double* __restrict__ grec = a.records + (size_t)gscan->env_id * L.rec_doubles;
    __syncwarp();
    for (int e = lane; e < N * N; e += 32) Csm[e] = grec[L.o_cinv + e];
    const bool replace = (a.flags & QD_FLAG_RADIAL) && gscan->rad_mode == 2;
    const long long pix0 = gscan->pix_offset;
    const bool vc_on = grec[L.o_par + QD_PAR_VC_ALPHA] != 0.0 || grec[L.o_par + QD_PAR_VC_BETA] != 0.0;

    // warm start across the pixels of the item: (basis state -> vector entry) of the previous pixel, gap estimate
    hkey[lane] = ~0ULL;
    hkey[lane + 32] = ~0ULL;
    double gtil = -1.0;
    bool any_fallback = false;
    __syncwarp();

    // lane -> entry of the relax kernel's per-pixel record: potentials [0, 8) for the lanes below 16, couplings [8, 15)
    // for lanes 16.., the cdd scale [15] for lane 31
    const int tp_idx = (lane < 16) ? (lane & 7) : ((lane == 31) ? 15 : 8 + ((lane - 16) & 7));
    uint64_t key_next = 0;
    double tp_next = 0.0;
    if (!replace) {
      const size_t nslot = (size_t)scan_id * a.tstride + p_begin;
      key_next = a.tkeys[nslot * 32 + lane];
      tp_next = a.tpot[nslot * 16 + tp_idx];
    }
    for (long long pix = p_begin; pix < p_end; ++pix) {
      double* const out = a.nbar + (pix0 + pix) * N;
      if (replace) {
        if (lane < N) out[lane] = 0.0;
        continue;
      }
      uint64_t key = key_next;
      // ---------------- potentials, tunnel couplings, cdd scale: formed once per pixel by the relax kernel ----------------
      double s_c = 1.0;
      {
        if (lane < N) gs[lane] = tp_next;
        if (lane >= 16 && lane < 16 + B) ts[lane - 16] = tp_next;      // |t|: its sign is a gauge (header)
        if (vc_on) s_c = shfl_f64(tp_next, 31);
      }
      if (pix + 1 < p_end) {                       // the next pixel's states and potentials, one pixel ahead
        const size_t nslot = (size_t)scan_id * a.tstride + pix + 1;
        key_next = a.tkeys[nslot * 32 + lane];
        tp_next = a.tpot[nslot * 16 + tp_idx];
      }
      __syncwarp();
      // ---------------- free energy of this lane's state (symmetric form: upper triangle once) ----------------
      int tc = 0;
      double Fm = 0.0;
      {
        double zz[N];
#pragma unroll
        for (int j = 0; j < N; ++j) {
          const int sj = (int)(signed char)(unsigned char)(key >> (8 * j));
          zz[j] = (double)sj - gs[j];
          tc += sj;
        }
#pragma unroll
        for (int i = 0; i < N; ++i) {
          double s0_ = 0.5 * C[i * N + i] * zz[i];
#pragma unroll
          for (int j = i + 1; j < N; ++j) s0_ = fma(C[i * N + j], zz[j], s0_);
          Fm = fma(zz[i], s0_, Fm);
        }
        Fm *= 2.0;
        if (vc_on) Fm /= s_c;
      }
      // ---------------- lanes sorted by (total charge, lane): sectors = lane segments ----------------
      int s0, s1, maxlen;
      unsigned seg;
      {
        const unsigned same = __match_any_sync(FULL, tc);
        int rank = __popc(same & ((1u << lane) - 1u));
        unsigned rem = FULL;
        while (rem) {
          const int leader = __ffs(rem) - 1;
          const int v = __shfl_sync(FULL, tc, leader);
          const unsigned grp = __shfl_sync(FULL, same, leader);
          if (v < tc) rank += __popc(grp);
          rem &= ~grp;
        }
        perm[rank] = lane;
        __syncwarp();
        const int src = perm[lane];
        __syncwarp();
        key = shfl_u64(key, src);
        Fm = shfl_f64(Fm, src);
        tc = __shfl_sync(FULL, tc, src);
        seg = __match_any_sync(FULL, tc);
        s0 = __ffs(seg) - 1;
        s1 = 31 - __clz(seg);
        maxlen = __reduce_max_sync(FULL, s1 - s0 + 1);
      }
      const int m = s1 - s0 + 1, ri = lane - s0;
      bool fallback = maxlen > 16;
      double x = 0.0;
      if (!fallback) {
        // ---------------- row `lane` of H, own sector's columns; Gershgorin radius ----------------
        double rowabs = 0.0;
        double* __restrict__ hrow = H + lane * QD_E2_LS;
#pragma unroll 1
        for (int u = 0; u < maxlen; ++u) {
          const int j = min(s0 + u, 31);
          const uint64_t kj = (N <= 4) ? (uint64_t)__shfl_sync(FULL, (unsigned)key, j) : shfl_u64(key, j);
          double val = (j == lane) ? Fm : 0.0;
          // a hop p -> p+1 takes one from byte p and adds one to byte p+1: as 64-bit integers the two packed states
          // differ by exactly 0xFF << 8p (no byte wraps: occupations stay inside 0..255)
          if constexpr (N <= 4) {                     // the packed state fits 32 bits: same test at half the instructions
            const int df = (int)((unsigned)kj - (unsigned)key);
            const unsigned ad = (unsigned)(df < 0 ? -df : df);
            const int tz = __ffs((int)ad) - 1;
            if ((tz & 7) == 0 && (ad >> (tz & 31)) == 0xFFu && u < m) {
              const unsigned pa = ((unsigned)key >> tz) & 0xffffu;
              const unsigned a0 = pa & 0xffu, a1 = pa >> 8;
              const double amp = (df > 0) ? sq_tab[a0] * sq_tab[a1 + 1] : sq_tab[a1] * sq_tab[a0 + 1];
              val = -ts[tz >> 3] * amp;
              rowabs -= val;
            }
          } else {
            const long long df = (long long)(kj - key);
            const uint64_t ad = (uint64_t)(df < 0 ? -df : df);
            const int tz = __ffsll((long long)ad) - 1;
            if ((tz & 7) == 0 && (ad >> (tz & 63)) == 0xFFull && u < m) {
              const unsigned pa = (unsigned)(key >> tz) & 0xffffu;
              const unsigned a0 = pa & 0xffu, a1 = pa >> 8;
              // df > 0: the partner has one more in dot p+1 (this state hops p -> p+1), else p+1 -> p
              const double amp = (df > 0) ? sq_tab[a0] * sq_tab[a1 + 1] : sq_tab[a1] * sq_tab[a0 + 1];
              val = -ts[tz >> 3] * amp;
              rowabs -= val;
            }
          }
          hrow[u] = (u < m) ? val : 0.0;
        }
        for (int u = maxlen; u < 16; ++u) hrow[u] = 0.0;
        // ---------------- warm start ----------------
        const unsigned k32 = (unsigned)key ^ (unsigned)(key >> 32);
        const int hslot = (int)((k32 * 0x9E3779B1u) >> 26);
        {                                            // open addressing, linear probing (the table is half empty)
          int h = hslot;
          x = 0.0;
          for (;;) {                                 // (per-lane loop: no votes, the lanes reconverge behind it)
            const uint64_t kk = hkey[h];
            if (kk == key) { x = hx[h]; break; }
            if (kk == ~0ULL) break;
            h = (h + 1) & 63;
          }
          __syncwarp();
        }
        x = fmax(x, 1e-3);
        colbuf[lane] = x;
        if (lane < 16) colbuf[32 + lane] = 0.0;          // (what a lane of the last sectors reads past lane 31)
        __syncwarp();
        double w = 0.0;
        {
          const double* __restrict__ xs = colbuf + s0;
#pragma unroll 1
          for (int u = 0; u < maxlen; ++u) w = fma(hrow[u], xs[u], w);
        }
        const double xx0 = seg_sum16(x * x, lane, s0, s1);
        const double xw = seg_sum16(x * w, lane, s0, s1);
        const double ixx = rcp_nr(xx0);
        const double rho0 = xw * ixx;
        const double rres = fma(-rho0, x, w);
        const double rr = seg_sum16(rres * rres, lane, s0, s1) * ixx;
        const double gersh = seg_min16(Fm - rowabs, lane, s0, s1);
        const double scale = warp_max_rx(fabs(Fm) + rowabs) + 1e-300;
        const double tiny = 1e-14 * scale, pfloor = 1e-15 * scale;
        double xs_ = rsqrt_nr(xx0);
        x *= xs_;
        double xx = xx0 * xs_ * xs_;                      // |x|^2 as produced (1 to ~1e-12)
        __syncwarp();

        // ---------------- sector state (uniform inside a sector) ----------------
        const double U0 = warp_min_rx(rho0);
        const bool isg = rho0 == U0;
        double lo = gersh, ub = rho0, sig;
        bool live = true, done = false, test = !isg, agg = false, valid = false, tested = false;
        double tested_at = 0.0, dinv = 1.0;
        bool nudged = false;
        float eps_prev = 1.0f;
        int nsol = 0;
        if (isg) {
          double eta = 1.5 * (double)sqrtf((float)rr);
          if (gtil > 0.0) eta = fmin(eta, (double)a.e2_kappa * rr / gtil);
          eta += 1e-13 * scale;
          sig = fmax(lo, rho0 - eta);
          agg = sig > lo;
        } else {
          sig = U0;
        }
        if (m == 1) { done = true; lo = ub = Fm; live = isg; x = 1.0; xx = 1.0; }
        bool need_fac = true;
#ifdef QD_E2_STATS
        int st_fac = 0, st_it = 0, st_aggfail = 0, st_testfail = 0;
#endif
        for (int it = 0;; ++it) {
          const double U = warp_min_rx(live ? ub : INF);
          if (live && !test && lo > U + tiny) live = false;
          const bool act = live && !done;
          if (!__any_sync(FULL, act)) break;
          if (it >= QD_E2_MAXIT) { fallback = true; break; }
          const int mact = __reduce_max_sync(FULL, act ? m : 0);
          if (need_fac) {
            if (test && live) sig = U;
            const bool fl = e2_factor_sm(hrow, Lm, lane, s0, ri, Fm - sig, pfloor, dinv, mact);
            const unsigned fm = __ballot_sync(FULL, fl);
            valid = (m <= mact) && !(fm & seg);
            __syncwarp();
          }
#ifdef QD_E2_STATS
          st_fac += need_fac; ++st_it;
          st_aggfail += __any_sync(FULL, act && !test && !valid && agg);
          st_testfail += __any_sync(FULL, act && test && !valid);
#endif
          double y = e2_solve_sm(Lm, lane, s0, ri, m, dinv, x, mact);
          const bool usable = valid && m <= mact && m > 1;
          if (!usable) y = x;
          const double ny2 = seg_sum16(y * y, lane, s0, s1);
          const double xy = seg_sum16(x * y, lane, s0, s1);
          bool nf = false, want_rmin = false;
          if (act) {
            if (test) {
              if (valid) {
                live = false;                       // every eigenvalue of this sector lies above U
              } else {
                nf = true;
                if (tested && tested_at - U < 1e-3 * (fabs(U) + 1.0)) { test = false; sig = lo; }   // a real competitor
                tested = true;
                tested_at = U;
              }
            } else if (!valid) {
              if (!agg) {
                // a rigorous lower bound that is singular to rounding: lambda_0 is known, the VECTOR may still be the start
                // vector -- step back by a hair (still 1e5 times closer than any gap that matters) and iterate on
                ub = fmin(ub, sig + tiny);
                if (!nudged) { sig = lo - 1e-10 * scale; nudged = true; nf = true; }
                else done = true;
              }
              else { ub = fmin(ub, sig); sig = lo; agg = false; nf = true; }   // the aggressive shift was above lambda_0
            } else {
              lo = fmax(lo, sig);
              const double iny2 = rcp_nr(ny2);
              ub = fmin(ub, fma(xy, iny2, sig));
              const double sin2 = fmax(0.0, 1.0 - (xy * xy) * iny2 * rcp_nr(xx));
              const float eps = sqrtf((float)sin2);
              ++nsol;
              if (nsol == 1) {
                if (agg) {
                  if (gtil > 0.0) {
                    const float q = fminf(1.0f, a.e2_qsafe * (float)((ub - sig) / gtil));
                    if (eps * q < a.e2_tol || eps < 3e-8f) done = true;
                    else if (q > 0.03f) want_rmin = true;
                  } else if (eps < 3e-8f) {
                    done = true;
                  }
                } else {
                  want_rmin = true;
                }
              } else {
                const float q = fminf(1.0f, eps / eps_prev);
                if (eps * q < a.e2_tol) done = true;
                else if (q > 0.03f) want_rmin = true;
              }
              eps_prev = eps;
            }
          }
          if (__any_sync(FULL, want_rmin)) {
            const double rmin = seg_min16(usable ? x * rcp_nr(y) : INF, lane, s0, s1);
            if (want_rmin) {
              lo = fmax(lo, fma(rmin, 1.0 - 1e-12, sig));
              sig = lo;
              agg = false;
              nf = true;
            }
          }
          if (usable) {                              // (a sector that is out still takes the free inverse-iteration step)
            const double s = rsqrt_nr(ny2);
            x = y * s;
            xx = ny2 * s * s;
          }
          need_fac = __any_sync(FULL, nf);
        }
        if (!fallback) {
          // ---------------- <n> from the winning sector ----------------
          const double Uf = warp_min_rx(live ? ub : INF);
          const bool win = live && ub == Uf;
          const double w2 = win ? x * x : 0.0;
          double v8[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v8[j] = (j < N) ? w2 * (double)(int)(signed char)(unsigned char)(key >> (8 * j)) : 0.0;
          const double tot = warp_sum(w2);
          const double sj = warp_sum8(v8, lane);
          if ((lane & 3) == 0 && (lane >> 2) < N) out[lane >> 2] = sj / tot;
#ifdef QD_E2_STATS
          __syncwarp();
          if (lane == 0 && N >= 4) { out[0] = st_fac; out[1] = st_it; out[2] = st_aggfail; out[3] = st_testfail; }
#endif
          // gap estimate for the next pixel (Temple's bound read backwards on this pixel's start vector)
          const double over = rho0 - ub;
          const double gcand = (win && over > 0.0 && rr > 0.0) ? rr / over : -1.0;
          gtil = warp_max_rx(gcand);
        }
      }
      hkey[lane] = ~0ULL;                            // the table holds the current pixel only
      hkey[lane + 32] = ~0ULL;
      __syncwarp();
      if (fallback) {
        if (lane == 0) out[0] = __longlong_as_double(0x7ff8000000000000LL);      // redone by the fix-up pass
        gtil = -1.0;
        any_fallback = true;
      } else {
        const unsigned k32 = (unsigned)key ^ (unsigned)(key >> 32);
        int h = (int)((k32 * 0x9E3779B1u) >> 26);
        // claim the first free slot from the home slot on with a shared-memory compare-and-swap (a warp-wide match per
        // probing round cost 4 % of the kernel's time in stalls)
        unsigned long long* hk = reinterpret_cast<unsigned long long*>(hkey);
        while (atomicCAS(hk + h, ~0ULL, (unsigned long long)key) != ~0ULL) h = (h + 1) & 63;
        hx[h] = x;
      }
      __syncwarp();
    }
    // item-level mark for the fix-up pass, in the (by now consumed) floor scratch of the item's first pixel
    if (lane == 0) a.tfloor[((size_t)scan_id * a.tstride + p_begin) * 8] = any_fallback ? 0xff : 0;
    __syncwarp();
  }
}

}  // namespace qd
