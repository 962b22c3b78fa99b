// qd_tunnel.cuh -- Path B: the tunnel-coupled ground state QADAPT's env.step runs in barrier mode
// (src/qarray_latched/DotArrays/ground_state.py:24-166; restated in oracle/path_b.py).  sm_100a, one WARP per pixel:
// the 32-state truncated basis maps one basis state to one lane.
//
// Per pixel (all 32 lanes cooperate):
//   1. dot potentials g = cgd[:N] v (scaled per pixel when the linear voltage-dependent capacitance model is on),
//      continuous relaxation: closed form, or the reference's 50 projected-gradient steps (in registers: lane 4i + p
//      owns two columns of row i, a 4-lane butterfly per step).
//   2. 4^N candidates floor(n_c) + {-1,0,1,2}^N.  E = z^T C z, z = r + delta.  The digits split into a high and a low
//      half (<= 256 combinations each; the most deeply empty dots go to the high half, chosen per work item).  A block
//      = one high combination.  Blocks are visited in increasing order of the Schur-complement lower bound
//      z_hi^T (Chh - Chl Cll^-1 Clh) z_hi and the walk stops when the bound exceeds the current 32nd-best energy: exact.
//      The running top-32 lives sorted across the lanes, ordered by (energy, index) = the reference's stable sort; it is
//      WARM-STARTED from the previous pixel's basis (re-evaluated with the same arithmetic, bitonic-sorted), so the walk
//      only inserts the newcomers.
//   3. H = diag(F) + nearest-neighbour hopping -t_d sqrt(n_from (n_to + 1)), t_d = tc_base exp(-alpha_d vb_eff_d).
//      Hopping conserves the total charge: the lanes are sorted by (total charge, lane), H is block diagonal, and every
//      dense step below runs on all SECTORS at once, each in its own lane segment (segmented shuffle scans).
//   4. Ground eigenvector: Householder tridiagonalisation in shared memory (lane = row, largest sector - 2 steps),
//      lowest eigenvalue bracketed by 32-way multisection -- x < lambda_0 iff every leading principal minor of
//      T - x I is positive, on the tridiagonal mapped to [0, 1] -- then per sector LDL^T (T - mu I is positive definite
//      at the lower bracket end: no pivoting) and inverse iteration by the sector's leader lane, back-transformation.
//   5. <n> = sum_m psi_m^2 n_m is written to a scratch buffer; latching, sensor and noise are then applied by
//      qd_scan_kernel<N, QD_ALG_TUNNEL> (lane per pixel), so a flat latching pass never serialises the eigen-solves.
#pragma once
#include "qd_kernels.cuh"

namespace qd {

constexpr int QD_T_HS = 33;                       // row stride of H in shared memory (bank-conflict free)

// Slot of qd_tunnel_gs_kernel (qd_kernels.cuh: slot layouts).  It stages the record's gs_doubles PREFIX only
// (qd_layout.h).
struct TunnelSlot {
  size_t rec_bytes;   // [gs_doubles] the record prefix (TMA destination); the offsets below count from its end
  int scan;           // qd_scan, the descriptor (TMA destination)
  int H;              // [32][QD_T_HS] the Hamiltonian
  int dd, ee, e2, qi, ll, yy;   // [32] each
  int vq;             // [64] interleaved (v_j, q_j) of the current Householder step, read as double2, + spare row [32]
  int vv;             // [16]
  int gs, ns, fs, hs, ts, nb;   // [8] each
  int Cp;             // [64] Cinv with rows / columns permuted so that the stiffest dots come first
  int Sp;             // [16] Schur complement of the permuted high block
  int Ql;             // [256] y^T Cp_ll y over the low digit combinations
  int pm;             // int[16] pm[j]: dot at permuted position j, pm[8 + d]: position of dot d (16 doubles reserved)
  int bar;            // mbarrier of the two copies (16 bytes)
  int bytes;
};
__host__ __device__ constexpr TunnelSlot qd_tunnel_slot(const qd_layout& L) {
  TunnelSlot S{};
  S.rec_bytes = (size_t)L.gs_doubles * 8;
  int o = 0;
  S.scan = o;     o += (int)sizeof(qd_scan);
  S.H = o;        o += 32 * QD_T_HS * 8;
  S.dd = o;       o += 32 * 8;
  S.ee = o;       o += 32 * 8;
  S.e2 = o;       o += 32 * 8;
  S.qi = o;       o += 32 * 8;
  S.ll = o;       o += 32 * 8;
  S.yy = o;       o += 32 * 8;
  S.vq = o;       o += 96 * 8;
  S.vv = o;       o += 16 * 8;
  S.gs = o;       o += 8 * 8;
  S.ns = o;       o += 8 * 8;
  S.fs = o;       o += 8 * 8;
  S.hs = o;       o += 8 * 8;
  S.ts = o;       o += 8 * 8;
  S.nb = o;       o += 8 * 8;
  S.Cp = o;       o += 64 * 8;
  S.Sp = o;       o += 16 * 8;
  S.Ql = o;       o += 256 * 8;
  S.pm = o;       o += 16 * 8;
  S.bar = o;      o += 16;
  S.bytes = qd_slot_round(S.rec_bytes + o);
  return S;
}

// Scales of the voltage-dependent capacitance models (voltage_dependent_capacitance.py:78-125; include/qdsim.h enum
// qd_vc_kind): cdd -> s_c cdd, cgd -> s_g cgd, from sum|v_k| and sum v_k^2 over ALL voltages of the pixel.
__device__ __forceinline__ void vc_scales(const double* __restrict__ par, double vabs, double v2, int NV, double& s_c, double& s_g) {
  const double vmean = vabs / (double)NV;
  s_g = fma(par[QD_PAR_VC_BETA], vmean, 1.0);
  const int kind = (int)par[QD_PAR_VC_KIND];
  if (kind == QD_VC_QUADRATIC) s_c = fma(par[QD_PAR_VC_ALPHA], v2, 1.0);
  else if (kind == QD_VC_SIGMOID) s_c = 1.0 + par[QD_PAR_VC_ALPHA] / (1.0 + exp(1.0 - sqrt(v2) / par[QD_PAR_VC_VCHAR]));
  else s_c = fma(par[QD_PAR_VC_ALPHA], vmean, 1.0);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double t = __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(v), o),
                                      __shfl_xor_sync(0xffffffffu, __double2loint(v), o));
    v += t;
  }
  return v;
}
// sum over the lane segment [s0, s1] that contains this lane (segments tile the warp); every lane gets its segment's sum
__device__ __forceinline__ double seg_sum(double v, int lane, int s0, int s1, bool wide) {
#pragma unroll
  for (int d = 1; d < 16; d <<= 1) {
    const double t = __hiloint2double(__shfl_up_sync(0xffffffffu, __double2hiint(v), d),
                                      __shfl_up_sync(0xffffffffu, __double2loint(v), d));
    if (lane - d >= s0) v += t;
  }
  if (wide) {                                      // segments longer than 16 lanes (warp-uniform flag)
    const double t = __hiloint2double(__shfl_up_sync(0xffffffffu, __double2hiint(v), 16),
                                      __shfl_up_sync(0xffffffffu, __double2loint(v), 16));
    if (lane - 16 >= s0) v += t;
  }
  return __hiloint2double(__shfl_sync(0xffffffffu, __double2hiint(v), s1), __shfl_sync(0xffffffffu, __double2loint(v), s1));
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, shfl_f64(v, (threadIdx.x & 31) ^ o));
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, shfl_f64(v, (threadIdx.x & 31) ^ o));
  return v;
}
__device__ __forceinline__ bool lex_less(double e1, int i1, double e2, int i2) {
  return e1 < e2 || (e1 == e2 && i1 < i2);
}

// lexicographic (energy, index) maximum over the warp and the lane that holds it
__device__ __forceinline__ void warp_lex_max(double e, int idx, int lane, double& me, int& mi, int& ml) {
  me = e; mi = idx; ml = lane;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double oe = shfl_f64(me, lane ^ o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    const int ol = __shfl_xor_sync(0xffffffffu, ml, o);
    const bool take = lex_less(me, mi, oe, oi) || (me == oe && mi == oi && ol > ml);
    if (take) { me = oe; mi = oi; ml = ol; }
  }
}

// Energy of the low candidate b = 32 i + lane_b inside a block with constants (base, c):  the digits of b split into
// bits taken from lane_b and bits taken from i.  Written once so that the streaming pass (which hoists the lane part
// out of its loop) and the warm start evaluate a candidate with the very same operations.
template <int NLO>
__device__ __forceinline__ double tunnel_lane_part(double base, const double (&c)[NLO], int lane_b) {
#pragma unroll
  for (int k = 0; k < NLO; ++k) {
    const int sh = 2 * (NLO - 1 - k);
    const int dg = (sh >= 5) ? 0 : ((lane_b >> sh) & 3 & ((sh == 4) ? 1 : 3));
    base = fma(2.0 * c[k], (double)(dg - 1), base);
  }
  return base;
}
template <int NLO>
__device__ __forceinline__ double tunnel_iter_part(double e, const double (&c)[NLO], int i) {
#pragma unroll
  for (int k = 0; k < NLO; ++k) {
    const int sh = 2 * (NLO - 1 - k);              // bit position of digit k inside b
    if (sh + 2 > 5) {                               // (part of) the digit comes from i
      const int di = (sh >= 5) ? ((i >> (sh - 5)) & 3) : ((i << (5 - sh)) & 3);
      e = fma(2.0 * c[k], (double)di, e);
    }
  }
  return e;
}
// block constants: base = E0 + 2 x.h_hi + x^T Cp_hh x;  c_k = h_lo[k] + sum_j Cp[lo k][hi j] x_j   (x = high deltas)
template <int N, int NHI, int NLO>
__device__ __forceinline__ void tunnel_block_constants(int mb, double E0, const double (&h)[N],
                                                       const double* __restrict__ Cp, double& base, double (&c)[NLO]) {
  base = E0;
#pragma unroll
  for (int k = 0; k < NLO; ++k) c[k] = h[NHI + k];
  double xh[NHI > 0 ? NHI : 1];
#pragma unroll
  for (int j = 0; j < NHI; ++j) xh[j] = (double)(((mb >> (2 * (NHI - 1 - j))) & 3) - 1);
#pragma unroll
  for (int j = 0; j < NHI; ++j) {
    double s = fma(Cp[j * N + j], xh[j], 2.0 * h[j]);          // symmetric: diagonal + twice the strict upper part
#pragma unroll
    for (int q = j + 1; q < NHI; ++q) s = fma(2.0 * Cp[j * N + q], xh[q], s);
    base = fma(xh[j], s, base);
#pragma unroll
    for (int k = 0; k < NLO; ++k) c[k] = fma(Cp[(NHI + k) * N + j], xh[j], c[k]);
  }
}

template <int N>
__global__ void __launch_bounds__(128, 3) qd_tunnel_gs_kernel(const KArgs a) {
  constexpr int NLO = N < 4 ? N : 4;
  constexpr int NHI = N - NLO;
  constexpr int NB_LO = 1 << (2 * NLO);            // low candidates per block
  constexpr int NB_HI = 1 << (2 * NHI);            // blocks
  constexpr int LO_IT = NB_LO >= 32 ? NB_LO / 32 : 1;
  constexpr int HI_IT = NB_HI >= 32 ? NB_HI / 32 : 1;
  constexpr int B = N - 1;

  extern __shared__ __align__(128) unsigned char qd_smem[];
  __shared__ double sq_tab[258];                   // sqrt(k), k = 0..257: hopping amplitudes sqrt(n_from (n_to + 1))
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const qd_layout& L = a.L;
  const int NV = L.n_volt, G = L.n_gate;
  const bool barriers = NV > G;
  for (int k = threadIdx.x; k < 258; k += blockDim.x) sq_tab[k] = sqrt((double)k);
  __syncthreads();

  unsigned char* slot = qd_smem + (size_t)warp * a.slot_bytes;
  const TunnelSlot S = qd_tunnel_slot(L);
  unsigned char* tail = slot + S.rec_bytes;
  double* rec = reinterpret_cast<double*>(slot);
  qd_scan* sc = reinterpret_cast<qd_scan*>(tail + S.scan);
  double* H = reinterpret_cast<double*>(tail + S.H);
  double* dd = reinterpret_cast<double*>(tail + S.dd);
  double* ee = reinterpret_cast<double*>(tail + S.ee);
  double* e2 = reinterpret_cast<double*>(tail + S.e2);
  double* qi = reinterpret_cast<double*>(tail + S.qi);
  double* ll = reinterpret_cast<double*>(tail + S.ll);
  double* yy = reinterpret_cast<double*>(tail + S.yy);
  double* vq = reinterpret_cast<double*>(tail + S.vq);
  double* vv = reinterpret_cast<double*>(tail + S.vv);
  double* gs = reinterpret_cast<double*>(tail + S.gs);
  double* ns = reinterpret_cast<double*>(tail + S.ns);
  double* fs = reinterpret_cast<double*>(tail + S.fs);
  double* hs = reinterpret_cast<double*>(tail + S.hs);
  double* ts = reinterpret_cast<double*>(tail + S.ts);
  double* nb = reinterpret_cast<double*>(tail + S.nb);
  double* Cp = reinterpret_cast<double*>(tail + S.Cp);
  double* Sp = reinterpret_cast<double*>(tail + S.Sp);
  double* Ql = reinterpret_cast<double*>(tail + S.Ql);
  int* pm = reinterpret_cast<int*>(tail + S.pm);
  uint64_t* bar = reinterpret_cast<uint64_t*>(tail + S.bar);

  const double* __restrict__ C = rec + L.o_cinv;
  const double INF = __longlong_as_double(0x7ff0000000000000LL);

  if (lane == 0) mbar_init(bar, 1);
  __syncwarp();
  uint32_t phase = 0;
  const uint32_t rec_bytes = (uint32_t)L.gs_doubles * 8u;

  const long long total_items = (long long)a.n_scan * a.items_per_scan;
  for (long long item = (long long)blockIdx.x * warps_per_cta + warp; item < total_items;
       item += (long long)gridDim.x * warps_per_cta) {
    const int scan_id = (int)(item / a.items_per_scan);
    const int part = (int)(item - (long long)scan_id * a.items_per_scan);
    const qd_scan* gscan = a.scans + scan_id;
    stage_item(a, gscan, rec_bytes, rec, sc, bar, phase, lane);

    const int nx = sc->nx, ny = sc->ny;
    const long long npix = (long long)nx * ny;
    const long long p_begin = (long long)part * a.rows_per_item;            // rows_per_item = pixels per item here
    const long long p_end = min(npix, p_begin + (long long)a.rows_per_item);
    if (p_begin >= npix) { __syncwarp(); continue; }

    const double* par = rec + L.o_par;
    const bool replace = (a.flags & QD_FLAG_RADIAL) && sc->rad_mode == 2;
    const long long pix0 = sc->pix_offset;
    const bool vc_on = par[QD_PAR_VC_ALPHA] != 0.0 || par[QD_PAR_VC_BETA] != 0.0;

    // ---- per-item split of the dots into a high and a low half ----
    // Any split is exact; its only job is to make the block bound bite.  Dots that are empty and far below their
    // first charge transition (very negative potential) have no cheap excitation: putting them in the HIGH half makes
    // every block that moves them cost far more than the 32nd-best energy, so it is never visited.  The order is
    // taken from the potentials at the item's first pixel; the tables of the two halves are rebuilt for it here.
    if (!replace) {
      const long long pf = p_begin;
      const int fy = (int)(pf / nx), fx = (int)(pf - (long long)fy * nx);
      if (lane < NV)
        vv[lane] = (a.points == nullptr) ? fma((double)fy, sc->dy[lane], fma((double)fx, sc->dx[lane], sc->v0[lane]))
                                         : a.points[(size_t)pf * NV + lane];
      __syncwarp();
      if (lane < N) {
        double acc = 0.0;
        for (int k = 0; k < NV; ++k) acc = fma(rec[L.o_a + lane * NV + k], vv[k], acc);
        gs[lane] = acc;
      }
      __syncwarp();
      if (lane == 0) {
        int ord[N];
        for (int j = 0; j < N; ++j) ord[j] = j;
        for (int i = 1; i < N; ++i) {                      // insertion sort, ascending potential (most negative first)
          const int o = ord[i];
          int j = i - 1;
          while (j >= 0 && gs[ord[j]] > gs[o]) { ord[j + 1] = ord[j]; --j; }
          ord[j + 1] = o;
        }
        for (int j = 0; j < N; ++j) { pm[j] = ord[j]; pm[8 + ord[j]] = j; }
      }
      __syncwarp();
      for (int e = lane; e < N * N; e += 32) Cp[e] = C[pm[e / N] * N + pm[e % N]];
      __syncwarp();
      if (lane == 0) {
        // Sp = Chh - Chl Cll^-1 Clh  (Gauss-Jordan on the low block, <= 4 x 4)
        double m[4][8];
        for (int i = 0; i < NLO; ++i)
          for (int j = 0; j < NLO; ++j) { m[i][j] = Cp[(NHI + i) * N + NHI + j]; m[i][NLO + j] = (i == j) ? 1.0 : 0.0; }
        for (int k = 0; k < NLO; ++k) {
          const double inv = 1.0 / m[k][k];
          for (int j = 0; j < 2 * NLO; ++j) m[k][j] *= inv;
          for (int i = 0; i < NLO; ++i) {
            if (i == k) continue;
            const double fac = m[i][k];
            for (int j = 0; j < 2 * NLO; ++j) m[i][j] -= fac * m[k][j];
          }
        }
        for (int i = 0; i < NHI; ++i)
          for (int j = 0; j < NHI; ++j) {
            double acc = Cp[i * N + j];
            for (int p = 0; p < NLO; ++p)
              for (int q = 0; q < NLO; ++q) acc -= Cp[i * N + NHI + p] * m[p][NLO + q] * Cp[(NHI + q) * N + j];
            Sp[i * NHI + j] = acc;
          }
      }
      for (int idx = lane; idx < NB_LO; idx += 32) {
        double acc = 0.0;
        for (int i = 0; i < NLO; ++i)
          for (int j = 0; j < NLO; ++j)
            acc += (double)(((idx >> (2 * (NLO - 1 - i))) & 3) - 1) * Cp[(NHI + i) * N + NHI + j] *
                   (double)(((idx >> (2 * (NLO - 1 - j))) & 3) - 1);
        Ql[idx] = acc;
      }
      __syncwarp();
    }

    {
      {
        uint64_t prev_key = ~0ULL;       // this lane's basis state at the previous pixel of the item (~0: none / padding)
        bool have_prev = false;
        for (long long pix = p_begin; pix < p_end; ++pix) {
        const int iy = (int)(pix / nx), ix = (int)(pix - (long long)iy * nx);
        double nbar[N];
        if (!replace) {
          // ---------------- 1. voltages, potentials, tunnel couplings ----------------
          if (lane < NV) {
            vv[lane] = (a.points == nullptr)
                           ? fma((double)iy, sc->dy[lane], fma((double)ix, sc->dx[lane], sc->v0[lane]))
                           : a.points[(size_t)pix * NV + lane];
          }
          __syncwarp();
          {
            if (lane < N) {
              double acc = 0.0;
              const double* arow = rec + L.o_a + lane * NV;
              for (int k = 0; k < NV; ++k) acc = fma(arow[k], vv[k], acc);
              if (vc_on) {
                // linear voltage-dependent capacitances (voltage_dependent_capacitance.py:78-91): cgd scales by
                // 1 + beta mean|v|, cdd by 1 + alpha mean|v| (so cdd^-1 by its inverse)
                double vabs = 0.0, v2 = 0.0, s_c, s_g;
                for (int k = 0; k < NV; ++k) { vabs += fabs(vv[k]); v2 = fma(vv[k], vv[k], v2); }
                vc_scales(par, vabs, v2, NV, s_c, s_g);
                acc *= s_g;
                if (lane == 0) ts[7] = s_c;
              }
              gs[lane] = acc;
            }
            if (lane >= 16 && lane < 16 + B) {
              const int d = lane - 16;
              double t = par[QD_PAR_TC_BASE];
              if (barriers) {
                double vb = vv[G + d];
                for (int k = 0; k < G; ++k) vb = fma(rec[L.o_cbg + d * G + k], vv[k], vb);
                t *= exp(-rec[L.o_alpha + d] * vb);
              }
              ts[d] = t;
            }
          }
          __syncwarp();
          // ---------------- continuous relaxation (charge_states.py:36-88) ----------------
          // Lane (4 i + p) works for dot i on the columns k = 2p, 2p + 1 of C: a projected-gradient step is two
          // products, a 4-lane butterfly and the update, all in registers (no shared-memory round trip per step).
          {
            const int di = lane >> 2, dp = lane & 3;
            const int k0 = 2 * dp, k1 = 2 * dp + 1;
            const bool own = di < N;
            const double gi = own ? gs[di] : 0.0;
            double ni = gi;
            if (__ballot_sync(0xffffffffu, own && gi < 0.0)) {
              const double c0 = (own && k0 < N) ? C[di * N + k0] : 0.0;
              const double c1 = (own && k1 < N) ? C[di * N + k1] : 0.0;
              const int l0 = (k0 < N) ? 4 * k0 : lane, l1 = (k1 < N) ? 4 * k1 : lane;   // lanes holding n_k0, n_k1
              double cg = fma(c0, (k0 < N) ? gs[k0] : 0.0, c1 * ((k1 < N) ? gs[k1] : 0.0));
              cg += shfl_f64(cg, lane ^ 1);
              cg += shfl_f64(cg, lane ^ 2);
              ni = fmax(gi, 0.0);
              const double lr = vc_on ? 0.1 / ts[7] : 0.1;       // the gradient carries cdd^-1 / s_c
              for (int it = 0; it < 50; ++it) {
                double part = fma(c0, shfl_f64(ni, l0), c1 * shfl_f64(ni, l1));
                part += shfl_f64(part, lane ^ 1);
                part += shfl_f64(part, lane ^ 2);
                ni = fmax(ni - lr * (part - cg), 0.0);
              }
            }
            ni = fmax(ni, 0.0);
            if (own && dp == 0) {
              const double fj = floor(ni);
              fs[di] = fj;
              ns[di] = fj - gi;                      // r = f - g
            }
          }
          __syncwarp();
          if (lane < N) {                            // h = C r
            double s = 0.0;
            for (int k = 0; k < N; ++k) s = fma(C[lane * N + k], ns[k], s);
            hs[lane] = s;
          }
          __syncwarp();
          double f[N], r[N], h[N];
#pragma unroll
          for (int j = 0; j < N; ++j) { const int d = pm[j]; f[j] = fs[d]; r[j] = ns[d]; h[j] = hs[d]; }   // permuted order
          double E0 = 0.0;
#pragma unroll
          for (int j = 0; j < N; ++j) E0 = fma(r[j], h[j], E0);

          // ---------------- 2. streaming top-32 over the 4^N candidates ----------------
          // lane l holds the l-th smallest (energy, index) seen so far; tau = lane 31's entry, replicated in every lane
          double le = INF;
          int lidx = -1;                             // -1: the reference's zero-state padding entry
          double tau = INF;
          int tau_idx = 0x7fffffff;
          // Warm start.  Neighbouring pixels keep almost the same 32 states: re-evaluate the previous pixel's basis at
          // this pixel (each lane its own state, with the streaming pass's own arithmetic), sort it, and let it be the
          // initial list.  The pass below then only inserts the few newcomers -- the final list is the exact
          // (energy, index) top-32 either way, the warm start only spares ~70 insertions per pixel.
          if (have_prev) {
            bool okp = prev_key != ~0ULL;
            int idx = 0;
#pragma unroll
            for (int j = 0; j < N; ++j) {
              const int dg = (int)(signed char)(unsigned char)(prev_key >> (8 * j)) - (int)fs[j] + 1;
              okp = okp && dg >= 0 && dg <= 3;
              idx |= (dg & 3) << (2 * (N - 1 - pm[8 + j]));
            }
            if (okp) {
              double base;
              double c[NLO];
              const int b = idx & (NB_LO - 1);
              tunnel_block_constants<N, NHI, NLO>(idx >> (2 * NLO), E0, h, Cp, base, c);
              le = tunnel_iter_part<NLO>(tunnel_lane_part<NLO>(base, c, b & 31) + Ql[b], c, b >> 5);
              lidx = idx;
            }
            // bitonic sort of the 32 (energy, index) pairs across the lanes, ascending; padding (inf, -1) goes last
#pragma unroll
            for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
              for (int j = k >> 1; j > 0; j >>= 1) {
                const double oe = shfl_f64(le, lane ^ j);
                const int oi = __shfl_xor_sync(0xffffffffu, lidx, j);
                const bool keep_min = ((lane & j) == 0) == ((lane & k) == 0);
                const bool take = keep_min ? lex_less(oe, oi, le, lidx) : lex_less(le, lidx, oe, oi);
                if (take) { le = oe; lidx = oi; }
              }
            }
            tau = shfl_f64(le, 31);
            tau_idx = __shfl_sync(0xffffffffu, lidx, 31);
            if (!(tau < INF)) tau_idx = 0x7fffffff;
          }
          // validity of this lane's low candidates and their digit vectors do not depend on the block
          unsigned lo_valid = 0;
#pragma unroll
          for (int i = 0; i < LO_IT; ++i) {
            const int b = i * 32 + lane;
            bool ok = b < NB_LO;
#pragma unroll
            for (int k = 0; k < NLO; ++k) {
              const int dg = (b >> (2 * (NLO - 1 - k))) & 3;
              ok = ok && !(dg == 0 && f[NHI + k] <= 0.0);
            }
            lo_valid |= ok ? (1u << i) : 0u;
          }
          // lower bounds of this lane's blocks
          double lb[HI_IT];
#pragma unroll
          for (int i = 0; i < HI_IT; ++i) {
            const int blk = i * 32 + lane;
            double v = INF;
            if (blk < NB_HI) {
              bool ok = true;
              double zh[NHI > 0 ? NHI : 1];
#pragma unroll
              for (int j = 0; j < NHI; ++j) {
                const int dg = (blk >> (2 * (NHI - 1 - j))) & 3;
                ok = ok && !(dg == 0 && f[j] <= 0.0);
                zh[j] = r[j] + (double)(dg - 1);
              }
              if (ok) {
                v = 0.0;
#pragma unroll
                for (int p = 0; p < NHI; ++p) {
                  double s = 0.0;
#pragma unroll
                  for (int q = 0; q < NHI; ++q) s = fma(Sp[p * NHI + q], zh[q], s);
                  v = fma(zh[p], s, v);
                }
              }
            }
            lb[i] = v;
          }
          while (true) {
            // next unvisited block with the smallest bound
            double m = INF;
            int mb = 0x7fffffff;
#pragma unroll
            for (int i = 0; i < HI_IT; ++i)
              if (lb[i] < m) { m = lb[i]; mb = i * 32 + lane; }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              const double om = shfl_f64(m, lane ^ o);
              const int ob = __shfl_xor_sync(0xffffffffu, mb, o);
              if (om < m || (om == m && ob < mb)) { m = om; mb = ob; }
            }
            if (!(m < INF)) break;
            if (m - 1e-12 * (fabs(m) + 1.0) > tau) break;      // every remaining candidate is above the 32nd best
#pragma unroll
            for (int i = 0; i < HI_IT; ++i)
              if (mb == i * 32 + lane) lb[i] = INF;
            double base;
            double c[NLO];
            tunnel_block_constants<N, NHI, NLO>(mb, E0, h, Cp, base, c);
            const double base_lane = tunnel_lane_part<NLO>(base, c, lane);      // lane part, once per block
#pragma unroll 1
            for (int ii = 0; ii < LO_IT; ++ii) {
              // start with the leading low digit at delta 0 / +1 (the candidates around the continuous minimum), so
              // that the running 32nd-best energy tightens early and the far candidates never enter the list
              const int i = (LO_IT >= 4) ? ((ii + LO_IT / 4) & (LO_IT - 1)) : ii;
              const int b = i * 32 + lane;
              const bool ok = (lo_valid >> i) & 1u;
              double e = INF;
              if (ok) {
                e = tunnel_iter_part<NLO>(base_lane + Ql[b], c, i);
              }
              const int cidx = mb * NB_LO + b;
              unsigned pm = __ballot_sync(0xffffffffu, ok && lex_less(e, cidx, tau, tau_idx));
              while (pm) {
                const int p = __ffs(pm) - 1;
                pm &= pm - 1u;
                const double pe = shfl_f64(e, p);
                const int pi = __shfl_sync(0xffffffffu, cidx, p);
                if (lex_less(pe, pi, tau, tau_idx)) {
                  if (have_prev && __any_sync(0xffffffffu, lidx == pi)) continue;     // already there (warm start)
                  // sorted insert: entries not below the newcomer move one lane up, the last one drops out
                  const unsigned below = __ballot_sync(0xffffffffu, lex_less(le, lidx, pe, pi));
                  const int pos = __popc(below);
                  const double ue = shfl_f64(le, (lane > 0) ? lane - 1 : 0);
                  const int ui = __shfl_sync(0xffffffffu, lidx, (lane > 0) ? lane - 1 : 0);
                  if (lane > pos) { le = ue; lidx = ui; }
                  else if (lane == pos) { le = pe; lidx = pi; }
                  tau = shfl_f64(le, 31);
                  tau_idx = __shfl_sync(0xffffffffu, lidx, 31);
                  if (!(tau < INF)) tau_idx = 0x7fffffff;      // padding entries lose against every real candidate
                  pm &= __ballot_sync(0xffffffffu, lex_less(e, cidx, tau, tau_idx));   // drop the ones now out of reach
                }
              }
            }
          }

          // ---------------- 3. basis states, free energies, Hamiltonian ----------------
          double st[N];
          uint64_t key = 0;
          int tc = 0;                                // total charge of this lane's state
#pragma unroll
          for (int j = 0; j < N; ++j) {
            // dot j sits at permuted position pm[8 + j]: its digit is read there
            const int sj = (lidx < 0) ? 0 : (int)fs[j] + (((lidx >> (2 * (N - 1 - pm[8 + j]))) & 3) - 1);
            st[j] = (double)sj;
            tc += sj;
            key |= (uint64_t)((unsigned)sj & 0xffu) << (8 * j);
          }
          double Fm = 0.0;
          {
            double zz[N];
#pragma unroll
            for (int j = 0; j < N; ++j) zz[j] = st[j] - gs[j];
#pragma unroll
            for (int i = 0; i < N; ++i) {
              double s = 0.0;
#pragma unroll
              for (int j = 0; j < N; ++j) s = fma(C[i * N + j], zz[j], s);
              Fm = fma(zz[i], s, Fm);
            }
            if (vc_on) Fm /= ts[7];
          }
          // Hopping conserves the total charge, so H is block diagonal once the basis is ordered by total charge: the
          // 32 kept states typically fall into 5-6 sectors of <= 10-16 states.  Sort the lanes by (total charge, lane)
          // -- the spectrum and the weights |psi_m|^2 do not depend on the order of the basis -- and run every dense
          // step below on all sectors AT ONCE, each in its own lane segment [s0, s1]: reductions are segmented, the
          // inner loops run over the sector's columns only, and the number of Householder steps is the largest sector
          // size minus two instead of 30.
          int s0, s1, maxlen;
          {
            const unsigned same = __match_any_sync(0xffffffffu, tc);
            int rank = __popc(same & ((1u << lane) - 1u));
            unsigned rem = 0xffffffffu;
            while (rem) {
              const int leader = __ffs(rem) - 1;
              const int v = __shfl_sync(0xffffffffu, tc, leader);
              const unsigned grp = __shfl_sync(0xffffffffu, same, leader);
              if (v < tc) rank += __popc(grp);
              rem &= ~grp;
            }
            int* perm = reinterpret_cast<int*>(vq);
            perm[rank] = lane;
            __syncwarp();
            const int src = perm[lane];
            __syncwarp();
            key = shfl_u64(key, src);
            Fm = shfl_f64(Fm, src);
            tc = __shfl_sync(0xffffffffu, tc, src);
            prev_key = __shfl_sync(0xffffffffu, (int)(lidx < 0), src) ? ~0ULL : key;     // warm start of the next pixel
            have_prev = true;
#pragma unroll
            for (int j = 0; j < N; ++j) st[j] = (double)(int)(signed char)(unsigned char)(key >> (8 * j));
            const unsigned seg = __match_any_sync(0xffffffffu, tc);
            s0 = __ffs(seg) - 1;
            s1 = 31 - __clz(seg);
            maxlen = __reduce_max_sync(0xffffffffu, s1 - s0 + 1);
          }
          // Row `lane` of H, columns of its own sector only.  Two states are connected by a hop iff they differ in
          // exactly two ADJACENT dots, by (-1, +1) or (+1, -1): test on the XOR of the packed states first (cheap
          // reject), then compare the byte pair.
#pragma unroll 1
          for (int u = 0; u < maxlen; ++u) {
            const int j = min(s0 + u, 31);
            const uint64_t kj = shfl_u64(key, j);
            double val = (j == lane) ? Fm : 0.0;
            const uint64_t Hm = 0x8080808080808080ULL;
            const uint64_t x = kj ^ key;
            const uint64_t nz = (((x & ~Hm) + ~Hm) | x) & Hm;
            if (__popcll(nz) == 2 && (nz & (nz >> 8))) {
              const int p0 = (__ffsll((long long)nz) - 1) >> 3;
              const unsigned pa = (unsigned)(key >> (8 * p0)) & 0xffffu, pb = (unsigned)(kj >> (8 * p0)) & 0xffffu;
              const unsigned a0 = pa & 0xffu, a1 = pa >> 8;
              if (pb == pa + 0xffu) val = -ts[p0] * (sq_tab[a0] * sq_tab[a1 + 1]);        // p0 -> p0+1
              else if (pb + 0xffu == pa) val = -ts[p0] * (sq_tab[a1] * sq_tab[a0 + 1]);   // p0+1 -> p0
            }
            if (s0 + u <= s1) H[lane * QD_T_HS + j] = val;
          }
          __syncwarp();

          // ---------------- 4. ground eigenvector ----------------
          // Householder tridiagonalisation of every sector at once: step t works on column k = s0 + t of each sector
          // that still has at least two rows below it.
          const bool wide = maxlen > 16;
          for (int t = 0; t + 2 < maxlen; ++t) {
            const int k = s0 + t;
            const bool act = k + 2 <= s1;
            const double x = (act && lane > k) ? H[lane * QD_T_HS + k] : 0.0;
            const double xk1 = shfl_f64(x, min(k + 1, 31));
            const double sig = seg_sum((lane > k + 1) ? x * x : 0.0, lane, s0, s1, wide);
            const bool refl = act && sig != 0.0;
            double v = 0.0, alpha = xk1;
            if (refl) {
              const double norm2 = sig + xk1 * xk1;
              alpha = (xk1 > 0.0) ? -sqrt(norm2) : sqrt(norm2);
              v = x;
              if (lane == k + 1) v -= alpha;
              v *= rsqrt(2.0 * (norm2 - alpha * xk1));
            }
            vq[2 * lane] = v;
            __syncwarp();
            double p = 0.0;
            if (refl && lane > k) {
              double p0 = 0.0, p1 = 0.0;
              const double* __restrict__ hrow = H + lane * QD_T_HS;
              int j = k + 1;
              for (; j + 1 <= s1; j += 2) {
                p0 = fma(hrow[j], vq[2 * j], p0);
                p1 = fma(hrow[j + 1], vq[2 * j + 2], p1);
              }
              if (j <= s1) p0 = fma(hrow[j], vq[2 * j], p0);
              p = p0 + p1;
            }
            const double K = seg_sum(v * p, lane, s0, s1, wide);
            const double q = p - K * v;
            vq[2 * lane + 1] = q;
            __syncwarp();
            if (act && lane > k) {
              double* __restrict__ hrow = H + lane * QD_T_HS;
              if (refl) {
                const double v2 = -2.0 * v, q2 = -2.0 * q;
                for (int j = k + 1; j <= s1; ++j) {
                  const double2 o = *reinterpret_cast<const double2*>(vq + 2 * j);     // (v_j, q_j)
                  hrow[j] = fma(v2, o.y, fma(q2, o.x, hrow[j]));
                }
              }
              hrow[k] = v;                                     // the dead column keeps the reflector (0: none)
            }
            if (act && lane == s0) ee[k] = alpha;
            __syncwarp();
          }
          dd[lane] = H[lane * QD_T_HS + lane];
          // last coupling inside each sector, and none across sectors
          if (lane == s1) ee[lane] = 0.0;
          else if (lane == s1 - 1) ee[lane] = H[s1 * QD_T_HS + lane];
          __syncwarp();
          double lo, hi;
          {
            const double rad = ((lane > 0) ? fabs(ee[lane - 1]) : 0.0) + ((lane < 31) ? fabs(ee[lane]) : 0.0);
            lo = warp_min(dd[lane] - rad);
            hi = warp_max(dd[lane] + rad);
          }
          // Lowest eigenvalue by 32-way multisection.  x < lambda_0  <=>  T - x I positive definite  <=>  every leading
          // principal minor p_i(x) > 0 (Sylvester); the minors obey p_{i+1} = (d_i - x) p_i - e_{i-1}^2 p_{i-1}.  The
          // tridiagonal is mapped onto [0, 1] first (Gershgorin interval), so |d - x| <= 1, e^2 <= 1 and the minors
          // cannot overflow; a positive rescale every 8 steps guards the underflow side.
          const double lo0 = lo, wid = fmax(hi - lo, 1e-300), iw = 1.0 / wid;
          qi[lane] = (dd[lane] - lo0) * iw;
          e2[lane] = (ee[lane] * iw) * (ee[lane] * iw);
          __syncwarp();
          lo = 0.0;
          hi = 1.0;
          for (int round = 0; round < 6; ++round) {
            const double x = fma((double)(lane + 1) * (1.0 / 33.0), hi - lo, lo);
            double pp = 1.0, pc = qi[0] - x;
            bool below = !(pc > 0.0);                  // some eigenvalue lies at or below x
#pragma unroll
            for (int i0 = 1; i0 < 32; i0 += 8) {
#pragma unroll
              for (int i = i0; i < i0 + 8 && i < 32; ++i) {
                const double pn = fma(qi[i] - x, pc, -e2[i - 1] * pp);
                below |= !(pn > 0.0);
                pp = pc;
                pc = pn;
              }
              if (pc < 1e-150) { pc *= 1e150; pp *= 1e150; }      // (irrelevant once `below` is set)
            }
            const unsigned mm = __ballot_sync(0xffffffffu, below);
            const int j = mm ? __ffs(mm) - 1 : 32;
            const double xl = shfl_f64(x, (j > 0) ? j - 1 : 0);
            const double xh = shfl_f64(x, (j < 32) ? j : 31);
            if (j > 0) lo = xl;
            if (j < 32) hi = xh;
          }
          lo = fma(lo, wid, lo0);
          __syncwarp();
          const double mu = lo;
          // LDL^T of T - mu I and the inverse-iteration solves, every sector by its own leader lane (the sectors are
          // decoupled: ee[s1] = 0), so the serial chains are one sector long instead of 32.
          if (lane == s0) {
            double q = dd[s0] - mu;
            for (int i = s0; i < s1; ++i) {
              if (!(q > 0.0)) q = 1e-300;
              const double iq = 1.0 / q;
              qi[i] = iq;
              const double l = ee[i] * iq;
              ll[i] = l;
              q = (dd[i + 1] - mu) - l * ee[i];
            }
            if (!(q > 0.0)) q = 1e-300;
            qi[s1] = 1.0 / q;
          }
          yy[lane] = 1.0 + (double)lane * (1.0 / 64.0);
          __syncwarp();
          for (int it = 0; it < 3; ++it) {
            if (lane == s0) {
              double zprev = yy[s0];
              for (int i = s0 + 1; i <= s1; ++i) { zprev = yy[i] - ll[i - 1] * zprev; yy[i] = zprev; }
              double ynext = yy[s1] * qi[s1];
              yy[s1] = ynext;
              for (int i = s1 - 1; i >= s0; --i) { ynext = yy[i] * qi[i] - ll[i] * ynext; yy[i] = ynext; }
            }
            __syncwarp();
            double yv = yy[lane];
            // scale first (the unnormalised iterate can overflow when mu is within rounding of lambda_0)
            const double ymax = warp_max(fabs(yv));
            yv *= 1.0 / ymax;
            const double nrm = warp_sum(yv * yv);
            yy[lane] = yv * rsqrt(nrm);
            __syncwarp();
          }
          double psi = yy[lane];
          for (int t = maxlen - 3; t >= 0; --t) {
            const int k = s0 + t;
            const double v = (k + 2 <= s1 && lane > k) ? H[lane * QD_T_HS + k] : 0.0;
            const double dot = seg_sum(v * psi, lane, s0, s1, wide);
            psi = fma(-2.0 * dot, v, psi);
          }
          {
            const double w2 = psi * psi;
#pragma unroll
            for (int j = 0; j < N; ++j) nbar[j] = warp_sum(w2 * st[j]);
          }

        } else {
#pragma unroll
          for (int j = 0; j < N; ++j) nbar[j] = 0.0;
        }
        // ---------------- <n> -> scratch ----------------
        if (lane == 0) {
#pragma unroll
          for (int j = 0; j < N; ++j) nb[j] = nbar[j];
        }
        __syncwarp();
        if (lane < N) a.nbar[(pix0 + pix) * N + lane] = nb[lane];
        __syncwarp();
        }
      }
    }
    __syncwarp();
  }
}


// =====================================================================================================================
// Split pipeline (default): the same per-pixel computation as qd_tunnel_gs_kernel in THREE kernels, so that none of them
// carries the union of the others' registers and shared memory (qd_tunnel_gs_kernel: 168 registers + 16.9 KB per warp
// -> 12 warps per SM, 38 % of the issue slots used; it stays as the QDSIM_TUNNEL_MONO=1 reference):
//   R  qd_tunnel_relax_kernel   one THREAD per pixel: potentials, the reference's closed form / 50 projected-gradient
//                               steps (an 8 x 8 mat-vec per step in registers), floor -> 8 bytes per pixel
//   S  qd_tunnel_select_kernel  one warp per pixel: block-bounded, warm-started streaming top-32 -> 32 packed states
//   E  qd_tunnel_eigen_kernel   one warp per pixel: Hamiltonian in total-charge sectors, ground eigenvector, <n>
// Scratch between them: 8 + 256 bytes per pixel of the current chunk of scans (the launcher cuts large batches).
// =====================================================================================================================
// Slots of the three kernels (qd_kernels.cuh: slot layouts).  Each stages the record's gs_doubles prefix only.
struct RelaxSlot {    // one per CTA
  size_t rec_bytes;   // [gs_doubles] the record prefix; the offsets below count from its end
  int scan;           // qd_scan, the descriptor
  int bytes;          // (not rounded)
};
__host__ __device__ constexpr RelaxSlot qd_tunnel_relax_slot(const qd_layout& L) {
  RelaxSlot S{};
  S.rec_bytes = (size_t)L.gs_doubles * 8;
  S.scan = 0;
  S.bytes = (int)(S.rec_bytes + sizeof(qd_scan));
  return S;
}

struct SelectSlot {
  size_t rec_bytes;   // [gs_doubles] the record prefix (TMA destination); the offsets below count from its end
  int scan;           // qd_scan, the descriptor (TMA destination)
  int vv;             // [16]
  int gs, ns, fs, hs; // [8] each
  int Mi;             // [9] inverse of rows / columns 1..3 of the low 4 x 4 block of Cp (NLO = 4): 16 doubles reserved
  int Cp;             // [64] Cinv with rows / columns permuted so that the stiffest dots come first
  int Sp;             // [16] Schur complement of the permuted high block
  int Ql;             // [256] y^T Cp_ll y over the low digit combinations
  int pm;             // int[16] pm[j]: dot at permuted position j, pm[8 + d]: position of dot d (16 doubles reserved)
  int bar;            // mbarrier of the two copies (16 bytes)
  int bytes;
};
__host__ __device__ constexpr SelectSlot qd_tunnel_select_slot(const qd_layout& L) {
  SelectSlot S{};
  S.rec_bytes = (size_t)L.gs_doubles * 8;
  int o = 0;
  S.scan = o;     o += (int)sizeof(qd_scan);
  S.vv = o;       o += 16 * 8;
  S.gs = o;       o += 8 * 8;
  S.ns = o;       o += 8 * 8;
  S.fs = o;       o += 8 * 8;
  S.hs = o;       o += 8 * 8;
  S.Mi = o;       o += 16 * 8;
  S.Cp = o;       o += 64 * 8;
  S.Sp = o;       o += 16 * 8;
  S.Ql = o;       o += 256 * 8;
  S.pm = o;       o += 16 * 8;
  S.bar = o;      o += 16;
  S.bytes = qd_slot_round(S.rec_bytes + o);
  return S;
}

struct EigenSlot {
  size_t rec_bytes;   // [gs_doubles] the record prefix (TMA destination); the offsets below count from its end
  int scan;           // qd_scan, the descriptor (TMA destination)
  int H;              // [32][QD_T_HS] the Hamiltonian
  int dd, ee, e2, qi, ll, yy;   // [32] each
  int vq;             // [64] interleaved (v_j, q_j) of the current Householder step, read as double2; + 8 spare
  int vv;             // [16]
  int gs, ts;         // [8] each
  int bar;            // mbarrier of the two copies (16 bytes)
  int bytes;
};
__host__ __device__ constexpr EigenSlot qd_tunnel_eigen_slot(const qd_layout& L) {
  EigenSlot S{};
  S.rec_bytes = (size_t)L.gs_doubles * 8;
  int o = 0;
  S.scan = o;     o += (int)sizeof(qd_scan);
  S.H = o;        o += 32 * QD_T_HS * 8;
  S.dd = o;       o += 32 * 8;
  S.ee = o;       o += 32 * 8;
  S.e2 = o;       o += 32 * 8;
  S.qi = o;       o += 32 * 8;
  S.ll = o;       o += 32 * 8;
  S.yy = o;       o += 32 * 8;
  S.vq = o;       o += 72 * 8;
  S.vv = o;       o += 16 * 8;
  S.gs = o;       o += 8 * 8;
  S.ts = o;       o += 8 * 8;
  S.bar = o;      o += 16;
  S.bytes = qd_slot_round(S.rec_bytes + o);
  return S;
}

// ---- R: relaxation, one thread per pixel ------------------------------------------------------------------------------
template <int N>
__global__ void __launch_bounds__(128) qd_tunnel_relax_kernel(const KArgs a) {
  extern __shared__ __align__(128) unsigned char qd_smem[];
  const qd_layout& L = a.L;
  const int NV = L.n_volt;
  const RelaxSlot S = qd_tunnel_relax_slot(L);
  double* rec = reinterpret_cast<double*>(qd_smem);
  qd_scan* sc = reinterpret_cast<qd_scan*>(qd_smem + S.rec_bytes + S.scan);
  const double* __restrict__ C = rec + L.o_cinv;
  const long long total_items = (long long)a.n_scan * a.items_per_scan;
  for (long long item = blockIdx.x; item < total_items; item += gridDim.x) {
    const int scan_id = (int)(item / a.items_per_scan);
    const int part = (int)(item - (long long)scan_id * a.items_per_scan);
    const qd_scan* gscan = a.scans + scan_id;
    __syncthreads();
    {
      const double* src = a.records + (size_t)gscan->env_id * L.rec_doubles;
      for (int i = threadIdx.x; i < L.gs_doubles; i += blockDim.x) rec[i] = src[i];
      const double* ssrc = reinterpret_cast<const double*>(gscan);
      double* sdst = reinterpret_cast<double*>(sc);
      for (int i = threadIdx.x; i < (int)(sizeof(qd_scan) / 8); i += blockDim.x) sdst[i] = ssrc[i];
    }
    __syncthreads();
    const int nx = sc->nx, ny = sc->ny;
    const long long npix = (long long)nx * ny;
    const long long p_begin = (long long)part * a.rows_per_item;
    const long long p_end = min(npix, p_begin + (long long)a.rows_per_item);
    const double* par = rec + L.o_par;
    const bool replace = (a.flags & QD_FLAG_RADIAL) && sc->rad_mode == 2;
    if (replace) continue;
    const bool vc_on = par[QD_PAR_VC_ALPHA] != 0.0 || par[QD_PAR_VC_BETA] != 0.0;
    for (long long pix = p_begin + threadIdx.x; pix < p_end; pix += blockDim.x) {
      const int iy = (int)(pix / nx), ix = (int)(pix - (long long)iy * nx);
      double g[N];
#pragma unroll
      for (int j = 0; j < N; ++j) g[j] = 0.0;
      double vabs = 0.0, v2 = 0.0;
      for (int k = 0; k < NV; ++k) {
        const double vk = (a.points == nullptr) ? fma((double)iy, sc->dy[k], fma((double)ix, sc->dx[k], sc->v0[k]))
                                                : a.points[(size_t)pix * NV + k];
        vabs += fabs(vk);
        v2 = fma(vk, vk, v2);
#pragma unroll
        for (int j = 0; j < N; ++j) g[j] = fma(rec[L.o_a + j * NV + k], vk, g[j]);
      }
      double lr = 0.1;
      double s_c = 1.0;
      if (vc_on) {
        double sb;
        vc_scales(par, vabs, v2, NV, s_c, sb);
#pragma unroll
        for (int j = 0; j < N; ++j) g[j] *= sb;
        lr = 0.1 / s_c;
      }
      // the per-pixel quantities the select and eigen kernels need again (the same operations in the same order as their own
      // former code): potentials, tunnel couplings t_d = |tc_base exp(-alpha_d vb_eff_d)|, scale of cdd
      if (a.tpot) {
        double* __restrict__ tp = a.tpot + ((size_t)scan_id * a.tstride + pix) * 16;
#pragma unroll
        for (int j = 0; j < N; ++j) tp[j] = g[j];
        const int G = L.n_gate;
        for (int d = 0; d < N - 1; ++d) {
          double t = par[QD_PAR_TC_BASE];
          if (NV > G) {
            double vb = (a.points == nullptr) ? fma((double)iy, sc->dy[G + d], fma((double)ix, sc->dx[G + d], sc->v0[G + d]))
                                              : a.points[(size_t)pix * NV + G + d];
            for (int k = 0; k < G; ++k) {
              const double vk = (a.points == nullptr) ? fma((double)iy, sc->dy[k], fma((double)ix, sc->dx[k], sc->v0[k]))
                                                      : a.points[(size_t)pix * NV + k];
              vb = fma(rec[L.o_cbg + d * G + k], vk, vb);
            }
            t *= exp(-rec[L.o_alpha + d] * vb);
          }
          tp[8 + d] = fabs(t);
        }
        tp[15] = s_c;
      }
      bool neg = false;
      double n[N];
#pragma unroll
      for (int j = 0; j < N; ++j) { neg |= g[j] < 0.0; n[j] = g[j]; }
      if (neg) {                                            // charge_states.py:64-87
        double cg[N];
#pragma unroll
        for (int i = 0; i < N; ++i) {
          double s0 = 0.0;
#pragma unroll
          for (int k = 0; k < N; ++k) s0 = fma(C[i * N + k], g[k], s0);
          cg[i] = s0;
          n[i] = fmax(g[i], 0.0);
        }
#pragma unroll 1
        for (int it = 0; it < 50; ++it) {
          double nn[N];
#pragma unroll
          for (int i = 0; i < N; ++i) {
            double s0 = 0.0;
#pragma unroll
            for (int k = 0; k < N; ++k) s0 = fma(C[i * N + k], n[k], s0);
            nn[i] = fmax(n[i] - lr * (s0 - cg[i]), 0.0);
          }
#pragma unroll
          for (int i = 0; i < N; ++i) n[i] = nn[i];
        }
      }
      uint64_t fk = 0;
      bool big = false;
#pragma unroll
      for (int j = 0; j < N; ++j) {
        const double fj = floor(fmax(n[j], 0.0));
        big |= !(fj < 250.0);
        fk |= (uint64_t)((unsigned)__double2int_rz(fmin(fj, 255.0)) & 0xffu) << (8 * j);
      }
      if (big && a.status) *reinterpret_cast<volatile unsigned*>(a.status) = QD_STATUS_OCC_OVERFLOW;
      *reinterpret_cast<uint64_t*>(a.tfloor + ((size_t)scan_id * a.tstride + pix) * 8) = fk;
    }
  }
}

// ---- S: streaming top-32 selection, one warp per pixel ---------------------------------------------------------------------
template <int N>
__global__ void __launch_bounds__(128, 4) qd_tunnel_select_kernel(const KArgs a) {
  constexpr int NLO = N < 4 ? N : 4;
  constexpr int NHI = N - NLO;
  constexpr int NB_LO = 1 << (2 * NLO);            // low candidates per block
  constexpr int NB_HI = 1 << (2 * NHI);            // blocks
  constexpr int LO_IT = NB_LO >= 32 ? NB_LO / 32 : 1;
  constexpr int HI_IT = NB_HI >= 32 ? NB_HI / 32 : 1;

  extern __shared__ __align__(128) unsigned char qd_smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const qd_layout& L = a.L;
  const int NV = L.n_volt;

  unsigned char* slot = qd_smem + (size_t)warp * a.slot_bytes;
  const SelectSlot S = qd_tunnel_select_slot(L);
  unsigned char* tail = slot + S.rec_bytes;
  double* rec = reinterpret_cast<double*>(slot);
  qd_scan* sc = reinterpret_cast<qd_scan*>(tail + S.scan);
  double* vv = reinterpret_cast<double*>(tail + S.vv);
  double* gs = reinterpret_cast<double*>(tail + S.gs);
  double* ns = reinterpret_cast<double*>(tail + S.ns);
  double* fs = reinterpret_cast<double*>(tail + S.fs);
  double* hs = reinterpret_cast<double*>(tail + S.hs);
  double* mi = reinterpret_cast<double*>(tail + S.Mi);
  double* Cp = reinterpret_cast<double*>(tail + S.Cp);
  double* Sp = reinterpret_cast<double*>(tail + S.Sp);
  double* Ql = reinterpret_cast<double*>(tail + S.Ql);
  int* pm = reinterpret_cast<int*>(tail + S.pm);
  uint64_t* bar = reinterpret_cast<uint64_t*>(tail + S.bar);

  const double* __restrict__ C = rec + L.o_cinv;
  const double INF = __longlong_as_double(0x7ff0000000000000LL);

  if (lane == 0) mbar_init(bar, 1);
  __syncwarp();
  uint32_t phase = 0;
  const uint32_t rec_bytes = (uint32_t)L.gs_doubles * 8u;

  const long long total_items = (long long)a.n_scan * a.items_per_scan;
  for (long long item = (long long)blockIdx.x * warps_per_cta + warp; item < total_items;
       item += (long long)gridDim.x * warps_per_cta) {
    const int scan_id = (int)(item / a.items_per_scan);
    const int part = (int)(item - (long long)scan_id * a.items_per_scan);
    const qd_scan* gscan = a.scans + scan_id;
    if (a.fixup) {
      // fix-up mode: only the pixels qd_tunnel_select2_kernel marked (first key = QD_S2_MARK; item-level mark = a NaN in the
      // <n> scratch of the item's first pixel) are done here, each from a cold start
      // (this launch uses shorter items than the marking kernel, so that an item whose pixels are all marked is shared by
      // several warps)
      const long long pb = (long long)part * a.rows_per_item;
      if (pb >= (long long)gscan->nx * gscan->ny) continue;
      const double fl = a.nbar[(gscan->pix_offset + (pb / a.mark_ppi) * a.mark_ppi) * N];
      if (fl == fl) continue;
    }
    stage_item(a, gscan, rec_bytes, rec, sc, bar, phase, lane);

    const int nx = sc->nx, ny = sc->ny;
    const long long npix = (long long)nx * ny;
    const long long p_begin = (long long)part * a.rows_per_item;            // rows_per_item = pixels per item here
    const long long p_end = min(npix, p_begin + (long long)a.rows_per_item);
    if (p_begin >= npix) { __syncwarp(); continue; }
    const double* par = rec + L.o_par;
    const bool replace = (a.flags & QD_FLAG_RADIAL) && sc->rad_mode == 2;
    if (replace) { __syncwarp(); continue; }
    const bool vc_on = par[QD_PAR_VC_ALPHA] != 0.0 || par[QD_PAR_VC_BETA] != 0.0;

    // ---- per-item split of the dots into a high and a low half (see qd_tunnel_gs_kernel) ----
    {
      const long long pf = p_begin;
      const int fy = (int)(pf / nx), fx = (int)(pf - (long long)fy * nx);
      if (lane < NV)
        vv[lane] = (a.points == nullptr) ? fma((double)fy, sc->dy[lane], fma((double)fx, sc->dx[lane], sc->v0[lane]))
                                         : a.points[(size_t)pf * NV + lane];
      __syncwarp();
      if (lane < N) {
        double acc = 0.0;
        for (int k = 0; k < NV; ++k) acc = fma(rec[L.o_a + lane * NV + k], vv[k], acc);
        gs[lane] = acc;
      }
      __syncwarp();
      if (lane == 0) {
        int ord[N];
        for (int j = 0; j < N; ++j) ord[j] = j;
        for (int i = 1; i < N; ++i) {                      // insertion sort, ascending potential (most negative first)
          const int o = ord[i];
          int j = i - 1;
          while (j >= 0 && gs[ord[j]] > gs[o]) { ord[j + 1] = ord[j]; --j; }
          ord[j + 1] = o;
        }
        for (int j = 0; j < N; ++j) { pm[j] = ord[j]; pm[8 + ord[j]] = j; }
      }
      __syncwarp();
      for (int e = lane; e < N * N; e += 32) Cp[e] = C[pm[e / N] * N + pm[e % N]];
      __syncwarp();
      if (lane == 0) {
        double m[4][8];
        for (int i = 0; i < NLO; ++i)
          for (int j = 0; j < NLO; ++j) { m[i][j] = Cp[(NHI + i) * N + NHI + j]; m[i][NLO + j] = (i == j) ? 1.0 : 0.0; }
        for (int k = 0; k < NLO; ++k) {
          const double inv = 1.0 / m[k][k];
          for (int j = 0; j < 2 * NLO; ++j) m[k][j] *= inv;
          for (int i = 0; i < NLO; ++i) {
            if (i == k) continue;
            const double fac = m[i][k];
            for (int j = 0; j < 2 * NLO; ++j) m[i][j] -= fac * m[k][j];
          }
        }
        for (int i = 0; i < NHI; ++i)
          for (int j = 0; j < NHI; ++j) {
            double acc = Cp[i * N + j];
            for (int p = 0; p < NLO; ++p)
              for (int q = 0; q < NLO; ++q) acc -= Cp[i * N + NHI + p] * m[p][NLO + q] * Cp[(NHI + q) * N + j];
            Sp[i * NHI + j] = acc;
          }
      }
      for (int idx = lane; idx < NB_LO; idx += 32) {
        double acc = 0.0;
        for (int i = 0; i < NLO; ++i)
          for (int j = 0; j < NLO; ++j)
            acc += (double)(((idx >> (2 * (NLO - 1 - i))) & 3) - 1) * Cp[(NHI + i) * N + NHI + j] *
                   (double)(((idx >> (2 * (NLO - 1 - j))) & 3) - 1);
        Ql[idx] = acc;
      }
      if constexpr (NLO == 4) {
        // Second-level bound (leading low digit fixed, the other three continuous): with the low block L = Cp_ll split as
        // [[L00, l^T], [l, L']],  min_y' E = alpha + beta y0 + gamma y0^2,  gamma = L00 - l^T L'^-1 l  (per item),
        // alpha = base - c'^T L'^-1 c',  beta = 2 (c0 - c'^T L'^-1 l)  (per block).  Stored: L'^-1 [9], L'^-1 l [3], gamma.
        if (lane == 0) {
          double Lm[4][4];
          for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) Lm[i][j] = Cp[(NHI + i) * N + NHI + j];
          const double a11 = Lm[1][1], a12 = Lm[1][2], a13 = Lm[1][3], a22 = Lm[2][2], a23 = Lm[2][3], a33 = Lm[3][3];
          const double c11 = a22 * a33 - a23 * a23, c12 = a13 * a23 - a12 * a33, c13 = a12 * a23 - a13 * a22;
          const double c22 = a11 * a33 - a13 * a13, c23 = a12 * a13 - a11 * a23, c33 = a11 * a22 - a12 * a12;
          const double idet = 1.0 / (a11 * c11 + a12 * c12 + a13 * c13);
          double* Mi = mi;
          Mi[0] = c11 * idet; Mi[1] = c12 * idet; Mi[2] = c13 * idet;
          Mi[3] = c12 * idet; Mi[4] = c22 * idet; Mi[5] = c23 * idet;
          Mi[6] = c13 * idet; Mi[7] = c23 * idet; Mi[8] = c33 * idet;
          const double l1 = Lm[1][0], l2 = Lm[2][0], l3 = Lm[3][0];
          Mi[9] = Mi[0] * l1 + Mi[1] * l2 + Mi[2] * l3;
          Mi[10] = Mi[3] * l1 + Mi[4] * l2 + Mi[5] * l3;
          Mi[11] = Mi[6] * l1 + Mi[7] * l2 + Mi[8] * l3;
          Mi[12] = Lm[0][0] - (l1 * Mi[9] + l2 * Mi[10] + l3 * Mi[11]);
        }
      }
      __syncwarp();
    }

    uint64_t prev_key = ~0ULL;       // this lane's basis state at the previous pixel of the item (~0: none / padding)
    bool have_prev = false;
    for (long long pix = p_begin; pix < p_end; ++pix) {
      const int iy = (int)(pix / nx), ix = (int)(pix - (long long)iy * nx);
      const size_t tslot = (size_t)scan_id * a.tstride + pix;
      if (a.fixup && a.tkeys[tslot * 32] != 0xfffffffffffffffeULL) { have_prev = false; continue; }
      // ---------------- potentials, floor (from the relax kernel), r = f - g, h = C r ----------------
      if (lane < NV) {
        vv[lane] = (a.points == nullptr) ? fma((double)iy, sc->dy[lane], fma((double)ix, sc->dx[lane], sc->v0[lane]))
                                         : a.points[(size_t)pix * NV + lane];
      }
      const uint64_t fk = *reinterpret_cast<const uint64_t*>(a.tfloor + tslot * 8);
      __syncwarp();
      if (lane < N) {
        double acc = 0.0;
        const double* arow = rec + L.o_a + lane * NV;
        for (int k = 0; k < NV; ++k) acc = fma(arow[k], vv[k], acc);
        if (vc_on) {
          double vabs = 0.0;
          for (int k = 0; k < NV; ++k) vabs += fabs(vv[k]);
          acc *= fma(par[QD_PAR_VC_BETA], vabs / (double)NV, 1.0);          // (s_g is the same in every model)
        }
        gs[lane] = acc;
        const double fj = (double)(unsigned)((fk >> (8 * lane)) & 0xffu);
        fs[lane] = fj;
        ns[lane] = fj - acc;                       // r = f - g
      }
      __syncwarp();
      if (lane < N) {                              // h = C r
        double s0 = 0.0;
        for (int k = 0; k < N; ++k) s0 = fma(C[lane * N + k], ns[k], s0);
        hs[lane] = s0;
      }
      __syncwarp();
      double f[N], r[N], h[N];
#pragma unroll
      for (int j = 0; j < N; ++j) { const int d = pm[j]; f[j] = fs[d]; r[j] = ns[d]; h[j] = hs[d]; }   // permuted order
      double E0 = 0.0;
#pragma unroll
      for (int j = 0; j < N; ++j) E0 = fma(r[j], h[j], E0);

      // ---------------- streaming top-32 over the 4^N candidates (see qd_tunnel_gs_kernel) ----------------
      double le = INF;
      int lidx = -1;                             // -1: the reference's zero-state padding entry
      double tau = INF;
      int tau_idx = 0x7fffffff;
      if (have_prev) {
        bool okp = prev_key != ~0ULL;
        int idx = 0;
#pragma unroll
        for (int j = 0; j < N; ++j) {
          const int dg = (int)(signed char)(unsigned char)(prev_key >> (8 * j)) - (int)fs[j] + 1;
          okp = okp && dg >= 0 && dg <= 3;
          idx |= (dg & 3) << (2 * (N - 1 - pm[8 + j]));
        }
        if (okp) {
          double base;
          double c[NLO];
          const int b = idx & (NB_LO - 1);
          tunnel_block_constants<N, NHI, NLO>(idx >> (2 * NLO), E0, h, Cp, base, c);
          le = tunnel_iter_part<NLO>(tunnel_lane_part<NLO>(base, c, b & 31) + Ql[b], c, b >> 5);
          lidx = idx;
        }
#pragma unroll
        for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
          for (int j = k >> 1; j > 0; j >>= 1) {
            const double oe = shfl_f64(le, lane ^ j);
            const int oi = __shfl_xor_sync(0xffffffffu, lidx, j);
            const bool keep_min = ((lane & j) == 0) == ((lane & k) == 0);
            const bool take = keep_min ? lex_less(oe, oi, le, lidx) : lex_less(le, lidx, oe, oi);
            if (take) { le = oe; lidx = oi; }
          }
        }
        tau = shfl_f64(le, 31);
        tau_idx = __shfl_sync(0xffffffffu, lidx, 31);
        if (!(tau < INF)) tau_idx = 0x7fffffff;
      }
      unsigned lo_valid = 0;
#pragma unroll
      for (int i = 0; i < LO_IT; ++i) {
        const int b = i * 32 + lane;
        bool ok = b < NB_LO;
#pragma unroll
        for (int k = 0; k < NLO; ++k) {
          const int dg = (b >> (2 * (NLO - 1 - k))) & 3;
          ok = ok && !(dg == 0 && f[NHI + k] <= 0.0);
        }
        lo_valid |= ok ? (1u << i) : 0u;
      }
      double lb[HI_IT];
#pragma unroll
      for (int i = 0; i < HI_IT; ++i) {
        const int blk = i * 32 + lane;
        double v = INF;
        if (blk < NB_HI) {
          bool ok = true;
          double zh[NHI > 0 ? NHI : 1];
#pragma unroll
          for (int j = 0; j < NHI; ++j) {
            const int dg = (blk >> (2 * (NHI - 1 - j))) & 3;
            ok = ok && !(dg == 0 && f[j] <= 0.0);
            zh[j] = r[j] + (double)(dg - 1);
          }
          if (ok) {
            v = 0.0;
#pragma unroll
            for (int p = 0; p < NHI; ++p) {
              double s0 = 0.0;
#pragma unroll
              for (int q = 0; q < NHI; ++q) s0 = fma(Sp[p * NHI + q], zh[q], s0);
              v = fma(zh[p], s0, v);
            }
          }
        }
        lb[i] = v;
      }
      while (true) {
        int mb;
        if (have_prev && tau < INF && (a.topt & 2)) {
          // Warm-started list: tau is (nearly) final from the start, so the ORDER of the visits hardly matters -- take any
          // block whose bound is not above tau (one ballot instead of a 5-step (bound, index) reduction).  The set of
          // candidates that end up in the list does not depend on the order; the walk ends when no such block is left.
          int mine = -1;
#pragma unroll
          for (int i = HI_IT - 1; i >= 0; --i)
            if (lb[i] - 1e-12 * (fabs(lb[i]) + 1.0) <= tau) mine = i * 32 + lane;       // (inf - inf = nan: not live)
          const unsigned live = __ballot_sync(0xffffffffu, mine >= 0);
          if (!live) break;
          mb = __shfl_sync(0xffffffffu, mine, __ffs(live) - 1);
        } else {
          // cold start (first pixel of an item): best-first, so that tau tightens as early as possible
          double m = INF;
          mb = 0x7fffffff;
#pragma unroll
          for (int i = 0; i < HI_IT; ++i)
            if (lb[i] < m) { m = lb[i]; mb = i * 32 + lane; }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            const double om = shfl_f64(m, lane ^ o);
            const int ob = __shfl_xor_sync(0xffffffffu, mb, o);
            if (om < m || (om == m && ob < mb)) { m = om; mb = ob; }
          }
          if (!(m < INF)) break;
          if (m - 1e-12 * (fabs(m) + 1.0) > tau) break;      // every remaining candidate is above the 32nd best
        }
#pragma unroll
        for (int i = 0; i < HI_IT; ++i)
          if (mb == i * 32 + lane) lb[i] = INF;
        double base;
        double c[NLO];
        tunnel_block_constants<N, NHI, NLO>(mb, E0, h, Cp, base, c);
        const double base_lane = tunnel_lane_part<NLO>(base, c, lane);      // lane part, once per block
        double alpha_b = 0.0, beta_b = 0.0, gamma_b = 0.0;
        if constexpr (NLO == 4) {
          const double* __restrict__ Mi = mi;
          const double u0 = fma(Mi[0], c[1], fma(Mi[1], c[2], Mi[2] * c[3]));
          const double u1 = fma(Mi[3], c[1], fma(Mi[4], c[2], Mi[5] * c[3]));
          const double u2 = fma(Mi[6], c[1], fma(Mi[7], c[2], Mi[8] * c[3]));
          alpha_b = base - fma(c[1], u0, fma(c[2], u1, c[3] * u2));
          beta_b = 2.0 * (c[0] - fma(c[1], Mi[9], fma(c[2], Mi[10], c[3] * Mi[11])));
          gamma_b = Mi[12];
        }
        // every candidate of inner iteration i has the leading low digit i >> 1: the iteration is skipped when even the
        // continuous minimum over the other three low digits lies above the current 32nd-best energy (tau only falls)
        double bnd4[4] = {-INF, -INF, -INF, -INF};
        if (NLO == 4 && (a.topt & 1)) {
#pragma unroll
          for (int dg = 0; dg < 4; ++dg) {
            const double y0 = (double)(dg - 1);
            const double bnd = fma(y0, fma(gamma_b, y0, beta_b), alpha_b);
            bnd4[dg] = bnd - 1e-12 * (fabs(bnd) + 1.0);
          }
        }
#pragma unroll 1
        for (int ii = 0; ii < LO_IT; ++ii) {
          const int i = (LO_IT >= 4) ? ((ii + LO_IT / 4) & (LO_IT - 1)) : ii;
          if (NLO == 4) {
            const int dg = i >> 1;
            const double bnd = (dg == 0) ? bnd4[0] : (dg == 1) ? bnd4[1] : (dg == 2) ? bnd4[2] : bnd4[3];
            if (bnd > tau) continue;
          }
          const int b = i * 32 + lane;
          const bool ok = (lo_valid >> i) & 1u;
          double e = INF;
          if (ok) e = tunnel_iter_part<NLO>(base_lane + Ql[b], c, i);
          const int cidx = mb * NB_LO + b;
          // cheap superset of lex_less(e, cidx, tau, tau_idx); the exact (energy, index) test is made on every candidate taken
          unsigned pmk = __ballot_sync(0xffffffffu, ok && !(e > tau));
          while (pmk) {
            const int p = __ffs(pmk) - 1;
            pmk &= pmk - 1u;
            const double pe = shfl_f64(e, p);
            const int pi = __shfl_sync(0xffffffffu, cidx, p);
            if (lex_less(pe, pi, tau, tau_idx)) {
              if (have_prev && __any_sync(0xffffffffu, lidx == pi)) continue;     // already there (warm start)
              const unsigned below = __ballot_sync(0xffffffffu, lex_less(le, lidx, pe, pi));
              const int pos = __popc(below);
              const double ue = shfl_f64(le, (lane > 0) ? lane - 1 : 0);
              const int ui = __shfl_sync(0xffffffffu, lidx, (lane > 0) ? lane - 1 : 0);
              if (lane > pos) { le = ue; lidx = ui; }
              else if (lane == pos) { le = pe; lidx = pi; }
              tau = shfl_f64(le, 31);
              tau_idx = __shfl_sync(0xffffffffu, lidx, 31);
              if (!(tau < INF)) tau_idx = 0x7fffffff;      // padding entries lose against every real candidate
              pmk &= __ballot_sync(0xffffffffu, lex_less(e, cidx, tau, tau_idx));   // drop the ones now out of reach
            }
          }
        }
      }
      // ---------------- the 32 kept states, packed (padding entries = the reference's zero state) ----------------
      uint64_t key = 0;
#pragma unroll
      for (int j = 0; j < N; ++j) {
        const int sj = (lidx < 0) ? 0 : (int)fs[j] + (((lidx >> (2 * (N - 1 - pm[8 + j]))) & 3) - 1);
        key |= (uint64_t)((unsigned)sj & 0xffu) << (8 * j);
      }
      a.tkeys[tslot * 32 + lane] = key;
      prev_key = (lidx < 0) ? ~0ULL : key;
      have_prev = true;
      __syncwarp();
    }
    __syncwarp();
  }
}


#ifndef QD_TE_MIN_BLOCKS
#define QD_TE_MIN_BLOCKS 4
#endif
// ---- E: Hamiltonian in total-charge sectors, ground eigenvector, <n>; one warp per pixel -------------------------------
template <int N>
__global__ void __launch_bounds__(128, QD_TE_MIN_BLOCKS) qd_tunnel_eigen_kernel(const KArgs a) {
  constexpr int B = N - 1;
  extern __shared__ __align__(128) unsigned char qd_smem[];
  __shared__ double sq_tab[258];                   // sqrt(k), k = 0..257: hopping amplitudes sqrt(n_from (n_to + 1))
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const qd_layout& L = a.L;
  const int NV = L.n_volt, G = L.n_gate;
  const bool barriers = NV > G;
  for (int k = threadIdx.x; k < 258; k += blockDim.x) sq_tab[k] = sqrt((double)k);
  __syncthreads();

  unsigned char* slot = qd_smem + (size_t)warp * a.slot_bytes;
  const EigenSlot S = qd_tunnel_eigen_slot(L);
  unsigned char* tail = slot + S.rec_bytes;
  double* rec = reinterpret_cast<double*>(slot);
  qd_scan* sc = reinterpret_cast<qd_scan*>(tail + S.scan);
  double* H = reinterpret_cast<double*>(tail + S.H);
  double* dd = reinterpret_cast<double*>(tail + S.dd);
  double* ee = reinterpret_cast<double*>(tail + S.ee);
  double* e2 = reinterpret_cast<double*>(tail + S.e2);
  double* qi = reinterpret_cast<double*>(tail + S.qi);
  double* ll = reinterpret_cast<double*>(tail + S.ll);
  double* yy = reinterpret_cast<double*>(tail + S.yy);
  double* vq = reinterpret_cast<double*>(tail + S.vq);
  double* vv = reinterpret_cast<double*>(tail + S.vv);
  double* gs = reinterpret_cast<double*>(tail + S.gs);
  double* ts = reinterpret_cast<double*>(tail + S.ts);
  uint64_t* bar = reinterpret_cast<uint64_t*>(tail + S.bar);
  const double* __restrict__ C = rec + L.o_cinv;

  if (lane == 0) mbar_init(bar, 1);
  __syncwarp();
  uint32_t phase = 0;
  const uint32_t rec_bytes = (uint32_t)L.gs_doubles * 8u;

  const long long total_items = (long long)a.n_scan * a.items_per_scan;
  for (long long item = (long long)blockIdx.x * warps_per_cta + warp; item < total_items;
       item += (long long)gridDim.x * warps_per_cta) {
    const int scan_id = (int)(item / a.items_per_scan);
    const int part = (int)(item - (long long)scan_id * a.items_per_scan);
    const qd_scan* gscan = a.scans + scan_id;
    if (a.fixup) {
      // fix-up mode: qd_tunnel_eigen2_kernel left an item-level mark in the floor scratch of its item's first pixel; an
      // item whose parent item holds no marked pixel is skipped before anything is staged (shorter items than the marking
      // kernel's: see qd_tunnel_select_kernel)
      const long long pb = (long long)part * a.rows_per_item;
      if (pb >= (long long)gscan->nx * gscan->ny) continue;
      if (a.tfloor[((size_t)scan_id * a.tstride + (pb / a.mark_ppi) * a.mark_ppi) * 8] != 0xff) continue;
    }
    stage_item(a, gscan, rec_bytes, rec, sc, bar, phase, lane);

    const int nx = sc->nx, ny = sc->ny;
    const long long npix = (long long)nx * ny;
    const long long p_begin = (long long)part * a.rows_per_item;
    const long long p_end = min(npix, p_begin + (long long)a.rows_per_item);
    if (p_begin >= npix) { __syncwarp(); continue; }
    const double* par = rec + L.o_par;
    const bool replace = (a.flags & QD_FLAG_RADIAL) && sc->rad_mode == 2;
    const long long pix0 = sc->pix_offset;
    const bool vc_on = par[QD_PAR_VC_ALPHA] != 0.0 || par[QD_PAR_VC_BETA] != 0.0;

    for (long long pix = p_begin; pix < p_end; ++pix) {
      const int iy = (int)(pix / nx), ix = (int)(pix - (long long)iy * nx);
      double nbar[N];
      // fix-up mode: only the pixels qd_tunnel_eigen2_kernel marked with a NaN are (re)done here
      if (a.fixup && a.nbar[(pix0 + pix) * N] == a.nbar[(pix0 + pix) * N]) continue;
      if (!replace) {
        uint64_t key = a.tkeys[((size_t)scan_id * a.tstride + pix) * 32 + lane];
        // ---------------- voltages, potentials, tunnel couplings ----------------
        if (lane < NV) {
          vv[lane] = (a.points == nullptr) ? fma((double)iy, sc->dy[lane], fma((double)ix, sc->dx[lane], sc->v0[lane]))
                                           : a.points[(size_t)pix * NV + lane];
        }
        __syncwarp();
        if (lane < N) {
          double acc = 0.0;
          const double* arow = rec + L.o_a + lane * NV;
          for (int k = 0; k < NV; ++k) acc = fma(arow[k], vv[k], acc);
          if (vc_on) {
            double vabs = 0.0, v2 = 0.0, s_c, s_g;
            for (int k = 0; k < NV; ++k) { vabs += fabs(vv[k]); v2 = fma(vv[k], vv[k], v2); }
            vc_scales(par, vabs, v2, NV, s_c, s_g);
            acc *= s_g;
            if (lane == 0) ts[7] = s_c;
          }
          gs[lane] = acc;
        }
        if (lane >= 16 && lane < 16 + B) {
          const int d = lane - 16;
          double t = par[QD_PAR_TC_BASE];
          if (barriers) {
            double vb = vv[G + d];
            for (int k = 0; k < G; ++k) vb = fma(rec[L.o_cbg + d * G + k], vv[k], vb);
            t *= exp(-rec[L.o_alpha + d] * vb);
          }
          ts[d] = t;
        }
        __syncwarp();
        // ---------------- basis states, free energies ----------------
        double st[N];
        int tc = 0;                                // total charge of this lane's state
#pragma unroll
        for (int j = 0; j < N; ++j) {
          const int sj = (int)(signed char)(unsigned char)(key >> (8 * j));
          st[j] = (double)sj;
          tc += sj;
        }
        double Fm = 0.0;
        {
          double zz[N];
#pragma unroll
          for (int j = 0; j < N; ++j) zz[j] = st[j] - gs[j];
#pragma unroll
          for (int i = 0; i < N; ++i) {
            double s0 = 0.0;
#pragma unroll
            for (int j = 0; j < N; ++j) s0 = fma(C[i * N + j], zz[j], s0);
            Fm = fma(zz[i], s0, Fm);
          }
          if (vc_on) Fm /= ts[7];
        }
      // Hopping conserves the total charge, so H is block diagonal once the basis is ordered by total charge: the
      // 32 kept states typically fall into 5-6 sectors of <= 10-16 states.  Sort the lanes by (total charge, lane)
      // -- the spectrum and the weights |psi_m|^2 do not depend on the order of the basis -- and run every dense
      // step below on all sectors AT ONCE, each in its own lane segment [s0, s1]: reductions are segmented, the
      // inner loops run over the sector's columns only, and the number of Householder steps is the largest sector
      // size minus two instead of 30.
      int s0, s1, maxlen;
      {
        const unsigned same = __match_any_sync(0xffffffffu, tc);
        int rank = __popc(same & ((1u << lane) - 1u));
        unsigned rem = 0xffffffffu;
        while (rem) {
          const int leader = __ffs(rem) - 1;
          const int v = __shfl_sync(0xffffffffu, tc, leader);
          const unsigned grp = __shfl_sync(0xffffffffu, same, leader);
          if (v < tc) rank += __popc(grp);
          rem &= ~grp;
        }
        int* perm = reinterpret_cast<int*>(vq);
        perm[rank] = lane;
        __syncwarp();
        const int src = perm[lane];
        __syncwarp();
        key = shfl_u64(key, src);
        Fm = shfl_f64(Fm, src);
        tc = __shfl_sync(0xffffffffu, tc, src);
          #pragma unroll
        for (int j = 0; j < N; ++j) st[j] = (double)(int)(signed char)(unsigned char)(key >> (8 * j));
        const unsigned seg = __match_any_sync(0xffffffffu, tc);
        s0 = __ffs(seg) - 1;
        s1 = 31 - __clz(seg);
        maxlen = __reduce_max_sync(0xffffffffu, s1 - s0 + 1);
      }
      // Row `lane` of H, columns of its own sector only.  Two states are connected by a hop iff they differ in
      // exactly two ADJACENT dots, by (-1, +1) or (+1, -1): test on the XOR of the packed states first (cheap
      // reject), then compare the byte pair.
#pragma unroll 1
      for (int u = 0; u < maxlen; ++u) {
        const int j = min(s0 + u, 31);
        const uint64_t kj = shfl_u64(key, j);
        double val = (j == lane) ? Fm : 0.0;
        const uint64_t Hm = 0x8080808080808080ULL;
        const uint64_t x = kj ^ key;
        const uint64_t nz = (((x & ~Hm) + ~Hm) | x) & Hm;
        if (__popcll(nz) == 2 && (nz & (nz >> 8))) {
          const int p0 = (__ffsll((long long)nz) - 1) >> 3;
          const unsigned pa = (unsigned)(key >> (8 * p0)) & 0xffffu, pb = (unsigned)(kj >> (8 * p0)) & 0xffffu;
          const unsigned a0 = pa & 0xffu, a1 = pa >> 8;
          if (pb == pa + 0xffu) val = -ts[p0] * (sq_tab[a0] * sq_tab[a1 + 1]);        // p0 -> p0+1
          else if (pb + 0xffu == pa) val = -ts[p0] * (sq_tab[a1] * sq_tab[a0 + 1]);   // p0+1 -> p0
        }
        if (s0 + u <= s1) H[lane * QD_T_HS + j] = val;
      }
      __syncwarp();

      // ---------------- 4. ground eigenvector ----------------
      // Householder tridiagonalisation of every sector at once: step t works on column k = s0 + t of each sector
      // that still has at least two rows below it.
      const bool wide = maxlen > 16;
      for (int t = 0; t + 2 < maxlen; ++t) {
        const int k = s0 + t;
        const bool act = k + 2 <= s1;
        const double x = (act && lane > k) ? H[lane * QD_T_HS + k] : 0.0;
        const double xk1 = shfl_f64(x, min(k + 1, 31));
        const double sig = seg_sum((lane > k + 1) ? x * x : 0.0, lane, s0, s1, wide);
        const bool refl = act && sig != 0.0;
        double v = 0.0, alpha = xk1;
        if (refl) {
          const double norm2 = sig + xk1 * xk1;
          alpha = (xk1 > 0.0) ? -sqrt(norm2) : sqrt(norm2);
          v = x;
          if (lane == k + 1) v -= alpha;
          v *= rsqrt(2.0 * (norm2 - alpha * xk1));
        }
        vq[2 * lane] = v;
        __syncwarp();
        double p = 0.0;
        if (refl && lane > k) {
          double p0 = 0.0, p1 = 0.0;
          const double* __restrict__ hrow = H + lane * QD_T_HS;
          int j = k + 1;
          for (; j + 1 <= s1; j += 2) {
            p0 = fma(hrow[j], vq[2 * j], p0);
            p1 = fma(hrow[j + 1], vq[2 * j + 2], p1);
          }
          if (j <= s1) p0 = fma(hrow[j], vq[2 * j], p0);
          p = p0 + p1;
        }
        const double K = seg_sum(v * p, lane, s0, s1, wide);
        const double q = p - K * v;
        vq[2 * lane + 1] = q;
        __syncwarp();
        if (act && lane > k) {
          double* __restrict__ hrow = H + lane * QD_T_HS;
          if (refl) {
            const double v2 = -2.0 * v, q2 = -2.0 * q;
            for (int j = k + 1; j <= s1; ++j) {
              const double2 o = *reinterpret_cast<const double2*>(vq + 2 * j);     // (v_j, q_j)
              hrow[j] = fma(v2, o.y, fma(q2, o.x, hrow[j]));
            }
          }
          hrow[k] = v;                                     // the dead column keeps the reflector (0: none)
        }
        if (act && lane == s0) ee[k] = alpha;
        __syncwarp();
      }
      dd[lane] = H[lane * QD_T_HS + lane];
      // last coupling inside each sector, and none across sectors
      if (lane == s1) ee[lane] = 0.0;
      else if (lane == s1 - 1) ee[lane] = H[s1 * QD_T_HS + lane];
      __syncwarp();
      // Which sectors can hold the ground state at all?  lambda_min(sector) lies in [min_i (d_i - r_i), min_i d_i] (Gershgorin /
      // Rayleigh quotients of the unit vectors, on the sector's own tridiagonal); a sector whose lower end exceeds the
      // smallest diagonal entry U of the whole matrix is out.  The multisection then runs over the lane range that covers
      // the candidate sectors only (the others inside that range have every eigenvalue above U: their minors stay positive).
      double lo, hi, wfull;
      int c_lo, c_hi;
      {
        const double rad = ((lane > 0) ? fabs(ee[lane - 1]) : 0.0) + ((lane < 31) ? fabs(ee[lane]) : 0.0);
        const double lower = dd[lane] - rad;
        const double U = warp_min(dd[lane]);
        double ls = lower;                                   // segmented minimum over the lane's own sector
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const double t = __hiloint2double(__shfl_up_sync(0xffffffffu, __double2hiint(ls), d),
                                            __shfl_up_sync(0xffffffffu, __double2loint(ls), d));
          if (lane - d >= s0) ls = fmin(ls, t);
        }
        ls = shfl_f64(ls, s1);
        const bool cand = ls <= U || !(a.topt & 4);
        const unsigned cm = __ballot_sync(0xffffffffu, cand);          // never empty: the sector that owns U is in
        c_lo = __ffs(cm) - 1;
        c_hi = 31 - __clz(cm);
        lo = warp_min(cand ? lower : U);
        hi = U;
        wfull = warp_max(dd[lane] + rad) - warp_min(lower);
        // bracket width for the scaling below: not narrower than 1e-3 of the full Gershgorin width, so that the scaled
        // entries stay <= 1e3 in magnitude and the minors cannot overflow within a sector
        hi = fmax(hi, lo + 1e-3 * wfull);
      }
      // Lowest eigenvalue by 32-way multisection.  x < lambda_0  <=>  T - x I positive definite  <=>  every leading
      // principal minor p_i(x) > 0 (Sylvester); the minors obey p_{i+1} = (d_i - x) p_i - e_{i-1}^2 p_{i-1}.  The
      // tridiagonal is mapped onto the bracket [0, 1] first; a positive rescale every 8 steps guards the underflow side.
      const double lo0 = lo, wid = fmax(hi - lo, 1e-300), iw = 1.0 / wid;
      qi[lane] = (dd[lane] - lo0) * iw;
      e2[lane] = (ee[lane] * iw) * (ee[lane] * iw);
      __syncwarp();
      lo = 0.0;
      hi = 1.0;
      for (int round = 0; round < 6; ++round) {
        const double x = fma((double)(lane + 1) * (1.0 / 33.0), hi - lo, lo);
        double pp = 1.0, pc = qi[c_lo] - x;
        bool below = !(pc > 0.0);                  // some eigenvalue lies at or below x
        int i = c_lo + 1;
        // whole groups of 8 steps, fully unrolled (immediate-offset shared-memory loads), then the remainder
#pragma unroll 1
        for (; i + 7 <= c_hi; i += 8) {
          const double* __restrict__ q8 = qi + i;
          const double* __restrict__ e8 = e2 + i - 1;
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const double pn = fma(q8[u] - x, pc, -e8[u] * pp);
            below |= !(pn > 0.0);
            pp = pc;
            pc = pn;
          }
          const double ap = fabs(pc);
          if (ap < 1e-150) { pc *= 1e150; pp *= 1e150; }      // (irrelevant once `below` is set)
          else if (ap > 1e150) { pc *= 1e-150; pp *= 1e-150; }
        }
#pragma unroll 1
        for (; i <= c_hi; ++i) {
          const double pn = fma(qi[i] - x, pc, -e2[i - 1] * pp);
          below |= !(pn > 0.0);
          pp = pc;
          pc = pn;
        }
        const unsigned mm = __ballot_sync(0xffffffffu, below);
        const int j = mm ? __ffs(mm) - 1 : 32;
        const double xl = shfl_f64(x, (j > 0) ? j - 1 : 0);
        const double xh = shfl_f64(x, (j < 32) ? j : 31);
        if (j > 0) lo = xl;
        if (j < 32) hi = xh;
      }
      // The shift: the lower end of the final bracket, pushed down by 2e-12 of the Gershgorin width.  That is nothing for the
      // convergence of the inverse iteration ((lambda_0 - mu) / (lambda_1 - mu) per step) but keeps T - mu I positive
      // definite IN FLOATING POINT, four orders of magnitude above the rounding noise of the factorisation below: with the
      // narrow bracket a shift within rounding of lambda_0 could otherwise meet a zero pivot.
      lo = fma(lo, wid, lo0) - 2e-12 * wfull;
      __syncwarp();
      const double mu = lo;
      const double qmin = fmax(1e-15 * wfull, 1e-300);       // pivot floor (never reached unless the matrix is degenerate)
      // LDL^T of T - mu I and the inverse-iteration solves, every sector by its own leader lane (the sectors are
      // decoupled: ee[s1] = 0), so the serial chains are one sector long instead of 32.
      if (lane == s0) {
        double q = dd[s0] - mu;
        for (int i = s0; i < s1; ++i) {
          if (!(q > qmin)) q = qmin;
          const double iq = 1.0 / q;
          qi[i] = iq;
          const double l = ee[i] * iq;
          ll[i] = l;
          q = (dd[i + 1] - mu) - l * ee[i];
        }
        if (!(q > qmin)) q = qmin;
        qi[s1] = 1.0 / q;
      }
      yy[lane] = 1.0 + (double)lane * (1.0 / 64.0);
      __syncwarp();
      for (int it = 0; it < 3; ++it) {
        if (lane == s0) {
          double zprev = yy[s0];
          for (int i = s0 + 1; i <= s1; ++i) { zprev = yy[i] - ll[i - 1] * zprev; yy[i] = zprev; }
          double ynext = yy[s1] * qi[s1];
          yy[s1] = ynext;
          for (int i = s1 - 1; i >= s0; --i) { ynext = yy[i] * qi[i] - ll[i] * ynext; yy[i] = ynext; }
        }
        __syncwarp();
        double yv = yy[lane];
        // scale first (the unnormalised iterate can overflow when mu is within rounding of lambda_0)
        const double ymax = warp_max(fabs(yv));
        yv *= 1.0 / ymax;
        const double nrm = warp_sum(yv * yv);
        yy[lane] = yv * rsqrt(nrm);
        __syncwarp();
      }
      double psi = yy[lane];
      for (int t = maxlen - 3; t >= 0; --t) {
        const int k = s0 + t;
        const double v = (k + 2 <= s1 && lane > k) ? H[lane * QD_T_HS + k] : 0.0;
        const double dot = seg_sum(v * psi, lane, s0, s1, wide);
        psi = fma(-2.0 * dot, v, psi);
      }
        {
          const double w2 = psi * psi;
#pragma unroll
          for (int j = 0; j < N; ++j) nbar[j] = warp_sum(w2 * st[j]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < N; ++j) nbar[j] = 0.0;
      }
      // ---------------- <n> -> scratch ----------------
      {
        double mine = 0.0;
#pragma unroll
        for (int j = 0; j < N; ++j) mine = (lane == j) ? nbar[j] : mine;
        if (lane < N) a.nbar[(pix0 + pix) * N + lane] = mine;
      }
      __syncwarp();
    }
    __syncwarp();
  }
}

}  // namespace qd
