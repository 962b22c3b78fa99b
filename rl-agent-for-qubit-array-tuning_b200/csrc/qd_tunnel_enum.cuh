// qd_tunnel_enum.cuh -- S2: the select stage of the tunnel-coupled path as a breadth-first lattice enumeration.
//
// Same contract as qd_tunnel_select_kernel (floor of the relaxed occupations in, the 32 candidates floor + {-1,0,1,2}^N of
// lowest (energy, index) out; reference: src/qarray_latched/DotArrays/charge_states.py:135-222), different algorithm.
//
// E(z) = z^T C z with C = L D L^T (unit lower L, natural dot order) is a sum of N non-negative terms,
//     E = sum_k d_k y_k^2,   y_k = z_k + sum_{j>k} L_jk z_j,
// and term k depends on dots k..N-1 only: fixing the dots from N-1 downwards, the partial sum over the fixed dots bounds
// every completion from below (Schnorr-Euchner).  With tau = the largest energy among the previous pixel's 32 states
// re-evaluated at this pixel (>= this pixel's 32nd-best energy whenever all 32 are still candidates), the candidates with
// E <= tau are enumerated level by level, a level's (node, digit) pairs spread over the lanes, survivors compacted into a
// shared-memory list by ballot + popc: ~100 nodes over all levels at 8 dots on the bench workload (tools/proto_se.py),
// 35 leaves, against ~2 000 candidates evaluated by the block walk of qd_tunnel_select_kernel.  The leaves are cut down to
// 32 by removing the (energy, index) maximum L - 32 times.  Energies of the warm start and of the enumeration are formed
// by the same rounded operations in the same order, so every warm state is found again bit for bit.
// Without a usable tau (first pixel of an item, states that left the candidate box when a floor moved) tau starts at the
// greedy leaf / the largest re-evaluated energy and grows until 32 leaves are inside.  A level that overflows its list
// (QD_S2_CAP nodes) marks the pixel; qd_tunnel_select_kernel redoes marked pixels in fix-up mode.
#pragma once
#include "qd_tunnel.cuh"

namespace qd {

constexpr int QD_S2_CAP = 320;                    // nodes per level list (two lists); leaves share them
constexpr unsigned long long QD_S2_MARK = 0xfffffffffffffffeULL;      // first key of a pixel left to the fix-up pass

// Slot of qd_tunnel_select2_kernel (qd_kernels.cuh: slot layouts).  Nothing is staged: the potentials come from the
// relax kernel, cdd_inv is read once per item for the factorisation, the four scalars of the scan descriptor straight
// from global memory.  The offsets count from the start of the slot.
struct Select2Slot {
  int rem;            // [8] rem[k]: lower bound of the levels below k
  int rs;             // [8] r = floor - g
  int rcm;            // [8]
  int rc;             // [8] rc_k = r_k + sum_{j>k} L_jk r_j
  int dd;             // [8]
  int Mt;             // [8][9] L^T with zeros below the diagonal: Mt[k * 9 + j] = L_jk for j > k, else 0
  int Lc;             // [64] Lc[j * N + k] = L_jk (j > k)
  int listP;          // [2][QD_S2_CAP]
  int listD;          // u32 [2][QD_S2_CAP]: QD_S2_CAP doubles
  int outk;           // u64 [32]
  int bytes;
};
__host__ __device__ constexpr Select2Slot qd_tunnel_select2_slot() {
  Select2Slot S{};
  int o = 16 * 8;                     // (the first 16 doubles are not used)
  S.rem = o;      o += 8 * 8;
  S.rs = o;       o += 8 * 8;
  S.rcm = o;      o += 8 * 8;
  S.rc = o;       o += 8 * 8;
  S.dd = o;       o += 8 * 8;
  S.Mt = o;       o += 72 * 8;
  S.Lc = o;       o += 64 * 8;
  S.listP = o;    o += 2 * QD_S2_CAP * 8;
  S.listD = o;    o += QD_S2_CAP * 8;
  S.outk = o;     o += 32 * 8;
  S.bytes = qd_slot_round(o);
  return S;
}

// One term of the energy, the same rounded operations wherever it is formed.  Digits enter as codes c = delta + 1 in
// 0..3 (what the packed node word holds): y_k = rcm_k + c_k + sum_{j>k} L_jk c_j with rcm_k = rc_k - 1 - sum_{j>k} L_jk.
__device__ __forceinline__ double s2_term(double rcm_k, double s, double code, double d_k, double P) {
  const double y = __dadd_rn(__dadd_rn(rcm_k, s), code);
  return __fma_rn(__dmul_rn(d_k, y), y, P);
}

template <int N>
__global__ void __launch_bounds__(128, 5) qd_tunnel_select2_kernel(const KArgs a) {
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ __align__(128) unsigned char qd_smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const qd_layout& L = a.L;

  // (9.5 KB per warp -> five CTAs per SM)
  constexpr Select2Slot S = qd_tunnel_select2_slot();
  unsigned char* slot = qd_smem + (size_t)warp * a.slot_bytes;
  double* gs = reinterpret_cast<double*>(slot + S.rem);
  double* rs = reinterpret_cast<double*>(slot + S.rs);
  double* fs = reinterpret_cast<double*>(slot + S.rcm);
  double* rc = reinterpret_cast<double*>(slot + S.rc);
  double* dd = reinterpret_cast<double*>(slot + S.dd);
  double* Mt = reinterpret_cast<double*>(slot + S.Mt);
  double* Lc = reinterpret_cast<double*>(slot + S.Lc);
  double* listP = reinterpret_cast<double*>(slot + S.listP);
  unsigned* listD = reinterpret_cast<unsigned*>(slot + S.listD);
  uint64_t* outk = reinterpret_cast<uint64_t*>(slot + S.outk);
  const double INF = __longlong_as_double(0x7ff0000000000000LL);

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
    const bool replace = (a.flags & QD_FLAG_RADIAL) && gscan->rad_mode == 2;
    const long long pix0 = gscan->pix_offset;
    if (replace) {
      if (lane == 0) a.nbar[(pix0 + p_begin) * N] = 0.0;
      continue;
    }
    const double* __restrict__ C = a.records + (size_t)gscan->env_id * L.rec_doubles + L.o_cinv;
    __syncwarp();

    // ---- per item: C = L D L^T (natural dot order), the whole warp on the N x N entries (a single lane doing it
    // serially showed up with 4.5 % of the kernel's stall samples) ----
    {
      double* __restrict__ W = listP;               // scratch: the lists are empty between items
      for (int e = lane; e < N * N; e += 32) W[e] = C[e];
      __syncwarp();
#pragma unroll 1
      for (int k = 0; k < N; ++k) {
        const double inv = 1.0 / W[k * N + k];
        for (int e = lane; e < N * N; e += 32) {
          const int i = e / N, j = e - i * N;
          if (i > k && j > k && j <= i) W[e] = fma(-(W[i * N + k] * inv), W[j * N + k], W[e]);
        }
        __syncwarp();
      }
      for (int e = lane; e < N * N; e += 32) {
        const int i = e / N, k = e - i * N;
        if (i > k) Lc[e] = W[e] / W[k * N + k];
      }
      if (lane < N) dd[lane] = W[lane * N + lane];
      __syncwarp();
      if (lane < N) {                               // (diagonal slot: 1 + column sum, for rcm)
        double cs = 0.0;
        for (int i = lane + 1; i < N; ++i) cs += Lc[i * N + lane];
        Lc[lane * N + lane] = 1.0 + cs;
      }
      __syncwarp();
    }
    for (int e = lane; e < N * N; e += 32) {
      const int k = e / N, j = e - k * N;
      Mt[k * 9 + j] = (j > k) ? Lc[j * N + k] : 0.0;
    }
    __syncwarp();
    double dmin = dd[0];
#pragma unroll
    for (int k = 1; k < N; ++k) dmin = fmin(dmin, dd[k]);

    uint64_t prev_key = ~0ULL;       // one of the previous pixel's 32 states (~0: none)
    bool any_marked = false;
    // floor and potential of a pixel are fetched one pixel ahead (their latency was 5 % of the stall samples)
    uint64_t fk_next = *reinterpret_cast<const uint64_t*>(a.tfloor + ((size_t)scan_id * a.tstride + p_begin) * 8);
    double g_next = a.tpot[((size_t)scan_id * a.tstride + p_begin) * 16 + (lane & 7)];
    for (long long pix = p_begin; pix < p_end; ++pix) {
      const size_t tslot = (size_t)scan_id * a.tstride + pix;
      // ---------------- potentials, floor (from the relax kernel), r = f - g, rc = L^T r ----------------
      const uint64_t fk = fk_next;
      if (lane < N) {                              // (the potentials come from the relax kernel)
        const double fj = (double)(unsigned)((fk >> (8 * lane)) & 0xffu);
        rs[lane] = fj - g_next;
      }
      if (pix + 1 < p_end) {
        fk_next = *reinterpret_cast<const uint64_t*>(a.tfloor + (tslot + 1) * 8);
        g_next = a.tpot[(tslot + 1) * 16 + (lane & 7)];
      }
      __syncwarp();
      // dots whose floor is 0 lose the digit -1 (negative occupation: not a candidate)
      unsigned zero_floor = 0;
#pragma unroll
      for (int j = 0; j < N; ++j) zero_floor |= (((fk >> (8 * j)) & 0xffu) == 0) ? (1u << j) : 0u;
      // rc, rcm, and the lower bound of the terms still to come below level k, whatever the digits: y_j lies in an interval
      // (digits in [lo, 2], interval arithmetic over the dots above j), term_j >= d_j dist(0, interval)^2.  Without it a
      // deeply empty dot at the bottom of the tree (all of its digits cost ~tau) would leave the levels above it unpruned.
      // Lane k < N owns dot k; fixed trip counts on the zero-padded Mt (no serial single-lane stretches).
      {
        const int kk = min(lane, N - 1);
        const double* __restrict__ mrow = Mt + kk * 9;
        double sacc = rs[kk], smin = 0.0, smax = 0.0;
#pragma unroll
        for (int j = 0; j < N; ++j) {
          const double l = mrow[j];
          sacc = fma(l, rs[j], sacc);
          const double a0 = ((zero_floor >> j) & 1u) ? 0.0 : -l, a1 = 2.0 * l;
          smin += fmin(a0, a1);
          smax += fmax(a0, a1);
        }
        const double ylo = sacc + (((zero_floor >> kk) & 1u) ? 0.0 : -1.0) + smin;
        const double yhi = sacc + 2.0 + smax;
        const double dist = (ylo > 0.0) ? ylo : ((yhi < 0.0) ? -yhi : 0.0);
        const double bound = (lane < N) ? dd[kk] * dist * dist * (1.0 - 1e-9) : 0.0;
        double incl = bound;                          // rem[k] = sum_{j < k} bound_j: exclusive scan over lanes 0..N-1
#pragma unroll
        for (int d = 1; d < N; d <<= 1) {
          const double t = __hiloint2double(__shfl_up_sync(FULL, __double2hiint(incl), d),
                                            __shfl_up_sync(FULL, __double2loint(incl), d));
          if (lane >= d) incl += t;
        }
        if (lane < N) {
          rc[lane] = sacc;
          fs[lane] = sacc - Lc[lane * N + lane];      // rcm
          gs[lane] = incl - bound;
        }
      }
      __syncwarp();
      const double* __restrict__ rem = gs;
      const double* __restrict__ rcm = fs;

      // ---------------- tau from the previous pixel's states ----------------
      double tau;
      int n_warm = 0;
      {
        bool ok = prev_key != ~0ULL;
        double dl[N];
#pragma unroll
        for (int j = 0; j < N; ++j) {
          const int dg = (int)((prev_key >> (8 * j)) & 0xffu) - (int)((fk >> (8 * j)) & 0xffu);
          ok = ok && dg >= -1 && dg <= 2;
          dl[j] = (double)(dg + 1);
        }
        double E = 0.0;
#pragma unroll
        for (int k = N - 1; k >= 0; --k) {
          double s = 0.0;
#pragma unroll
          for (int j = k + 1; j < N; ++j) s = __fma_rn(Lc[j * N + k], dl[j], s);
          E = s2_term(rcm[k], s, dl[k], dd[k], E);
        }
        const unsigned okm = __ballot_sync(FULL, ok);
        n_warm = __popc(okm);
        tau = warp_max(ok ? E : -INF);
      }
      if (n_warm == 0) {
        // greedy leaf: at every level the best digit given the digits above (a real candidate, so at least one leaf)
        double dl[N];
        double E = 0.0;
#pragma unroll
        for (int k = N - 1; k >= 0; --k) {
          double s = 0.0;
#pragma unroll
          for (int j = k + 1; j < N; ++j) s = __fma_rn(Lc[j * N + k], dl[j], s);
          double best = INF, bd = 0.0;
#pragma unroll
          for (int cd = 0; cd <= 3; ++cd) {
            if (cd == 0 && ((zero_floor >> k) & 1u)) continue;
            const double e = s2_term(rcm[k], s, (double)cd, dd[k], E);
            if (e < best) { best = e; bd = (double)cd; }
          }
          dl[k] = bd;
          E = best;
        }
        tau = E;
      }

      // ---------------- enumeration, tau grown until 32 leaves are inside ----------------
      int nleaf = 0, cur = 0;
      bool marked = false;
      for (int pass = 0;; ++pass) {
        if (pass >= 24) { marked = true; break; }
        // level 0: the root's children (dot N-1)
        int cnt = 0;
        cur = 0;
        {
          const int k = N - 1;
          const int dg = lane - 1;
          const bool act = lane < 4 && !(dg == -1 && ((zero_floor >> k) & 1u));
          const double P2 = s2_term(rcm[k], 0.0, (double)(dg + 1), dd[k], 0.0);
          const bool keep = act && P2 + rem[k] <= tau;
          const unsigned mk = __ballot_sync(FULL, keep);
          if (keep) {
            const int pos = __popc(mk & ((1u << lane) - 1u));
            listP[pos] = P2;
            listD[pos] = (unsigned)(dg + 1) << (2 * (N - 1 - k));
          }
          cnt = __popc(mk);
        }
        __syncwarp();
        bool overflow = false;
        // (levels unrolled: k is a compile-time constant in each body, so the digits of the dots above come out of the node
        // word with constant shifts and the L entries with immediate offsets)
#pragma unroll
        for (int k = N - 2; k >= 0; --k) {
          if (cnt > 0 && !overflow) {
            const double* __restrict__ inP = listP + cur * QD_S2_CAP;
            const unsigned* __restrict__ inD = listD + cur * QD_S2_CAP;
            double* __restrict__ outP = listP + (cur ^ 1) * QD_S2_CAP;
            unsigned* __restrict__ outD = listD + (cur ^ 1) * QD_S2_CAP;
            const double rck = rcm[k], dk = dd[k], remk = rem[k];
            const bool no_minus = (zero_floor >> k) & 1u;
            const int pairs = 4 * cnt;
            int out = 0;
#pragma unroll 1
            for (int base = 0; base < pairs; base += 32) {
              const int pr = base + lane;
              const int node = min(pr >> 2, cnt - 1);
              const int cd = pr & 3;
              const double P = inP[node];
              const unsigned dgs = inD[node];
              double s = 0.0;
#pragma unroll
              for (int j = k + 1; j < N; ++j)
                s = __fma_rn(Lc[j * N + k], (double)((dgs >> (2 * (N - 1 - j))) & 3u), s);
              const double P2 = s2_term(rck, s, (double)cd, dk, P);
              const bool keep = pr < pairs && !(cd == 0 && no_minus) && P2 + remk <= tau;
              const unsigned mk = __ballot_sync(FULL, keep);
              const int pos = out + __popc(mk & ((1u << lane) - 1u));
              out += __popc(mk);
              if (out > QD_S2_CAP) { overflow = true; break; }
              if (keep) {
                outP[pos] = P2;
                outD[pos] = dgs | ((unsigned)cd << (2 * (N - 1 - k)));
              }
            }
            if (!overflow) {
              cnt = out;
              cur ^= 1;
            }
            __syncwarp();
          }
        }
        if (overflow) { marked = true; break; }
        nleaf = cnt;
        if (nleaf >= 32) break;
        // fewer than 32 candidates inside: grow tau (the count grows like tau^(N/2); aim at a factor ~3)
        double emin = INF;
        for (int i = lane; i < nleaf; i += 32) emin = fmin(emin, listP[cur * QD_S2_CAP + i]);
        emin = warp_min(emin);
        if (!(emin < INF)) emin = tau;
        const double span = fmax(tau - emin, 0.1 * dmin);
        tau = emin + span * ((N >= 6) ? 1.25 : 1.6);
        __syncwarp();
      }

      // ---------------- the 32 best of the leaves: drop the (energy, index) maximum nleaf - 32 times ----------------
      uint64_t key = ~0ULL;
      if (!marked) {
        const double* __restrict__ lp = listP + cur * QD_S2_CAP;
        const unsigned* __restrict__ ld = listD + cur * QD_S2_CAP;
        const int T = (nleaf + 31) >> 5;           // leaves lane, lane + 32, ... of this lane (<= 10)
        unsigned alive = 0;
        for (int t = 0; t < T; ++t) alive |= (lane + 32 * t < nleaf) ? (1u << t) : 0u;
#pragma unroll 1
        for (int r = nleaf - 32; r > 0; --r) {
          double me = -INF;
          int mi = -1, mt = 0;
          for (int t = 0; t < T; ++t) {
            if ((alive >> t) & 1u) {
              const double e = lp[lane + 32 * t];
              const int ii = (int)ld[lane + 32 * t];
              if (lex_less(me, mi, e, ii)) { me = e; mi = ii; mt = t; }
            }
          }
          double we;
          int wi, wl;
          warp_lex_max(me, mi, lane, we, wi, wl);
          if (lane == wl) alive &= ~(1u << mt);
        }
        // compact the survivors: lane order inside each stride, strides in order
        int before = 0;
        for (int t = 0; t < T; ++t) {
          const bool al = (alive >> t) & 1u;
          const unsigned mk = __ballot_sync(FULL, al);
          if (al) {
            const int pos = before + __popc(mk & ((1u << lane) - 1u));
            const unsigned idx = ld[lane + 32 * t];
            uint64_t kk = 0;
#pragma unroll
            for (int j = 0; j < N; ++j) {
              const unsigned sj = (unsigned)((fk >> (8 * j)) & 0xffu) + ((idx >> (2 * (N - 1 - j))) & 3u) - 1u;
              kk |= (uint64_t)(sj & 0xffu) << (8 * j);
            }
            outk[pos] = kk;
          }
          before += __popc(mk);
        }
        __syncwarp();
        key = outk[lane];
        a.tkeys[tslot * 32 + lane] = key;
      } else {
        if (lane == 0) a.tkeys[tslot * 32] = QD_S2_MARK;
        any_marked = true;
      }
      if (!marked) prev_key = key;       // (a marked pixel leaves the older states in place: still a usable tau)
      __syncwarp();
    }
    // item-level mark for the fix-up pass (the eigen stage overwrites this scratch afterwards)
    if (lane == 0) a.nbar[(pix0 + p_begin) * N] = any_marked ? __longlong_as_double(0x7ff8000000000000LL) : 0.0;
    __syncwarp();
  }
}

}  // namespace qd
