// qd_layout.h -- layout of one env's model record in HBM / shared memory (fp64 words), shared by host packing code
// and the kernels.  One record is a single 16-byte-aligned blob so that a warp stages it with ONE TMA bulk copy.
#pragma once
#include <stdint.h>

#include "../../include/qdsim.h"

// Parameter slots inside the record's `par` block.
enum {
  QD_PAR_KT = 0,
  QD_PAR_THRESHOLD = 1,
  QD_PAR_WHITE = 2,
  QD_PAR_P01 = 3,
  QD_PAR_P10 = 4,
  QD_PAR_TELE_AMP = 5,
  QD_PAR_TELE_STAT = 6,   // p01 / (p01 + p10): stationary probability of the "on" state
  QD_PAR_LATCH = 7,       // 1.0 if the env has a LatchingModel
  QD_PAR_MAXC = 8,        // max_charge_carriers
  QD_PAR_TC_BASE = 9,
  QD_PAR_VC_ALPHA = 10,   // linear voltage-dependent capacitance model (tunnel path), 0 = off
  QD_PAR_VC_BETA = 11,
  QD_PAR_PINK = 12,       // amplitude of the 1/f input-noise term (QD_FLAG_PINK)
  QD_PAR_VC_KIND = 13,    // enum qd_vc_kind
  QD_PAR_VC_VCHAR = 14,   // sigmoid model: characteristic voltage
  QD_PAR_COUNT = 16       // (even: the blocks after `par` stay 16-byte aligned)
};

struct qd_layout {
  int32_t n_dot, n_volt, n_gate, algorithm;
  int32_t num_states, chunk;
  int32_t o_cinv;    // [N*N]      ground-state quadratic form (cdd_inv)
  int32_t o_cdd;     // [N*N]      Maxwell cdd (M-matrix) for the exact relaxation
  int32_t o_a;       // [N*NV]     cgd rows of the dots
  int32_t o_sw;      // [S*N]      cdd_inv_full[N+s, 0:N]      sensor <-> dot couplings, row s per sensor
  int32_t o_css;     // [S*S]      cdd_inv_full[N+s, N+o]      sensor block
  int32_t o_sa;      // [S*NV]     cgd_full[N+s, :]            sensor rows
  int32_t o_par;     // [QD_PAR_COUNT]
  int32_t o_alpha;   // [8]        barrier alphas (tunnel)
  int32_t o_pleads;  // [8]
  int32_t o_pinter;  // [64]       stride 8
  int32_t o_spos;    // [8]        2 * sum_{k != j} max(Cinv_jk, 0)   (dominance bounds of the candidate search)
  int32_t o_sneg;    // [8]        2 * sum_{k != j} min(Cinv_jk, 0)
  int32_t o_q;       // [2^N]      Q[delta] = delta^T cdd_inv delta, delta in {0,1}^N, dot 0 = most significant bit
  int32_t o_cbg;     // [B*G]      (tunnel) raw positive barrier-gate matrix
  int32_t gs_doubles;   // (tunnel) length of the record PREFIX the ground-state kernel stages: cinv | a | par | alpha | cbg
  int32_t n_sensor;     // S, 1..QD_MAX_SENSORS
  int32_t pad1;
  int32_t rec_doubles;  // total, multiple of 2 (16 bytes)
};

// With one sensor (n_sensor = 1) every offset and rec_doubles are those of a layout without the sensor count.
static constexpr qd_layout qd_make_layout(int n_dot, int n_volt, int n_gate, int algorithm, int num_states, int chunk,
                                          int n_sensor = 1) {
  qd_layout L{};
  const int S = n_sensor;
  L.n_dot = n_dot; L.n_volt = n_volt; L.n_gate = n_gate; L.algorithm = algorithm;
  L.num_states = num_states; L.chunk = chunk;
  int o = 0;
  L.o_cinv = o;   o += n_dot * n_dot;
  if (algorithm == QD_ALG_TUNNEL) {
    // Everything qd_tunnel_gs_kernel reads comes first, so that its warps stage a short prefix only (their shared
    // memory also holds a 32 x 32 Hamiltonian; the smaller the slot, the more warps stay resident).
    L.o_a = o;      o += n_dot * n_volt;
    L.o_par = o;    o += QD_PAR_COUNT;
    L.o_alpha = o;  o += 8;
    L.o_cbg = o;    o += (n_volt - n_gate) * n_gate;
    o = (o + 1) & ~1;
    L.gs_doubles = o;
    L.o_cdd = o;    o += n_dot * n_dot;
    L.o_sw = o;     o += S * n_dot;
    L.o_css = o;    o += S * S;
    L.o_sa = o;     o += S * n_volt;
    L.o_pleads = o; o += 8;
    L.o_pinter = o; o += 64;
    L.o_spos = o;   o += 8;
    L.o_sneg = o;   o += 8;
    o = (o + 1) & ~1;
    L.o_q = o;
  } else {
    L.o_cdd = o;    o += n_dot * n_dot;
    L.o_a = o;      o += n_dot * n_volt;
    L.o_sw = o;     o += S * n_dot;
    L.o_css = o;    o += S * S;
    L.o_sa = o;     o += S * n_volt;
    L.o_par = o;    o += QD_PAR_COUNT;
    L.o_alpha = o;  o += 8;
    L.o_pleads = o; o += 8;
    L.o_pinter = o; o += 64;
    L.o_spos = o;   o += 8;
    L.o_sneg = o;   o += 8;
    o = (o + 1) & ~1;                       // Q rows are read as 16-byte pairs
    L.o_q = o;
    if (algorithm == QD_ALG_DEFAULT || algorithm == QD_ALG_THRESHOLDED) o += (1 << n_dot);
    L.o_cbg = o;
    L.gs_doubles = 0;
  }
  L.n_sensor = S;
  L.pad1 = 0;
  // (the tunnel path's block tables depend on a per-item permutation of the dots and are built inside the kernel)
  L.rec_doubles = (o + 1) & ~1;
  return L;
}
