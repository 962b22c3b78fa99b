/*
 * qd_cport_closed.c -- plain-C restatement of the closed-array scan (total charge q on the dots; CPU baseline; TEST
 * INFRASTRUCTURE, see oracle/__init__.py): the decisions of oracle/closed.py, in the reference formulation of
 * qd_cport.c -- every candidate's full quadratic form, the 11 full-system sensor free energies, sequential latching and
 * telegraph loops.  It includes qd_cport.c for the shared pieces (Philox, energy, the open restatement itself); the
 * scan loop below is qd_cport.c's scan_rows with the closed ground state in place of the open one.
 *
 * Build: gcc -O3 -march=x86-64-v3 -fopenmp -fPIC -shared -o libqd_cport_closed.so qd_cport_closed.c -lm
 */
#include "qd_cport.c"

/* ---- closed arrays (total charge q on the dots; oracle/closed.py: ground_state_closed) ---- */

/* exact closed relaxation, min (n-g)^T cinv (n-g) over n >= 0, sum n = q: for every free set F the equality-constrained
 * solution n_F = cinv_FF^-1 (cinv_F g + t 1), sum n_F = q; the feasible (n_F >= 0) one of lowest energy */
static void relax_closed(int n, const double* g, const double* cinv, double q, double* nc) {
  double ag[MAXN], best = INFINITY;
  for (int i = 0; i < n; ++i) { double a = 0; for (int j = 0; j < n; ++j) a += cinv[i * n + j] * g[j]; ag[i] = a; }
  for (int i = 0; i < n; ++i) nc[i] = 0.0;
  for (unsigned mask = 1; mask < (1u << n); ++mask) {
    int idx[MAXN], k = 0;
    for (int i = 0; i < n; ++i) if ((mask >> i) & 1u) idx[k++] = i;
    /* solve cinv_FF [u v] = [ag_F 1] */
    double m[MAXN][MAXN + 2];
    for (int a = 0; a < k; ++a) {
      for (int b = 0; b < k; ++b) m[a][b] = cinv[idx[a] * n + idx[b]];
      m[a][k] = ag[idx[a]];
      m[a][k + 1] = 1.0;
    }
    for (int p = 0; p < k; ++p)
      for (int a = p + 1; a < k; ++a) {
        const double f = m[a][p] / m[p][p];
        for (int b = p; b < k + 2; ++b) m[a][b] -= f * m[p][b];
      }
    double u[MAXN], v[MAXN], su = 0, sv = 0;
    for (int a = k - 1; a >= 0; --a) {
      double s0 = m[a][k], s1 = m[a][k + 1];
      for (int b = a + 1; b < k; ++b) { s0 -= m[a][b] * u[b]; s1 -= m[a][b] * v[b]; }
      u[a] = s0 / m[a][a];
      v[a] = s1 / m[a][a];
      su += u[a];
      sv += v[a];
    }
    const double t = (q - su) / sv;
    double cand[MAXN] = {0};
    int ok = 1;
    for (int a = 0; a < k; ++a) { cand[idx[a]] = u[a] + t * v[a]; if (cand[idx[a]] < -1e-12) ok = 0; }
    if (!ok) continue;
    const double e = energy(n, cand, g, cinv);
    if (e < best) { best = e; memcpy(nc, cand, sizeof(double) * n); }
  }
  for (int i = 0; i < n; ++i) nc[i] = nc[i] < 0 ? 0 : (nc[i] > q ? q : nc[i]);
}

/* candidates of one pixel: first pass argmin (and second-lowest energy), second pass Boltzmann accumulation */
static void closed_take(int n, const double* conf, double e, int pass, double kT, double* best, double* second,
                        double* best_conf, double* z, double* acc) {
  if (pass == 0) {
    if (e < *best) { *second = *best; *best = e; memcpy(best_conf, conf, sizeof(double) * n); }
    else if (e < *second) *second = e;
  } else {
    const double wgt = exp(-(e - *best) / kT);
    *z += wgt;
    for (int i = 0; i < n; ++i) acc[i] += wgt * conf[i];
  }
}

static void ground_state_closed(int n, int alg, const double* g, const double* cinv, int q, double kT, double* nd,
                                double* margin) {
  double conf[MAXN], best_conf[MAXN], best = INFINITY, second = INFINITY, z = 0.0, acc[MAXN] = {0};
  double fl[MAXN];
  int fsum = 0;
  if (alg != QD_ALG_BRUTE_FORCE) {
    double nc[MAXN];
    relax_closed(n, g, cinv, (double)q, nc);
    for (int i = 0; i < n; ++i) { fl[i] = floor(nc[i]); fsum += (int)fl[i]; }
  }
  for (int pass = 0; pass < (kT > 0 ? 2 : 1); ++pass) {
    if (alg == QD_ALG_BRUTE_FORCE) {
      /* every composition of q into n parts, ascending (dot 0 slowest): an odometer over the first n-1 dots that carries
       * as soon as they hold all q carriers; the last dot takes the rest */
      int c[MAXN] = {0}, used = 0;
      while (1) {
        for (int i = 0; i < n - 1; ++i) conf[i] = c[i];
        conf[n - 1] = q - used;
        closed_take(n, conf, energy(n, conf, g, cinv), pass, kT, &best, &second, best_conf, &z, acc);
        int i = n - 2;
        for (; i >= 0; --i) {
          if (used < q) { ++c[i]; ++used; break; }
          used -= c[i];
          c[i] = 0;
        }
        if (i < 0) break;
      }
    } else {
      for (unsigned d = 0; d < (1u << n); ++d) {
        int sum = fsum;
        for (int i = 0; i < n; ++i) { const int b = (d >> (n - 1 - i)) & 1; conf[i] = fl[i] + b; sum += b; }
        if (sum != q) continue;
        closed_take(n, conf, energy(n, conf, g, cinv), pass, kT, &best, &second, best_conf, &z, acc);
      }
    }
  }
  for (int i = 0; i < n; ++i) nd[i] = kT > 0 ? acc[i] / z : best_conf[i];
  if (margin) *margin = second - best;
}

/* qd_cport.c's scan_rows with the closed ground state of total charge q */
static void scan_rows_closed(const qd_scan* s, int n, int nv, int alg, unsigned flags, const double* cinv,
                             const double* cinv_full, const double* cgd_full, const qd_env_params* p, int row0, int row1,
                             float* z_out, double* n_out, double* margin_out, int q) {
  const int d = n + 1, nx = s->nx;
  const double kT = (flags & QD_FLAG_THERMAL) ? p->kT : 0.0;
  const int latch = (flags & QD_FLAG_LATCH) && p->latching;
  const int noise = flags & QD_FLAG_NOISE;
  const int rad_mode = (flags & QD_FLAG_RADIAL) ? s->rad_mode : 0;
  const int carry = flags & QD_FLAG_CARRY_ROWS;
  double held[MAXN], heldk[MAXN];
  int have_held = 0, tele = 0, tele_init = 0;
  const double tot = p->tele_p01 + p->tele_p10;
  for (int iy = row0; iy < row1; ++iy) {
    if (!carry) { have_held = 0; tele_init = 0; }
    for (int ix = 0; ix < nx; ++ix) {
      const uint64_t pix = (uint64_t)iy * nx + ix;
      uint32_t w[4];
      philox(s->seed, pix, 0, w);
      const double u1 = ((double)(w[0] >> 8) + 1.0) / 16777216.0, u2 = u24(w[1]);
      const double rr = sqrt(-2.0 * log(u1)), ang = 2.0 * M_PI * u2;
      const double z_white = rr * cos(ang), z_rad = rr * sin(ang), u_latch = u24(w[2]), u_tele = u24(w[3]);
      double v[QD_MAX_VOLT], g[MAXN], nd[MAXN];
      for (int k = 0; k < nv; ++k) v[k] = (s->v0[k] + ix * s->dx[k]) + iy * s->dy[k];
      for (int i = 0; i < n; ++i) { double a = 0; for (int k = 0; k < nv; ++k) a += cgd_full[i * nv + k] * v[k]; g[i] = a; }
      double mg = INFINITY;
      ground_state_closed(n, alg, g, cinv, q, kT, nd, margin_out ? &mg : NULL);
      if (margin_out) margin_out[s->pix_offset + (int64_t)pix] = mg;
      if (latch) {
        double key[MAXN];
        for (int i = 0; i < n; ++i) key[i] = (flags & QD_FLAG_LATCH_EXACT) ? nd[i] : floor(nd[i] + 0.5);
        if (!have_held) { memcpy(held, nd, sizeof(double) * n); memcpy(heldk, key, sizeof(double) * n); have_held = 1; }
        else {
          int nd_ = 0, d0 = -1, d1 = -1;
          for (int i = 0; i < n; ++i) if (key[i] != heldk[i]) { if (nd_ == 0) d0 = i; else d1 = i; ++nd_; }
          int accept = 1;
          if (nd_ == 1) accept = u_latch < p->p_leads[d0];
          else if (nd_ == 2) accept = u_latch < p->p_inter[d0 * QD_MAX_DOTS + d1];
          if (accept) { memcpy(held, nd, sizeof(double) * n); memcpy(heldk, key, sizeof(double) * n); }
          else memcpy(nd, held, sizeof(double) * n);
        }
      }
      double noise_in = 0.0, noise_out = 0.0;
      if (noise) {
        if (flags & QD_FLAG_WHITE_ON_OUTPUT) noise_out = p->white_amp * z_white; else noise_in = p->white_amp * z_white;
        if (p->tele_amp != 0.0) {
          if (!tele_init) {
            if (carry) tele = 0;
            else { uint32_t wr[4]; philox(s->seed, (uint64_t)iy, 1, wr); tele = (tot > 0 && u24(wr[0]) < p->tele_p01 / tot) ? 1 : 0; }
            tele_init = 1;
          }
          if (u_tele < (tele ? p->tele_p10 : p->tele_p01)) tele ^= 1;
          noise_in += p->tele_amp * tele;
        }
      }
      /* sensor: eleven full-system free energies, first differences, ten Lorentzians */
      double vdash[MAXN + 1], nf[MAXN + 1], f[11];
      for (int i = 0; i < d; ++i) { double a = 0; for (int k = 0; k < nv; ++k) a += cgd_full[i * nv + k] * v[k]; vdash[i] = a; }
      const double ns = nearbyint(vdash[n]);
      for (int i = 0; i < n; ++i) nf[i] = nd[i];
      for (int k = -5; k <= 5; ++k) {
        nf[n] = ns + k + noise_in;
        double e = 0.0;
        for (int i = 0; i < d; ++i) { double sacc = 0; for (int j = 0; j < d; ++j) sacc += cinv_full[i * d + j] * (nf[j] - vdash[j]); e += (nf[i] - vdash[i]) * sacc; }
        f[k + 5] = e;
      }
      double z = 0.0;
      for (int k = 0; k < 10; ++k) { double x = (f[k + 1] - f[k]) / s->peak_width; z += 1.0 / (x * x + 1.0); }
      z += noise_out;
      if (rad_mode == 1) {
        double vx = s->rad_x0 + ix * s->rad_dx, vy = s->rad_y0 + iy * s->rad_dy;
        double amp = s->rad_alpha * (sqrt(vx * vx + vy * vy) - s->rad_zero_radius);
        amp = amp < 0 ? 0 : (amp > s->rad_max_amp ? s->rad_max_amp : amp);
        z += z_rad * amp;
      } else if (rad_mode == 2) z = z_rad;
      const int64_t o = s->pix_offset + (int64_t)pix;
      if (z_out) z_out[o] = (float)z;
      if (n_out) for (int i = 0; i < n; ++i) n_out[o * n + i] = nd[i];
    }
  }
}

/* Closed arrays: as qd_cport_scans, scan i with total charge n_charge[i] on the dots (algorithm default or brute_force;
 * -2 for any other algorithm or a charge outside 0..251 / 0..15). */
int qd_cport_scans_closed(int n_scan, const qd_scan* scans, const int32_t* n_charge, int n_dot, int n_volt, int algorithm,
                          unsigned flags, const double* cdd_inv_gs, const double* cdd_inv_full, const double* cgd_full,
                          const qd_env_params* params, float* z_out, double* n_out, double* margin_out, int threads) {
  const int n = n_dot, d = n_dot + 1, nv = n_volt;
  if (n < 1 || n > MAXN || nv > QD_MAX_VOLT) return -1;
  if (algorithm != QD_ALG_DEFAULT && algorithm != QD_ALG_BRUTE_FORCE) return -2;
  for (int i = 0; i < n_scan; ++i)
    if (n_charge[i] < 0 || n_charge[i] > (algorithm == QD_ALG_BRUTE_FORCE ? 15 : 251)) return -2;
#ifdef _OPENMP
  if (threads > 0) omp_set_num_threads(threads);
#endif
  const int carry = flags & QD_FLAG_CARRY_ROWS;
  for (int i = 0; i < n_scan; ++i) {
    const qd_scan* s = scans + i;
    const int e = s->env_id;
    const double* ci = cdd_inv_gs + (size_t)e * n * n;
    const double* cf = cdd_inv_full + (size_t)e * d * d;
    const double* cg = cgd_full + (size_t)e * d * nv;
    if (carry) {
      scan_rows_closed(s, n, nv, algorithm, flags, ci, cf, cg, params + e, 0, s->ny, z_out, n_out, margin_out, n_charge[i]);
    } else {
#pragma omp parallel for schedule(dynamic, 1)
      for (int iy = 0; iy < s->ny; ++iy)
        scan_rows_closed(s, n, nv, algorithm, flags, ci, cf, cg, params + e, iy, iy + 1, z_out, n_out, margin_out,
                         n_charge[i]);
    }
  }
  return 0;
}