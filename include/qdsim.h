/*
 * qdsim.h -- C ABI of libqdsim.so, the B200-native charge-stability simulator.
 *
 * The reference (edwindn/rl-agent-for-qubit-array-tuning) has no FFI: its boundary for this path is the Python
 * import surface of `qarray` / `qarray_latched` consumed by src/qadapt/environment/qarray_base_class.py:12-17.
 * The Python classes in rl-agent-for-qubit-array-tuning_b200/{qarray,qarray_latched} keep those names and
 * signatures and call the entry points below through ctypes.  Each entry point cites what it replaces.
 *
 * Conventions: plain pointers and sizes, no C++ / torch types; every function returns 0 (QD_OK) or a negative
 * qd_err and never throws or aborts; qd_last_error() gives the message.  A qd_ctx belongs to one CUDA device
 * and is NOT thread-safe.  All matrices are fp64, row-major, in the reference's Maxwell sign convention
 * (cgd = -Cgd).  "device pointer" = memory of ctx's device (e.g. a torch tensor's data_ptr()).
 */
#ifndef QDSIM_H
#define QDSIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QD_ABI_VERSION 3
#define QD_MAX_DOTS 8   /* BASELINE.json configs go to 8 dots                                  */
#define QD_MAX_VOLT 16  /* n_gate + n_barrier = (N+1) + (N-1)                                  */
#define QD_MAX_SENSORS 4 /* charge sensors of a model set (qd_model_desc.n_sensor)                   */

typedef struct qd_ctx qd_ctx;

enum qd_err {
  QD_OK = 0,
  QD_ERR_INVALID = -1,     /* bad argument (the reference raises ValueError / AssertionError)        */
  QD_ERR_CUDA = -2,        /* a CUDA runtime call failed                                             */
  QD_ERR_NOMEM = -3,
  QD_ERR_STATE = -4,       /* e.g. scan before qd_set_models                                         */
  QD_ERR_UNSUPPORTED = -5
};

/* Ground-state algorithm; mirrors `algorithm=` of ChargeSensedDotArray
 * (qarray_base_class.py:753; allowed values _helper_functions.py:202-210). QD_ALG_TUNNEL is the
 * TunnelCoupledChargeSensed path (qarray_latched/DotArrays/ground_state.py:24-166). */
enum qd_algorithm { QD_ALG_DEFAULT = 0, QD_ALG_THRESHOLDED = 1, QD_ALG_BRUTE_FORCE = 2, QD_ALG_TUNNEL = 3 };

/* Output element type of the charge map. */
enum qd_ntype { QD_N_NONE = 0, QD_N_U8 = 1, QD_N_F32 = 2, QD_N_F64 = 3 };

/* Element type of a compact observation image (qd_scan_obs_host / qd_normalise_obs_typed): fp32, IEEE half, or uint8
 * = rint(255 * x) of an image normalised to [0, 1].  fp32 stays the parity format; the compact types exist because the
 * host-buffer path is bound by the device-to-host copy of the images, not by the kernels. */
enum qd_ztype { QD_Z_F32 = 0, QD_Z_F16 = 1, QD_Z_U8 = 2 };

/* bits of qd_status() */
#define QD_STATUS_OCC_OVERFLOW 0x1u  /* a scan window reaches occupations >= 254 carriers per dot: uint8 charge maps  */
                                     /* and the packed latching keys would saturate (results of that launch invalid) */

/* flags of qd_scan_open / qd_points_open */
#define QD_FLAG_LATCH            0x01u  /* apply the envs' LatchingModel (S5)                              */
#define QD_FLAG_NOISE            0x02u  /* white + telegraph sensor noise (S6)                             */
#define QD_FLAG_RADIAL           0x04u  /* QADAPT radial noise / replacement (S7), per-scan rad_mode       */
#define QD_FLAG_THERMAL          0x08u  /* honour per-env kT > 0 (Boltzmann average; non-integer charges)  */
#define QD_FLAG_CARRY_ROWS       0x10u  /* latching + telegraph state carried across row ends (flat pass)  */
#define QD_FLAG_LATCH_EXACT      0x20u  /* compare raw (not rounded) occupations when latching: identical to the */
                                        /* rounded compare on integer occupations; QD_ERR_UNSUPPORTED on         */
                                        /* non-integer ones (QD_FLAG_THERMAL, QD_ALG_TUNNEL)                     */
#define QD_FLAG_WHITE_ON_OUTPUT  0x40u  /* white noise added to the signal instead of the sensor occupation */
#define QD_FLAG_PINK             0x80u  /* 1/f sensor input noise of amplitude pink_amp (north_star's "1-f noise"; the   */
                                        /* reference itself has no 1/f model, SURVEY 8a S6): sum of four Ornstein-        */
                                        /* Uhlenbeck chains along the fast axis, correlation lengths 2, 8, 32, 128 pixels  */

/* Per-env scalar parameters: the constructor arguments of ChargeSensedDotArray / TunnelCoupledChargeSensed,
 * LatchingModel, WhiteNoise, TelegraphNoise and BarrierVoltageModel (qarray_base_class.py:726-756, 779-838). */
typedef struct qd_env_params {
  double kT;                               /* k_B * T (ground_state.py:48); 0 = hard argmin                 */
  double threshold;                        /* thresholded algorithm                                         */
  double white_amp;                        /* WhiteNoise(amplitude)                                         */
  double tele_p01, tele_p10, tele_amp;     /* TelegraphNoise(p01, p10, amplitude)                           */
  double p_leads[QD_MAX_DOTS];             /* LatchingModel.p_leads                                         */
  double p_inter[QD_MAX_DOTS * QD_MAX_DOTS]; /* LatchingModel.p_inter, row-major, stride QD_MAX_DOTS        */
  double tc_base;                          /* BarrierVoltageModel.tc_base            (QD_ALG_TUNNEL)        */
  double alpha[QD_MAX_DOTS];               /* BarrierVoltageModel.alpha[n_barrier]   (QD_ALG_TUNNEL)        */
  double vc_alpha, vc_beta;                /* voltage-dependent capacitances (QD_ALG_TUNNEL), per pixel in   */
                                           /* the ground state: cdd *= s_c(v; vc_kind, vc_alpha [, vc_vchar]), */
                                           /* cgd *= 1 + vc_beta mean|v| (voltage_dependent_capacitance.py:   */
                                           /* 78-167); 0, 0 = constant capacitances                          */
  int32_t max_charge_carriers;             /* brute_force                                                   */
  int32_t latching;                        /* 0: env has no LatchingModel                                   */
  double pink_amp;                         /* QD_FLAG_PINK: standard deviation of the 1/f input-noise term   */
  double vc_vchar;                         /* vc_kind = sigmoid: characteristic voltage v_char                */
  int32_t vc_kind;                         /* enum qd_vc_kind: how vc_alpha scales cdd (see below)            */
  int32_t reserved0;
} qd_env_params;

/* Voltage-dependent capacitance models of the tunnel path (voltage_dependent_capacitance.py:78-167).  In all of them
 * cgd scales by 1 + vc_beta mean|v|; cdd scales by
 *   QD_VC_LINEAR     1 + vc_alpha mean|v|                                   (create_linear_capacitance_model, :123-135)
 *   QD_VC_QUADRATIC  1 + vc_alpha sum v^2           (vc_alpha = gamma)      (create_quadratic_capacitance_model, :138-151)
 *   QD_VC_SIGMOID    1 + vc_alpha sigmoid(|v|_2 / vc_vchar - 1)  (vc_alpha = delta)   (create_sigmoid_..., :154-168)
 * over ALL entries of the pixel's voltage vector (ground_state.py:53-58). */
enum qd_vc_kind { QD_VC_LINEAR = 0, QD_VC_QUADRATIC = 1, QD_VC_SIGMOID = 2 };

/* Shape and algorithm of a model set (all envs of one set share them). */
typedef struct qd_model_desc {
  int32_t n_env;
  int32_t n_dot;            /* N, 1..QD_MAX_DOTS                                                          */
  int32_t n_sensor;         /* S, 1..QD_MAX_SENSORS (see "Several charge sensors" below)                 */
  int32_t n_volt;           /* columns of cgd: n_gate (Path A) or n_gate + n_barrier (tunnel)             */
  int32_t n_gate;           /* physical gates incl. the sensor gates                                      */
  int32_t algorithm;        /* enum qd_algorithm                                                          */
  int32_t num_charge_states;        /* tunnel: basis size (32)                                            */
  int32_t charge_state_batch_size;  /* tunnel: chunk of the candidate scan (1000), 0 = unchunked          */
} qd_model_desc;

/* One scan window: v(ix, iy) = v0 + ix*dx + iy*dy over all n_volt voltages -- the affine form of
 * GateVoltageComposer.do2d / meshgrid_virtual_coupled (GateVoltageComposer.py:170-211, 224-255); for the tunnel
 * path the barrier voltages are the trailing entries of v0 with dx = dy = 0 (qarray_base_class.py:160). */
typedef struct qd_scan {
  double v0[QD_MAX_VOLT];
  double dx[QD_MAX_VOLT];
  double dy[QD_MAX_VOLT];
  double peak_width;        /* coulomb_peak_width, mutable per scan (qarray_base_class.py:192-196)        */
  double rad_x0, rad_dx;    /* pixel-to-ground-truth offset along x: x0 + ix*dx (qarray_base_class.py:476) */
  double rad_y0, rad_dy;
  double rad_alpha, rad_zero_radius, rad_max_amp;
  uint64_t seed;            /* Philox key of this scan                                                    */
  int64_t pix_offset;       /* index (in pixels) of this scan's first pixel inside z_out / n_out          */
  int32_t env_id;
  int32_t nx, ny;
  int32_t rad_mode;         /* 0 off, 1 additive, 2 replace the scan by unit white noise (:463-468)       */
} qd_scan;

int qd_abi_version(void);

/* One context per (process, device). */
int qd_create(int device, qd_ctx** out);
void qd_destroy(qd_ctx* ctx);
const char* qd_last_error(const qd_ctx* ctx);   /* ctx-owned, valid until the next call on ctx; ctx may be NULL */

/* Upload the per-env constants (HOST pointers; copied).  Replaces the Maxwell matrices held by a
 * ChargeSensedDotArray / TunnelCoupledChargeSensed instance (TunnelCoupledChargeSensed.py:94-143).
 *   cdd_inv_gs   [n_env, N, N]  matrix of the ground-state quadratic form: the dot-only cdd_inv for Path A,
 *                               cdd_inv_full[:N,:N] for the tunnel path (ground_state.py:60-65, charge_states.py:61-76)
 *   cdd_gs       [n_env, N, N]  dot-only Maxwell cdd (inverse of the above; M-matrix) -- Path A relaxation; may be
 *                               NULL for QD_ALG_TUNNEL / QD_ALG_BRUTE_FORCE
 *   cdd_inv_full [n_env, D, D]  D = N + n_sensor
 *   cgd_full     [n_env, D, n_volt]   rows [:N] are also the ground-state cgd
 *   cbg          [n_env, B, n_gate]   raw positive barrier-gate matrix (barrier_voltage_model.py:129) or NULL
 *   params       [n_env]
 *
 * Several charge sensors (n_sensor = S > 1; qarray's ChargeSensedDotArray with an (S, n_dot) Cds).  Every sensor output
 * z_out / z_out_host below is then float [pixels, S], pixel-major like n_out: scan i's block starts at element
 * pix_offset_i * S.  With S = 1 this is the one-float-per-pixel layout.  Sensor s at a pixel, with u = cgd_full v,
 * dot residuals e_j = n_j - u_j, t_o = rint(u_{N+o}) + xi_o - u_{N+o} for every sensor o (xi_o: sensor o's input
 * noise) and C = cdd_inv_full:
 *     dPhi_k = C_ss (2 (t_s + k) + 1) + 2 sum_j C_{s,j} e_j + 2 sum_{o != s} C_{s,o} t_o,   k = -5..4
 *     z_s    = sum_k 1 / (1 + (dPhi_k / gamma)^2) + eta_s
 * (sensor s perturbed, the others at their rounded, noisy occupations; indices s, o of C count from row N).  Each sensor
 * draws its own white, telegraph and 1/f noise with the env's amplitudes and probabilities: Philox counter word c3 =
 * sensor index for every stream purpose, so sensor 0 draws what a one-sensor model draws.  The latching uniform is per
 * pixel (sensor 0's block).  Radial noise: mode 1 adds z_rad,s * amp(ix, iy) to channel s (one amplitude map, each
 * channel's own normal), mode 2 replaces channel s by its own unit normal.  QD_FLAG_WHITE_ON_OUTPUT moves each sensor's
 * white noise to its own eta_s.  Limits: n_volt <= QD_MAX_VOLT still holds (the tunnel path with barriers: 2N + S - 1
 * <= 16).  A device z_out of a two- or four-sensor set must be aligned to 4 S bytes (one vector store per pixel).
 * qd_scan_obs_host (the one-sensor observation of the env) returns QD_ERR_UNSUPPORTED for S > 1.
 */
int qd_set_models(qd_ctx* ctx, const qd_model_desc* desc, const double* cdd_inv_gs, const double* cdd_gs,
                  const double* cdd_inv_full, const double* cgd_full, const double* cbg,
                  const qd_env_params* params);

/* Simulate n_scan scan windows in one launch.  Replaces, per scan, ChargeSensedDotArray.do2d_open /
 * TunnelCoupledChargeSensed.charge_sensor_open + QarrayBaseClass._apply_radial_noise
 * (qarray_base_class.py:128-139, 163, 202-206).
 *   scans   HOST pointer, [n_scan]; copied to the device inside the call (stream-ordered)
 *   z_out   DEVICE pointer, float [total pixels, n_sensor]: scan i occupies pixels [pix_offset_i, pix_offset_i + nx_i*ny_i),
 *           row-major (iy, ix), fast axis x (sizeof(qd_scan) is 480, a multiple of 16: staged by one TMA bulk copy)
 *   n_out   DEVICE pointer or NULL, element type n_type, [pixels, N]
 *   stream  cudaStream_t (NULL = default stream).  Asynchronous: returns after enqueueing.
 */
int qd_scan_open(qd_ctx* ctx, int n_scan, const qd_scan* scans, float* z_out, void* n_out, int n_type,
                 unsigned flags, void* stream);

/* The two halves of qd_scan_open, for callers that reuse one set of descriptors (bench.py's HBM-resident timing,
 * CUDA-graph capture): qd_scan_upload validates and copies the descriptors into the context (stream-ordered);
 * qd_scan_launch enqueues one launch over the descriptors uploaded last. */
int qd_scan_upload(qd_ctx* ctx, int n_scan, const qd_scan* scans, void* stream);
int qd_scan_launch(qd_ctx* ctx, float* z_out, void* n_out, int n_type, unsigned flags, void* stream);

/* Same, with HOST output buffers: runs the launch, copies the results back and synchronises. This is the call the
 * drop-in Python classes make for a single do2d_open. */
int qd_scan_open_host(qd_ctx* ctx, int n_scan, const qd_scan* scans, float* z_out_host, void* n_out_host,
                      int n_type, unsigned flags);

/* Arbitrary voltage list (the escape hatch behind ground_state_open(vg) / charge_sensor_open(vg[, vb]) called with
 * an explicit array, TunnelCoupledChargeSensed.py:312-380).  HOST buffers.
 *   v       [ny*nx, n_volt]   (gate voltages followed by barrier voltages)
 *   z_out   float [ny*nx, n_sensor] or NULL;  n_out [ny*nx, N] of n_type or NULL
 *   (ny, nx) = measurement shape: latching / telegraph run along nx.
 * `scan` supplies env_id, peak_width, seed and the radial fields; its v0/dx/dy/nx/ny are ignored. */
int qd_points_open_host(qd_ctx* ctx, const qd_scan* scan, int ny, int nx, const double* v, float* z_out_host,
                        void* n_out_host, int n_type, unsigned flags);

/* Closed arrays: a fixed total number of carriers per scan, n_charge = sum of the dot occupations (ChargeSensedDotArray's
 * closed methods, qarray 1.6.0).  The ground state is the closed form of the model set's algorithm: the minimiser of the
 * free energy over the charge configurations with sum n = n_charge -- `default`: floor of the exact closed relaxation
 * (n >= 0, sum n = n_charge) plus {0,1}^N, kept where the sum is n_charge; `brute_force`: every n in {0..n_charge}^N of that
 * sum (max_charge_carriers unused).  Latching, sensor, noise and radial noise are those of the open path.  Same model set
 * as the open entry points (qd_set_models); QD_ERR_UNSUPPORTED for QD_ALG_THRESHOLDED and QD_ALG_TUNNEL, QD_ERR_INVALID for
 * an n_charge outside 0..251 (default) / 0..15 (brute_force).
 *   n_charge  HOST, [n_scan]: total charge of each scan; copied to the device next to the descriptors (stream-ordered) */

/* Replaces, per scan, ChargeSensedDotArray.do2d_closed (+ QarrayBaseClass._apply_radial_noise).  Asynchronous, DEVICE
 * outputs, as qd_scan_open. */
int qd_scan_closed(qd_ctx* ctx, int n_scan, const qd_scan* scans, const int32_t* n_charge, float* z_out, void* n_out,
                   int n_type, unsigned flags, void* stream);

/* ChargeSensedDotArray.do2d_closed with HOST outputs, as qd_scan_open_host. */
int qd_scan_closed_host(qd_ctx* ctx, int n_scan, const qd_scan* scans, const int32_t* n_charge, float* z_out_host,
                        void* n_out_host, int n_type, unsigned flags);

/* ChargeSensedDotArray.ground_state_closed / charge_sensor_closed / do1d_closed on an explicit voltage list, as
 * qd_points_open_host, with the one total charge n_charge. */
int qd_points_closed_host(qd_ctx* ctx, const qd_scan* scan, int32_t n_charge, int ny, int nx, const double* v,
                          float* z_out_host, void* n_out_host, int n_type, unsigned flags);

/* Percentile normalisation of the observation images, per env (K8; replaces QuantumDeviceEnv._normalise_obs,
 * src/qadapt/environment/env.py:471-509): for each of n_env consecutive blocks of per_env floats,
 *   p_low, p_high = np.percentile(block, q_low_pct), np.percentile(block, q_high_pct)   (numpy 'linear' method)
 *   out = clip((block - p_low) / (p_high - p_low), 0, 1)   or zeros when p_high <= p_low
 * z and out are DEVICE pointers (out may alias z); stats (DEVICE, [n_env, 2] doubles: p_low, p_high) may be NULL.
 * Asynchronous on `stream`. */
int qd_normalise_obs(qd_ctx* ctx, const float* z, float* out, int64_t per_env, int n_env, double q_low_pct,
                     double q_high_pct, double* stats, void* stream);

/* qd_normalise_obs with a typed output (enum qd_ztype): out holds n_env * per_env elements of z_type, each the fp64
 * value x above rounded as QD_Z_F32 = (float)x, QD_Z_F16 = half((float)x), QD_Z_U8 = rint(255 * x).  z, out, stats
 * are DEVICE pointers. */
int qd_normalise_obs_typed(qd_ctx* ctx, const float* z, void* out, int z_type, int64_t per_env, int n_env,
                           double q_low_pct, double q_high_pct, double* stats, void* stream);

/* The observation of one batched env.step, delivered to HOST memory in a compact element type: simulate the scans
 * (as qd_scan_open_host), optionally percentile-normalise per env on the device (QuantumDeviceEnv._normalise_obs,
 * env.py:471-509 -- what the policy is fed), convert to z_type and copy back; chunks of envs are pipelined so that the
 * copy of one chunk overlaps the kernels of the next.
 *   scans          env-major: scans_per_env consecutive descriptors per env, all of one size, pix_offset = i * nx * ny
 *   out_host       [n_scan * ny * nx] elements of z_type (pinned memory for full copy speed); one-sensor model sets only
 *   normalise      0: raw sensor signal (QD_Z_F32 / QD_Z_F16 only); 1: percentile-normalised to [0, 1]
 *   stats_host     [n_scan / scans_per_env, 2] doubles (p_low, p_high per env) or NULL
 */
int qd_scan_obs_host(qd_ctx* ctx, int n_scan, const qd_scan* scans, int scans_per_env, void* out_host, int z_type,
                     int normalise, double q_low_pct, double q_high_pct, double* stats_host, unsigned flags);

/* Sticky status bits (QD_STATUS_*) raised by the kernels of this context; `clear` != 0 resets them.  The *_host entry
 * points check it themselves and return QD_ERR_INVALID; callers of the asynchronous entry points call this after
 * synchronising their stream. */
int qd_status(qd_ctx* ctx, int clear);

/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
int64_t qd_launch_count(const qd_ctx* ctx);

/* FP64 FMA micro-benchmark used as the roofline denominator of this FP-pipe-bound path: runs `iters` dependent-free
 * DFMA chains on every SM and returns achieved TFLOP/s in *tflops (device-timed). */
int qd_measure_fp64_peak(qd_ctx* ctx, int iters, double* tflops);
int qd_measure_fp32_peak(qd_ctx* ctx, int iters, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* QDSIM_H */
