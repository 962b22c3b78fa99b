// qd_api.cu -- the C ABI of libqdsim.so (include/qdsim.h): context, model upload, launches.
// No torch, no C++ types across the boundary; every entry point returns a qd_err.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <new>
#include <stdlib.h>

#include <algorithm>
#include <chrono>
#include <type_traits>
#include <vector>

#include "qd_kernels.cuh"
#include "qd_tunnel.cuh"
#include "qd_tunnel_noda.cuh"
#include "qd_tunnel_enum.cuh"
#include "qd_normalise.cuh"

static_assert(sizeof(qd_scan) == 480, "qd_scan must be 480 bytes (multiple of 16 for the TMA bulk copy)");
static_assert(sizeof(qd_scan) % 16 == 0, "qd_scan size");

struct qd_ctx {
  int device = 0;
  int sm_count = 0;
  char err[512] = {0};
  bool have_models = false;
  qd_layout L{};
  int n_env = 0;
  double* d_records = nullptr;
  size_t records_bytes = 0;
  // staging for scan descriptors
  qd_scan* d_scans = nullptr;
  size_t scans_cap = 0;
  qd_scan* h_scans = nullptr;   // pinned
  size_t h_scans_cap = 0;
  // scratch for the *_host entry points
  float* d_z = nullptr;
  size_t z_cap = 0;
  void* d_n = nullptr;
  size_t n_cap = 0;
  double* d_pts = nullptr;
  size_t pts_cap = 0;
  double* d_nbar = nullptr;       // tunnel path: <n> of every pixel between the two launches
  size_t nbar_cap = 0;
  unsigned char* d_tfloor = nullptr;   // tunnel path, split pipeline: floor(n_c) of the current chunk, 8 bytes per pixel
  size_t tfloor_cap = 0;
  double* d_tpot = nullptr;            // same chunk: dot potentials [8], tunnel couplings [7], cdd scale: 128 bytes per pixel
  size_t tpot_cap = 0;
  unsigned long long* d_tkeys = nullptr;   // ... and its 32 kept basis states, 256 bytes per pixel
  size_t tkeys_cap = 0;
  void* d_obs = nullptr;          // qd_scan_obs_host: compact (typed) observation images before the copy-back
  size_t obs_cap = 0;
  double* d_stats = nullptr;      // qd_scan_obs_host: per-env (p_low, p_high)
  size_t stats_cap = 0;
  unsigned* h_status = nullptr;   // sticky QD_STATUS_* word: mapped pinned host memory, kernels write it on errors only
  unsigned* d_status = nullptr;   // its device alias
  unsigned char* h_small = nullptr;   // mapped pinned output buffer of the small-call fast path (kernel writes it directly)
  unsigned char* d_small = nullptr;   // its device alias
  size_t small_cap = 0;
  cudaEvent_t last_launch = nullptr;  // recorded after every launch: the context's scratch (d_scans, d_nbar) is free
  cudaStream_t last_stream = nullptr; //   for a launch on ANOTHER stream only once this has fired
  bool have_last = false;
  bool staged_pending = false;    // an asynchronous H2D out of h_scans may still be in flight
  cudaEvent_t staged = nullptr;   // h_scans may be rewritten once this has fired
  cudaStream_t s_compute = nullptr, s_copy = nullptr;   // qd_scan_open_host: launches / result copies, overlapped
  cudaEvent_t chunk_done[16] = {nullptr};
  int up_n_scan = 0;              // descriptors currently resident in d_scans
  int up_max_ny = 0;
  long long up_pixels = 0;        // extent of the output buffers they address
  long long up_max_pix = 0;       // largest scan, in pixels
  int64_t launches = 0;
  // QDSIM_TRACE=1: accumulated host-side phases of the small-call path (setup+launch, sync, copy-out), printed at destroy
  double tr_launch = 0, tr_sync = 0, tr_copy = 0;
  long tr_calls = 0;
};

namespace {

char g_err[512] = "no context";

int fail(qd_ctx* ctx, int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(ctx ? ctx->err : g_err, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define QD_CUDA(ctx, call)                                                                      \
  do {                                                                                          \
    cudaError_t e_ = (call);                                                                    \
    if (e_ != cudaSuccess)                                                                      \
      return fail(ctx, QD_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

template <typename T>
int grow(qd_ctx* ctx, T** p, size_t* cap, size_t need_bytes) {
  if (*cap >= need_bytes) return QD_OK;
  if (*p) cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  size_t want = need_bytes + need_bytes / 4 + 256;
  cudaError_t e = cudaMalloc((void**)p, want);
  if (e != cudaSuccess) return fail(ctx, QD_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
  *cap = want;
  return QD_OK;
}

size_t n_elem_size(int n_type) {
  switch (n_type) {
    case QD_N_U8: return 1;
    case QD_N_F32: return 4;
    case QD_N_F64: return 8;
    default: return 0;
  }
}

using kernel_fn = void (*)(const qd::KArgs);

// The instance of a kernel template for n_dot = n: `k` maps std::integral_constant<int, N> to the instance for N dots.
// Only MIN_N..QD_MAX_DOTS are instantiated; any other n gives nullptr.
template <int MIN_N, int N = QD_MAX_DOTS, typename F>
kernel_fn pick_dots(int n, F k) {
  if constexpr (N < MIN_N) return nullptr;
  else return n == N ? k(std::integral_constant<int, N>{}) : pick_dots<MIN_N, N - 1>(n, k);
}

// default / thresholded search with a hard argmin on affine windows runs the restructured kernel (qd_scan_fast_kernel);
// QDSIM_GENERIC_SCAN=1 keeps the generic one (A/B timing, and the parity tests run both)
bool use_fast_kernel(const qd_layout& L, unsigned flags, bool points) {
  if (points || (flags & (QD_FLAG_THERMAL | QD_FLAG_PINK))) return false;
  if (L.algorithm != QD_ALG_DEFAULT && L.algorithm != QD_ALG_THRESHOLDED) return false;
  const char* e = getenv("QDSIM_GENERIC_SCAN");
  return !(e && e[0] == '1');
}

template <int ALG, bool THERMAL>
kernel_fn pick_p(int n, bool points) {
  if (points) return pick_dots<1>(n, [](auto k) { return qd::qd_scan_kernel<decltype(k)::value, ALG, THERMAL, true>; });
  return pick_dots<1>(n, [](auto k) { return qd::qd_scan_kernel<decltype(k)::value, ALG, THERMAL, false>; });
}

kernel_fn pick_kernel(const qd_layout& L, unsigned flags, bool points) {
  const bool thermal = flags & QD_FLAG_THERMAL;
  if (L.algorithm == QD_ALG_TUNNEL) return pick_p<QD_ALG_TUNNEL, false>(L.n_dot, points);
  if (L.algorithm == QD_ALG_BRUTE_FORCE)
    return thermal ? pick_p<QD_ALG_BRUTE_FORCE, true>(L.n_dot, points) : pick_p<QD_ALG_BRUTE_FORCE, false>(L.n_dot, points);
  if (L.algorithm == QD_ALG_DEFAULT || L.algorithm == QD_ALG_THRESHOLDED)
    return thermal ? pick_p<QD_ALG_DEFAULT, true>(L.n_dot, points) : pick_p<QD_ALG_DEFAULT, false>(L.n_dot, points);
  return nullptr;
}

int validate_launch(qd_ctx* ctx, int n_type, unsigned flags, const void* n_out) {
  if (!ctx) return fail(nullptr, QD_ERR_INVALID, "ctx is NULL");
  if (!ctx->have_models) return fail(ctx, QD_ERR_STATE, "qd_set_models has not been called");
  if (n_type < QD_N_NONE || n_type > QD_N_F64) return fail(ctx, QD_ERR_INVALID, "bad n_type %d", n_type);
  if (n_type != QD_N_NONE && !n_out) return fail(ctx, QD_ERR_INVALID, "n_out is NULL but n_type != QD_N_NONE");
  if ((flags & QD_FLAG_THERMAL) && n_type == QD_N_U8)
    return fail(ctx, QD_ERR_INVALID, "QD_FLAG_THERMAL yields non-integer occupations: use QD_N_F32/F64 or QD_N_NONE");
  // QD_FLAG_LATCH_EXACT: with integer occupations (hard argmin) the raw and the rounded compare coincide, so the flag
  // is accepted and changes nothing; on non-integer occupations (thermal average, tunnel path) the kernel only has the
  // rounded compare -- refuse instead of silently answering a different question.
  if ((flags & QD_FLAG_LATCH) && (flags & QD_FLAG_LATCH_EXACT) &&
      ((flags & QD_FLAG_THERMAL) || ctx->L.algorithm == QD_ALG_TUNNEL))
    return fail(ctx, QD_ERR_UNSUPPORTED,
                "QD_FLAG_LATCH_EXACT: exact-compare latching of non-integer occupations (thermal / tunnel path) is not supported");
  if (ctx->L.algorithm == QD_ALG_TUNNEL && n_type == QD_N_U8)
    return fail(ctx, QD_ERR_INVALID, "the tunnel path yields non-integer occupations <n>: use QD_N_F32/F64 or QD_N_NONE");
  return QD_OK;
}

// shared-memory attributes of a kernel: set once per context (two driver calls saved per launch)
// Function attributes belong to the CUDA context of a device, not to a qd_ctx: the table is process-wide, keyed by
// (device, kernel), and the dynamic size only ever grows (two qd_ctx of one process must not lower each other's setting).
struct KernelConfig { int device; const void* fn; size_t smem; };
KernelConfig g_kernel_config[512];
int g_n_kernel_config = 0;

int configure_kernel(qd_ctx* ctx, const void* fn, size_t smem) {
  int at = -1;
  for (int i = 0; i < g_n_kernel_config; ++i)
    if (g_kernel_config[i].fn == fn && g_kernel_config[i].device == ctx->device) { at = i; break; }
  if (at >= 0 && g_kernel_config[at].smem >= smem) return QD_OK;
  const size_t want = std::max<size_t>(smem, 48 * 1024);
  QD_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)want));
  // every warp stages its own record: ask for the largest shared-memory carveout so that registers, not shared
  // memory, bound the resident warps
  if (at < 0) QD_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  if (at < 0 && g_n_kernel_config < 512) at = g_n_kernel_config++;
  if (at >= 0) g_kernel_config[at] = KernelConfig{ctx->device, fn, want};
  return QD_OK;
}

// Enqueue one kernel: configured first if it takes dynamic shared memory (the others keep the driver's defaults), the
// grid clamped to what one launch takes, the launch checked and counted in ctx->launches.
template <typename... P, typename... A>
int issue(qd_ctx* ctx, void (*fn)(P...), long long grid, int threads, size_t smem, cudaStream_t stream, const A&... args) {
  if (smem) {
    const int rc = configure_kernel(ctx, (const void*)fn, smem);
    if (rc) return rc;
  }
  fn<<<(unsigned)std::min(grid, 0x7fffffffLL), threads, smem, stream>>>(args...);
  QD_CUDA(ctx, cudaGetLastError());
  ctx->launches += 1;
  return QD_OK;
}

// The context's scratch buffers (d_scans, d_nbar) are shared by all launches.  A launch on stream B that follows one on
// stream A must not re-stage them before A's kernels are done with them: every launch records `last_launch`, and work
// enqueued on a different stream waits for it first (same stream: already ordered, no call made).
int order_after_last_launch(qd_ctx* ctx, cudaStream_t stream) {
  if (ctx->have_last && ctx->last_stream != stream) QD_CUDA(ctx, cudaStreamWaitEvent(stream, ctx->last_launch, 0));
  return QD_OK;
}
int mark_launch(qd_ctx* ctx, cudaStream_t stream) {
  QD_CUDA(ctx, cudaEventRecord(ctx->last_launch, stream));
  ctx->last_stream = stream;
  ctx->have_last = true;
  return QD_OK;
}

// Items of the warp-per-pixel tunnel kernels over a.n_scan scans of <= max_pix pixels: <= 64 consecutive pixels of one
// scan each (the warm start runs along an item), about four per warp resident at `warps_per_sm` warps per SM; one warp
// per CTA while four would leave SMs idle.  Sets a.rows_per_item (pixels per item) and a.items_per_scan.
struct PixelItems { int warps; long long grid; };
PixelItems plan_pixel_items(const qd_ctx* ctx, qd::KArgs& a, long long max_pix, int warps_per_sm) {
  const long long want_items = (long long)ctx->sm_count * warps_per_sm * 4;
  const long long ppi = std::min<long long>(std::max<long long>(((long long)a.n_scan * max_pix) / want_items, 1), 64);
  a.rows_per_item = (int)ppi;
  a.items_per_scan = (int)((max_pix + ppi - 1) / ppi);
  const long long items = (long long)a.n_scan * a.items_per_scan;
  const int warps = (items < (long long)ctx->sm_count * 4) ? 1 : 4;
  return {warps, (items + warps - 1) / warps};
}

// One stage of the split tunnel pipeline: a primary kernel and the older kernel it falls back on.  `primary` (nullptr
// when it does not apply or a switch turns it off) runs with the arguments `pa` and marks the pixels it could not do;
// `fallback` then redoes only those (fix-up mode), or does every pixel when there is no primary.  fix = false skips
// the second launch and leaves the marks in place.  `g` holds the items of plan_pixel_items.
int primary_then_fixup(qd_ctx* ctx, const qd::KArgs& g, const PixelItems& p, kernel_fn primary, const qd::KArgs& pa,
                       kernel_fn fallback, int fallback_slot_bytes, bool fix, cudaStream_t stream) {
  if (primary) {
    const int rc = issue(ctx, primary, p.grid, p.warps * 32, (size_t)pa.slot_bytes * p.warps, stream, pa);
    if (rc) return rc;
  }
  if (!fix) return QD_OK;
  qd::KArgs fa = g;
  fa.slot_bytes = fallback_slot_bytes;
  long long grid = p.grid;
  if (primary) {
    // items of 8 pixels (no state is carried between marked pixels), so that a stretch of marked pixels is spread over
    // several warps; mark_ppi carries the marking kernel's item length to the mark look-up
    fa.fixup = 1;
    fa.mark_ppi = g.rows_per_item;
    fa.rows_per_item = (g.rows_per_item % 8 == 0) ? 8 : g.rows_per_item;   // (must divide the marking kernel's item length)
    fa.items_per_scan = (int)((ctx->up_max_pix + fa.rows_per_item - 1) / fa.rows_per_item);
    grid = ((long long)fa.n_scan * fa.items_per_scan + p.warps - 1) / p.warps;
    // (almost every item is skipped on its mark: a resident-size grid looping over the items instead of one CTA per four)
    grid = std::min<long long>(grid, (long long)ctx->sm_count * 32);
  }
  return issue(ctx, fallback, grid, p.warps * 32, (size_t)fa.slot_bytes * p.warps, stream, fa);
}

// Path B: the tunnel-coupled ground state <n> of every pixel into d_nbar, for the scan kernel's latching / sensor / noise
int tunnel_ground_state(qd_ctx* ctx, int n_scan, const qd_scan* d_scans, const double* d_points, unsigned flags,
                        cudaStream_t stream) {
  const int N = ctx->L.n_dot;
  const kernel_fn gs = pick_dots<2>(N, [](auto n) { return qd::qd_tunnel_gs_kernel<decltype(n)::value>; });
  if (!gs) return fail(ctx, QD_ERR_UNSUPPORTED, "tunnel path needs 2..8 dots, got %d", N);
  int rc = grow(ctx, &ctx->d_nbar, &ctx->nbar_cap, (size_t)ctx->up_pixels * N * sizeof(double));
  if (rc) return rc;
  qd::KArgs g;
  memset(&g, 0, sizeof(g));
  g.L = ctx->L; g.records = ctx->d_records; g.scans = d_scans; g.points = d_points; g.z_out = nullptr;
  g.n_out = nullptr; g.nbar = ctx->d_nbar; g.n_scan = n_scan; g.n_type = QD_N_NONE; g.flags = flags;
  g.status = ctx->d_status;
  g.topt = 7;
  if (const char* e = getenv("QDSIM_TUNNEL_OPT")) g.topt = atoi(e) & 7;
  const long long max_pix = ctx->up_max_pix;
  const char* mono_e = getenv("QDSIM_TUNNEL_MONO");
  if (mono_e && mono_e[0] == '1') {
    // the single-kernel form (one warp per pixel does everything): kept as the A/B reference of the split pipeline
    g.slot_bytes = qd::qd_tunnel_slot_bytes(ctx->L);
    const PixelItems p = plan_pixel_items(ctx, g, max_pix, 12);
    return issue(ctx, gs, p.grid, p.warps * 32, (size_t)g.slot_bytes * p.warps, stream, g);
  }
  // split pipeline R -> S -> E over chunks of scans (8 + 128 + 256 bytes of scratch per pixel of a chunk)
  const kernel_fn kr = pick_dots<2>(N, [](auto n) { return qd::qd_tunnel_relax_kernel<decltype(n)::value>; });
  const kernel_fn ks = pick_dots<2>(N, [](auto n) { return qd::qd_tunnel_select_kernel<decltype(n)::value>; });
  const kernel_fn ke = pick_dots<2>(N, [](auto n) { return qd::qd_tunnel_eigen_kernel<decltype(n)::value>; });
  // S: the lattice-enumeration kernel first (four dots and more: fewer than 32 candidates can be valid below four dots,
  // and the block walk pads; QDSIM_SELECT=block skips it), then the block walk -- as the fix-up pass over the pixels the
  // enumeration marked, or for everything
  const char* sel_e = getenv("QDSIM_SELECT");
  const kernel_fn ks2 = (sel_e && sel_e[0] == 'b')
                            ? nullptr
                            : pick_dots<4>(N, [](auto n) { return qd::qd_tunnel_select2_kernel<decltype(n)::value>; });
  // E: the Noda-iteration kernel first (QDSIM_EIGEN=householder skips it); what it could not do (sectors of more
  // than 16 states, no convergence) is marked with a NaN and redone by the Householder kernel in fix-up mode
  const char* eig_e = getenv("QDSIM_EIGEN");
  const bool no_fixup = eig_e && eig_e[0] == 'n';          // (measurement only: leaves the NaN marks in place)
  const kernel_fn ke2 = (eig_e && eig_e[0] == 'h')
                            ? nullptr
                            : pick_dots<2>(N, [](auto n) { return qd::qd_tunnel_eigen2_kernel<decltype(n)::value>; });
  long long chunk_pix = 8LL << 20;
  if (const char* e = getenv("QDSIM_TUNNEL_CHUNK_PIX")) chunk_pix = atoll(e) > 0 ? atoll(e) : chunk_pix;
  const long long spc = std::min<long long>(std::max<long long>(chunk_pix / max_pix, 1), n_scan);   // scans per chunk
  rc = grow(ctx, &ctx->d_tfloor, &ctx->tfloor_cap, (size_t)spc * max_pix * 8);
  if (rc) return rc;
  rc = grow(ctx, &ctx->d_tkeys, &ctx->tkeys_cap, (size_t)spc * max_pix * 256);
  if (rc) return rc;
  rc = grow(ctx, &ctx->d_tpot, &ctx->tpot_cap, (size_t)spc * max_pix * 128);
  if (rc) return rc;
  g.tfloor = ctx->d_tfloor;
  g.tpot = ctx->d_tpot;
  g.tkeys = ctx->d_tkeys;
  g.tstride = max_pix;
  for (long long c0 = 0; c0 < n_scan; c0 += spc) {
    g.scans = d_scans + c0;
    g.n_scan = (int)std::min<long long>(spc, n_scan - c0);
    // R: one thread per pixel, a CTA per <= 1024 pixels of one scan
    qd::KArgs r = g;
    r.rows_per_item = (int)std::min<long long>(1024, max_pix);
    r.items_per_scan = (int)((max_pix + r.rows_per_item - 1) / r.rows_per_item);
    rc = issue(ctx, kr, (long long)r.n_scan * r.items_per_scan, 128, qd::qd_tunnel_relax_smem_bytes(ctx->L), stream, r);
    if (rc) return rc;
    // S and E: one warp per pixel
    const PixelItems p = plan_pixel_items(ctx, g, max_pix, 16);
    qd::KArgs sa = g;
    sa.slot_bytes = qd::qd_tunnel_select2_slot_bytes(ctx->L);
    rc = primary_then_fixup(ctx, g, p, ks2, sa, ks, qd::qd_tunnel_select_slot_bytes(ctx->L), true, stream);
    if (rc) return rc;
    qd::KArgs ea = g;
    ea.e2_kappa = 4.0f; ea.e2_qsafe = 4.0f; ea.e2_tol = 2e-10f;
    if (const char* e = getenv("QDSIM_E2_KAPPA")) ea.e2_kappa = (float)atof(e);
    if (const char* e = getenv("QDSIM_E2_QSAFE")) ea.e2_qsafe = (float)atof(e);
    if (const char* e = getenv("QDSIM_E2_TOL")) ea.e2_tol = (float)atof(e);
    ea.slot_bytes = qd::qd_tunnel_eigen2_slot_bytes(ctx->L);
    rc = primary_then_fixup(ctx, g, p, ke2, ea, ke, qd::qd_tunnel_eigen_slot_bytes(ctx->L), !no_fixup, stream);
    if (rc) return rc;
  }
  return QD_OK;
}

// enqueue one launch over device-resident descriptors
int launch(qd_ctx* ctx, int n_scan, const qd_scan* d_scans, int max_ny, const double* d_points, float* d_z, void* d_n,
           int n_type, unsigned flags, cudaStream_t stream, int rows_cap = 0, const qd_scan* h_one = nullptr) {
  int rc = order_after_last_launch(ctx, stream);     // the scratch of an earlier launch on another stream
  if (rc) return rc;
  const bool fast = use_fast_kernel(ctx->L, flags, d_points != nullptr);
  const kernel_fn fn =
      fast ? pick_dots<1>(ctx->L.n_dot, [](auto n) { return qd::qd_scan_fast_kernel<decltype(n)::value>; })
           : pick_kernel(ctx->L, flags, d_points != nullptr);
  if (!fn) return fail(ctx, QD_ERR_UNSUPPORTED, "no kernel for n_dot=%d algorithm=%d", ctx->L.n_dot, ctx->L.algorithm);
  qd::KArgs a;
  memset(&a, 0, sizeof(a));
  if (ctx->L.algorithm == QD_ALG_TUNNEL) {
    // the tunnel-coupled ground state first; the scan kernel below reads it from d_nbar
    rc = tunnel_ground_state(ctx, n_scan, d_scans, d_points, flags, stream);
    if (rc) return rc;
    a.nbar = ctx->d_nbar;
  }
  a.L = ctx->L;
  a.records = ctx->d_records;
  a.scans = d_scans;
  a.points = d_points;
  a.z_out = d_z;
  a.n_out = (n_type == QD_N_NONE) ? nullptr : d_n;
  a.n_scan = n_scan;
  a.n_type = n_type;
  a.flags = flags;
  a.status = ctx->d_status;
  if (h_one && ctx->L.algorithm != QD_ALG_TUNNEL) { a.use_one = 1; a.one = *h_one; }
  a.slot_bytes = fast ? qd::qd_fast_slot_bytes(ctx->L) : qd::qd_slot_bytes(ctx->L);
  // item = block of rows of one scan handled by one warp.  Large batches: one scan per warp (staging amortised over
  // the whole scan).  Small batches: split rows so that every SM gets work.  A flat (carry-rows) pass is sequential
  // over the whole scan by definition.
  const long long target_items = (long long)ctx->sm_count * (fast ? 16 : 12) * 4;
  long long rows = ((long long)n_scan * max_ny) / target_items;
  if (rows < 1) rows = 1;
  if (rows > max_ny) rows = max_ny;
  // a pipelined caller launches several times per batch: shorter items keep the idle tail of each launch short
  if (rows_cap > 0 && rows > rows_cap) rows = rows_cap;
  if (flags & QD_FLAG_CARRY_ROWS) rows = max_ny;
  a.rows_per_item = (int)rows;
  a.items_per_scan = (max_ny + a.rows_per_item - 1) / a.rows_per_item;
  // A launch too small to give every SM a warp (a single do2d_open) is also split ALONG the rows when no state is carried
  // from pixel to pixel (no latching, telegraph or 1/f chain): each item is then one 32-pixel chunk.
  a.col_parts = 1;
  if (!(flags & (QD_FLAG_LATCH | QD_FLAG_NOISE | QD_FLAG_PINK | QD_FLAG_CARRY_ROWS)) && rows == 1 &&
      (long long)n_scan * a.items_per_scan < (long long)ctx->sm_count) {
    const long long chunks_x = (ctx->up_max_pix / std::max(1, max_ny) + 31) / 32;      // 32-pixel chunks per row of the largest scan
    long long cp = (long long)ctx->sm_count * 2 / std::max<long long>(1, (long long)n_scan * a.items_per_scan);
    cp = std::min<long long>(std::max<long long>(cp, 1), std::max<long long>(chunks_x, 1));
    a.col_parts = (int)cp;
    a.items_per_scan *= a.col_parts;
  }
  const long long total_items = (long long)n_scan * a.items_per_scan;
  // warps per CTA: the warps of a CTA are independent, but a CTA's slot (registers, shared memory) is only released when
  // its SLOWEST warp is done; scans differ in work (Gray-walk widths, latching events), so the restructured kernel runs
  // one warp per CTA and lets the hardware scheduler balance (16 CTAs of 11.9 KB per SM).  QDSIM_WPC overrides (A/B).
  int wpc = (total_items < (long long)ctx->sm_count * 4) ? 1 : (fast ? 1 : QD_CTA_WARPS);
  if (const char* e = getenv("QDSIM_WPC")) { const int v = atoi(e); if (v == 1 || v == 2 || v == 4) wpc = v; }
  rc = issue(ctx, fn, (total_items + wpc - 1) / wpc, wpc * 32, (size_t)a.slot_bytes * wpc, stream, a);
  if (rc) return rc;
  return mark_launch(ctx, stream);
}

int check_scan(qd_ctx* ctx, int i, const qd_scan& s) {
  if (s.env_id < 0 || s.env_id >= ctx->n_env)
    return fail(ctx, QD_ERR_INVALID, "scan %d: env_id %d out of range [0,%d)", i, s.env_id, ctx->n_env);
  if (s.nx <= 0 || s.ny <= 0) return fail(ctx, QD_ERR_INVALID, "scan %d: nx, ny must be positive", i);
  if (s.pix_offset < 0) return fail(ctx, QD_ERR_INVALID, "scan %d: negative pix_offset", i);
  return QD_OK;
}

int stage_scans(qd_ctx* ctx, int n_scan, const qd_scan* scans, cudaStream_t stream, int* max_ny,
                bool caller_syncs = false) {
  if (n_scan <= 0) return fail(ctx, QD_ERR_INVALID, "n_scan must be positive");
  if (!scans) return fail(ctx, QD_ERR_INVALID, "scans is NULL");
  const size_t bytes = (size_t)n_scan * sizeof(qd_scan);
  int rc = grow(ctx, &ctx->d_scans, &ctx->scans_cap, bytes);
  if (rc) return rc;
  rc = order_after_last_launch(ctx, stream);     // an earlier launch on another stream may still read d_scans
  if (rc) return rc;
  // Descriptors already in pinned host memory (e.g. a torch pin_memory() buffer) are copied straight from there and
  // must stay untouched until the copy has run; pageable ones go through the context's pinned staging buffer.  A few
  // descriptors are always staged (the memcpy is cheaper than asking the driver what kind of pointer it is).
  bool pinned = false;
  if (bytes > 64 * 1024) {
    cudaPointerAttributes attr;
    pinned = cudaPointerGetAttributes(&attr, scans) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    if (!pinned) cudaGetLastError();
  }
  const qd_scan* src = scans;
  if (!pinned) {
    if (ctx->staged_pending) {
      QD_CUDA(ctx, cudaEventSynchronize(ctx->staged));   // the previous H2D out of the staging buffer has finished
      ctx->staged_pending = false;
    }
    if (ctx->h_scans_cap < bytes) {
      if (ctx->h_scans) cudaFreeHost(ctx->h_scans);
      ctx->h_scans = nullptr;
      ctx->h_scans_cap = 0;
      const size_t want = bytes + bytes / 4 + 4096;
      QD_CUDA(ctx, cudaMallocHost((void**)&ctx->h_scans, want));
      ctx->h_scans_cap = want;
    }
    memcpy(ctx->h_scans, scans, bytes);
    src = ctx->h_scans;
  }
  // the copy is issued first and runs while the host validates the descriptors (nothing is launched on a failure)
  QD_CUDA(ctx, cudaMemcpyAsync(ctx->d_scans, src, bytes, cudaMemcpyHostToDevice, stream));
  if (!pinned && !caller_syncs) {
    QD_CUDA(ctx, cudaEventRecord(ctx->staged, stream));
    ctx->staged_pending = true;
  }
  ctx->up_n_scan = 0;
  int mny = 0;
  long long ext = 0, mpix = 0;
  for (int i = 0; i < n_scan; ++i) {
    const qd_scan& s = scans[i];
    const long long np_ = (long long)s.nx * s.ny;
    if (s.pix_offset + np_ > ext) ext = s.pix_offset + np_;
    if (np_ > mpix) mpix = np_;
    rc = check_scan(ctx, i, s);
    if (rc) return rc;
    if (s.ny > mny) mny = s.ny;
  }
  *max_ny = mny;
  ctx->up_n_scan = n_scan;
  ctx->up_max_ny = mny;
  ctx->up_pixels = ext;
  ctx->up_max_pix = mpix;
  return QD_OK;
}

// sticky status word -> error of a synchronous entry point
int check_status(qd_ctx* ctx) {
  const unsigned st = *reinterpret_cast<volatile unsigned*>(ctx->h_status);
  if (!st) return QD_OK;
  *ctx->h_status = 0u;
  if (st & QD_STATUS_OCC_OVERFLOW)
    return fail(ctx, QD_ERR_INVALID,
                "a scan window reaches 252 or more carriers on a dot: outside the 0..255 range of the uint8 charge map "
                "and of the packed latching keys");
  return fail(ctx, QD_ERR_INVALID, "kernel status 0x%x", st);
}

// Pipeline plan of the *_host entry points: the scans are cut into chunks (multiples of `align` scans) whose output pixel
// ranges [lo, hi) are disjoint and increasing; chunk c+1 computes on one stream while chunk c's images travel back over
// PCIe on another.  Chunk sizes: equal, except that the last three halve (1, ..., 1, 1/2, 1/4, 1/8): the copy of the LAST
// chunk is the only one that cannot hide behind compute, so it is kept small as long as it still fills the chip.
struct ChunkPlan {
  int n_chunk = 1;
  std::vector<int> cut;
  std::vector<long long> lo, hi;
  bool tiled = true;       // the scans tile [0, pixels) without gaps
};

ChunkPlan plan_chunks(const qd_ctx* ctx, int n_scan, const qd_scan* scans, int align) {
  ChunkPlan P;
  const long long pixels = ctx->up_pixels;
  int n_chunk = n_scan / 2048;          // >= 2048 scans per chunk keeps every launch a full-chip wave or more
  int chunk_cap = 16;                   // measured (DESIGN.md, host-buffer pipeline): 16 chunks 43.6 ms, 12: 44.3, 8: 45.4
  if (const char* e = getenv("QDSIM_PIPE_CHUNKS")) chunk_cap = atoi(e) > 0 ? atoi(e) : chunk_cap;
  if (chunk_cap > 16) chunk_cap = 16;   // chunk_done[16]
  if (n_chunk > chunk_cap) n_chunk = chunk_cap;
  if (n_chunk < 1) n_chunk = 1;
  if (align < 1) align = 1;
  long long sum = 0;
  for (int i = 0; i < n_scan; ++i) sum += (long long)scans[i].nx * scans[i].ny;
  P.tiled = sum == pixels;
  P.cut.assign(n_chunk + 1, 0);
  {
    std::vector<double> w(n_chunk, 1.0);
    if (n_chunk >= 6) { w[n_chunk - 3] = 0.5; w[n_chunk - 2] = 0.25; w[n_chunk - 1] = 0.125; }
    double tot = 0.0;
    for (double x : w) tot += x;
    if (n_chunk >= 6 && (double)n_scan * w[n_chunk - 1] / tot < 2048.0) { std::fill(w.begin(), w.end(), 1.0); tot = n_chunk; }
    double acc = 0.0;
    for (int c = 0; c < n_chunk; ++c) {
      acc += w[c];
      int at = (int)((double)n_scan * acc / tot);
      at -= at % align;
      P.cut[c + 1] = std::max(at, P.cut[c]);
    }
    P.cut[n_chunk] = n_scan;
  }
  P.lo.assign(n_chunk, 0);
  P.hi.assign(n_chunk, 0);
  bool ok = true;
  for (int c = 0; c < n_chunk && ok; ++c) {
    long long a = -1, b = 0;
    for (int i = P.cut[c]; i < P.cut[c + 1]; ++i) {
      const long long p0 = scans[i].pix_offset, p1 = p0 + (long long)scans[i].nx * scans[i].ny;
      if (a < 0 || p0 < a) a = p0;
      if (p1 > b) b = p1;
    }
    if (a < 0) ok = false;                                   // empty chunk
    P.lo[c] = a; P.hi[c] = b;
    if (c > 0 && P.lo[c] < P.hi[c - 1]) ok = false;          // output ranges interleave: no pipeline
  }
  if (!ok || n_chunk == 1) {
    P.n_chunk = 1;
    P.cut.assign({0, n_scan});
    P.lo.assign({0});
    P.hi.assign({pixels});
  } else {
    P.n_chunk = n_chunk;
  }
  return P;
}

int pipe_rows_cap() {
  int rows_cap = 16;
  if (const char* e = getenv("QDSIM_PIPE_ROWS")) rows_cap = atoi(e) > 0 ? atoi(e) : rows_cap;
  return rows_cap;
}

}  // namespace

template <typename T>
int measure_peak(qd_ctx* ctx, int iters, double* tflops) {
  if (!ctx || !tflops) return fail(ctx, QD_ERR_INVALID, "NULL argument");
  if (iters <= 0) iters = 4096;
  QD_CUDA(ctx, cudaSetDevice(ctx->device));
  const int blocks = ctx->sm_count * 8, threads = 256;
  T* d = nullptr;
  QD_CUDA(ctx, cudaMalloc((void**)&d, sizeof(T) * blocks * threads));
  cudaEvent_t e0, e1;
  QD_CUDA(ctx, cudaEventCreate(&e0));
  QD_CUDA(ctx, cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    QD_CUDA(ctx, cudaEventRecord(e0));
    qd::qd_fma_peak_kernel<T><<<blocks, threads>>>(d, iters, (T)1.0000001, (T)1e-7);
    QD_CUDA(ctx, cudaEventRecord(e1));
    QD_CUDA(ctx, cudaEventSynchronize(e1));
    float ms = 0.f;
    QD_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 64.0 * (double)iters * blocks * threads;
    const double tf = flops / (ms * 1e-3) * 1e-12;
    if (rep > 0 && tf > best) best = tf;
    ctx->launches += 1;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *tflops = best;
  return QD_OK;
}

extern "C" {

int qd_abi_version(void) { return QD_ABI_VERSION; }

int qd_create(int device, qd_ctx** out) {
  if (!out) return fail(nullptr, QD_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess) return fail(nullptr, QD_ERR_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(nullptr, QD_ERR_INVALID, "device %d out of range (have %d)", device, count);
  qd_ctx* ctx = new (std::nothrow) qd_ctx();
  if (!ctx) return fail(nullptr, QD_ERR_NOMEM, "out of host memory");
  ctx->device = device;
  e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->staged, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->last_launch, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaHostAlloc((void**)&ctx->h_status, 64, cudaHostAllocMapped);
  if (e == cudaSuccess) {
    *ctx->h_status = 0u;
    e = cudaHostGetDevicePointer((void**)&ctx->d_status, ctx->h_status, 0);
  }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->s_compute, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking);
  for (int i = 0; i < 16 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&ctx->chunk_done[i], cudaEventDisableTiming);
  if (e != cudaSuccess) {
    fail(nullptr, QD_ERR_CUDA, "device %d init failed: %s", device, cudaGetErrorString(e));
    delete ctx;
    return QD_ERR_CUDA;
  }
  *out = ctx;
  return QD_OK;
}

void qd_destroy(qd_ctx* ctx) {
  if (!ctx) return;
  if (ctx->tr_calls > 0 && getenv("QDSIM_TRACE"))
    fprintf(stderr, "[qdsim] small-call path: %ld calls, per call launch %.2f us, sync %.2f us, copy-out %.2f us\n", ctx->tr_calls,
            ctx->tr_launch / ctx->tr_calls, ctx->tr_sync / ctx->tr_calls, ctx->tr_copy / ctx->tr_calls);
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  if (ctx->d_records) cudaFree(ctx->d_records);
  if (ctx->d_scans) cudaFree(ctx->d_scans);
  if (ctx->h_scans) cudaFreeHost(ctx->h_scans);
  if (ctx->d_z) cudaFree(ctx->d_z);
  if (ctx->d_n) cudaFree(ctx->d_n);
  if (ctx->d_pts) cudaFree(ctx->d_pts);
  if (ctx->d_nbar) cudaFree(ctx->d_nbar);
  if (ctx->d_tfloor) cudaFree(ctx->d_tfloor);
  if (ctx->d_tpot) cudaFree(ctx->d_tpot);
  if (ctx->d_tkeys) cudaFree(ctx->d_tkeys);
  if (ctx->d_obs) cudaFree(ctx->d_obs);
  if (ctx->d_stats) cudaFree(ctx->d_stats);
  if (ctx->h_status) cudaFreeHost(ctx->h_status);
  if (ctx->h_small) cudaFreeHost(ctx->h_small);
  if (ctx->last_launch) cudaEventDestroy(ctx->last_launch);
  if (ctx->staged) cudaEventDestroy(ctx->staged);
  for (int i = 0; i < 16; ++i) if (ctx->chunk_done[i]) cudaEventDestroy(ctx->chunk_done[i]);
  if (ctx->s_compute) cudaStreamDestroy(ctx->s_compute);
  if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
  delete ctx;
}

const char* qd_last_error(const qd_ctx* ctx) { return ctx ? ctx->err : g_err; }

int64_t qd_launch_count(const qd_ctx* ctx) { return ctx ? ctx->launches : 0; }

int qd_set_models(qd_ctx* ctx, const qd_model_desc* desc, const double* cdd_inv_gs, const double* cdd_gs,
                  const double* cdd_inv_full, const double* cgd_full, const double* cbg, const qd_env_params* params) {
  if (!ctx) return fail(nullptr, QD_ERR_INVALID, "ctx is NULL");
  if (!desc || !cdd_inv_gs || !cdd_inv_full || !cgd_full || !params)
    return fail(ctx, QD_ERR_INVALID, "NULL argument to qd_set_models");
  const int N = desc->n_dot, NV = desc->n_volt, G = desc->n_gate, D = N + desc->n_sensor;
  if (desc->n_env <= 0) return fail(ctx, QD_ERR_INVALID, "n_env must be positive");
  if (N < 1 || N > QD_MAX_DOTS) return fail(ctx, QD_ERR_INVALID, "n_dot must be in 1..%d, got %d", QD_MAX_DOTS, N);
  if (desc->n_sensor != 1) return fail(ctx, QD_ERR_UNSUPPORTED, "n_sensor must be 1, got %d", desc->n_sensor);
  if (NV < 1 || NV > QD_MAX_VOLT || G < 1 || G > NV)
    return fail(ctx, QD_ERR_INVALID, "bad n_volt=%d / n_gate=%d (max %d)", NV, G, QD_MAX_VOLT);
  const int alg = desc->algorithm;
  if (alg < QD_ALG_DEFAULT || alg > QD_ALG_TUNNEL) return fail(ctx, QD_ERR_INVALID, "Algorithm %d not supported", alg);
  if (alg == QD_ALG_TUNNEL) {
    if (N < 2) return fail(ctx, QD_ERR_INVALID, "the tunnel-coupled path needs at least 2 dots");
    if (desc->num_charge_states != 32)
      return fail(ctx, QD_ERR_UNSUPPORTED, "num_charge_states must be 32 (one basis state per lane), got %d",
                  desc->num_charge_states);
    if (NV != G && NV != G + N - 1)
      return fail(ctx, QD_ERR_INVALID, "tunnel path: n_volt must be n_gate or n_gate + n_dot - 1 (one barrier per gap)");
    if (NV != G && !cbg) return fail(ctx, QD_ERR_INVALID, "cbg is required when barrier voltages are present");
  }
  if ((alg == QD_ALG_DEFAULT || alg == QD_ALG_THRESHOLDED) && !cdd_gs)
    return fail(ctx, QD_ERR_INVALID, "cdd_gs is required for the default / thresholded algorithms");
  QD_CUDA(ctx, cudaSetDevice(ctx->device));

  const qd_layout L = qd_make_layout(N, NV, G, alg, desc->num_charge_states, desc->charge_state_batch_size);
  const size_t bytes = (size_t)desc->n_env * L.rec_doubles * sizeof(double);
  std::vector<double> host;
  try {
    host.assign((size_t)desc->n_env * L.rec_doubles, 0.0);
  } catch (...) {
    return fail(ctx, QD_ERR_NOMEM, "out of host memory packing %d model records", desc->n_env);
  }
  for (int e = 0; e < desc->n_env; ++e) {
    double* r = host.data() + (size_t)e * L.rec_doubles;
    const qd_env_params& p = params[e];
    if (alg == QD_ALG_BRUTE_FORCE && (p.max_charge_carriers < 0 || p.max_charge_carriers > 15))
      return fail(ctx, QD_ERR_INVALID, "env %d: max_charge_carriers must be in 0..15", e);
    if (!(p.kT >= 0.0)) return fail(ctx, QD_ERR_INVALID, "env %d: kT must be >= 0", e);
    if ((p.vc_alpha != 0.0 || p.vc_beta != 0.0) && alg != QD_ALG_TUNNEL)
      return fail(ctx, QD_ERR_UNSUPPORTED, "env %d: voltage-dependent capacitances exist on the tunnel path only", e);
    if (!(p.vc_alpha >= 0.0) || !(p.vc_beta >= 0.0))
      return fail(ctx, QD_ERR_INVALID, "env %d: vc_alpha / vc_beta must be >= 0", e);
    if (p.vc_kind < QD_VC_LINEAR || p.vc_kind > QD_VC_SIGMOID)
      return fail(ctx, QD_ERR_INVALID, "env %d: vc_kind %d is not a qd_vc_kind", e, p.vc_kind);
    if (p.vc_kind == QD_VC_SIGMOID && p.vc_alpha != 0.0 && !(p.vc_vchar > 0.0))
      return fail(ctx, QD_ERR_INVALID, "env %d: the sigmoid capacitance model needs vc_vchar > 0", e);
    memcpy(r + L.o_cinv, cdd_inv_gs + (size_t)e * N * N, sizeof(double) * N * N);
    if (cdd_gs) memcpy(r + L.o_cdd, cdd_gs + (size_t)e * N * N, sizeof(double) * N * N);
    const double* cg = cgd_full + (size_t)e * D * NV;
    memcpy(r + L.o_a, cg, sizeof(double) * N * NV);
    memcpy(r + L.o_sa, cg + (size_t)N * NV, sizeof(double) * NV);
    const double* ci = cdd_inv_full + (size_t)e * D * D;
    for (int j = 0; j < N; ++j) r[L.o_sw + j] = ci[(size_t)N * D + j];
    r[L.o_css] = ci[(size_t)N * D + N];
    double* par = r + L.o_par;
    par[QD_PAR_KT] = p.kT;
    par[QD_PAR_THRESHOLD] = p.threshold;
    par[QD_PAR_WHITE] = p.white_amp;
    par[QD_PAR_P01] = p.tele_p01;
    par[QD_PAR_P10] = p.tele_p10;
    par[QD_PAR_TELE_AMP] = p.tele_amp;
    const double tot = p.tele_p01 + p.tele_p10;
    par[QD_PAR_TELE_STAT] = tot > 0.0 ? p.tele_p01 / tot : 0.0;
    par[QD_PAR_LATCH] = p.latching ? 1.0 : 0.0;
    par[QD_PAR_MAXC] = (double)p.max_charge_carriers;
    par[QD_PAR_TC_BASE] = p.tc_base;
    par[QD_PAR_VC_ALPHA] = p.vc_alpha;
    par[QD_PAR_VC_BETA] = p.vc_beta;
    par[QD_PAR_PINK] = p.pink_amp;
    par[QD_PAR_VC_KIND] = (double)p.vc_kind;
    par[QD_PAR_VC_VCHAR] = p.vc_vchar;
    for (int j = 0; j < 8; ++j) r[L.o_alpha + j] = p.alpha[j];
    for (int j = 0; j < 8; ++j) r[L.o_pleads + j] = p.p_leads[j];
    for (int j = 0; j < 64; ++j) r[L.o_pinter + j] = p.p_inter[j];
    for (int j = 0; j < N; ++j) {
      double sp = 0.0, sn = 0.0;
      for (int k = 0; k < N; ++k) {
        if (k == j) continue;
        const double c = 2.0 * r[L.o_cinv + j * N + k];
        if (c > 0.0) sp += c; else sn += c;
      }
      r[L.o_spos + j] = sp;
      r[L.o_sneg + j] = sn;
    }
    if (alg == QD_ALG_TUNNEL) {
      if (cbg && NV > G) memcpy(r + L.o_cbg, cbg + (size_t)e * (NV - G) * G, sizeof(double) * (NV - G) * G);
    }
  }
  QD_CUDA(ctx, cudaDeviceSynchronize());   // nothing in flight may still read the old records
  int rc = grow(ctx, &ctx->d_records, &ctx->records_bytes, bytes);
  if (rc) return rc;
  QD_CUDA(ctx, cudaMemcpy(ctx->d_records, host.data(), bytes, cudaMemcpyHostToDevice));
  ctx->L = L;
  ctx->n_env = desc->n_env;
  ctx->up_n_scan = 0;
  if (alg == QD_ALG_DEFAULT || alg == QD_ALG_THRESHOLDED) {
    const long long total = (long long)desc->n_env << N;
    long long blocks = (total + 255) / 256;
    if (blocks > 65535) blocks = 65535;
    rc = issue(ctx, qd::qd_build_q_kernel, blocks, 256, 0, nullptr, L, ctx->d_records, desc->n_env);
    if (rc) return rc;
    QD_CUDA(ctx, cudaDeviceSynchronize());
  }
  ctx->have_models = true;
  return QD_OK;
}

int qd_scan_open(qd_ctx* ctx, int n_scan, const qd_scan* scans, float* z_out, void* n_out, int n_type, unsigned flags,
                 void* stream) {
  int rc = validate_launch(ctx, n_type, flags, n_out);
  if (rc) return rc;
  QD_CUDA(ctx, cudaSetDevice(ctx->device));
  int max_ny = 0;
  rc = stage_scans(ctx, n_scan, scans, (cudaStream_t)stream, &max_ny);
  if (rc) return rc;
  return launch(ctx, n_scan, ctx->d_scans, max_ny, nullptr, z_out, n_out, n_type, flags, (cudaStream_t)stream);
}

int qd_scan_upload(qd_ctx* ctx, int n_scan, const qd_scan* scans, void* stream) {
  if (!ctx) return fail(nullptr, QD_ERR_INVALID, "ctx is NULL");
  if (!ctx->have_models) return fail(ctx, QD_ERR_STATE, "qd_set_models has not been called");
  QD_CUDA(ctx, cudaSetDevice(ctx->device));
  int max_ny = 0;
  return stage_scans(ctx, n_scan, scans, (cudaStream_t)stream, &max_ny);
}

int qd_scan_launch(qd_ctx* ctx, float* z_out, void* n_out, int n_type, unsigned flags, void* stream) {
  int rc = validate_launch(ctx, n_type, flags, n_out);
  if (rc) return rc;
  if (ctx->up_n_scan <= 0) return fail(ctx, QD_ERR_STATE, "qd_scan_upload has not been called");
  QD_CUDA(ctx, cudaSetDevice(ctx->device));
  return launch(ctx, ctx->up_n_scan, ctx->d_scans, ctx->up_max_ny, nullptr, z_out, n_out, n_type, flags,
                (cudaStream_t)stream);
}

int qd_scan_open_host(qd_ctx* ctx, int n_scan, const qd_scan* scans, float* z_out_host, void* n_out_host, int n_type,
                      unsigned flags) {
  int rc = validate_launch(ctx, n_type, flags, n_out_host);
  if (rc) return rc;
  QD_CUDA(ctx, cudaSetDevice(ctx->device));
  *ctx->h_status = 0u;      // report what THIS call's kernels raise (a caller of the async entries polls qd_status itself)
  int max_ny = 0;
  // one scan of a Path A model (a single do2d_open): the descriptor goes into the kernel parameters, no H2D copy
  const bool one = n_scan == 1 && scans && ctx->L.algorithm != QD_ALG_TUNNEL && scans[0].pix_offset == 0 &&
                   (long long)scans[0].nx * scans[0].ny * (4 + ctx->L.n_dot * (long long)n_elem_size(n_type)) <= (1 << 20);
  if (one) {
    const qd_scan& s0 = scans[0];
    rc = check_scan(ctx, 0, s0);
    if (rc) return rc;
    rc = order_after_last_launch(ctx, ctx->s_compute);
    if (rc) return rc;
    max_ny = s0.ny;
    ctx->up_n_scan = 0;                 // nothing resident for qd_scan_launch
    ctx->up_max_ny = s0.ny;
    ctx->up_pixels = ctx->up_max_pix = (long long)s0.nx * s0.ny;
  } else {
    rc = stage_scans(ctx, n_scan, scans, ctx->s_compute, &max_ny, true);
    if (rc) return rc;
  }
  const long long pixels = ctx->up_pixels;
  const int N = ctx->L.n_dot;
  const size_t esz = n_elem_size(n_type);
  const size_t zbytes = z_out_host ? (size_t)pixels * sizeof(float) : 0, nbytes = (size_t)pixels * N * esz;
  // ---- small calls (a single do2d_open): the kernel writes its outputs straight into mapped pinned host memory, so the
  // call is one descriptor copy, one launch (two on the tunnel path) and one synchronisation -- no device-to-host copies
  if (zbytes + nbytes <= (1u << 20) && n_scan <= 64) {
    const size_t zoff = (zbytes + 255) & ~(size_t)255;
    const size_t need = zoff + nbytes + 256;
    if (ctx->small_cap < need) {
      if (ctx->h_small) cudaFreeHost(ctx->h_small);
      ctx->h_small = ctx->d_small = nullptr;
      ctx->small_cap = 0;
      QD_CUDA(ctx, cudaHostAlloc((void**)&ctx->h_small, (1u << 20) + 4096, cudaHostAllocMapped));
      QD_CUDA(ctx, cudaHostGetDevicePointer((void**)&ctx->d_small, ctx->h_small, 0));
      ctx->small_cap = (1u << 20) + 4096;
    }
    long long sum = 0;
    for (int i = 0; i < n_scan; ++i) sum += (long long)scans[i].nx * scans[i].ny;
    if (sum != pixels) memset(ctx->h_small, 0, need);          // gaps between scans read as zeros
    using clk = std::chrono::steady_clock;
    const auto t0 = clk::now();
    rc = launch(ctx, n_scan, ctx->d_scans, max_ny, nullptr, z_out_host ? (float*)ctx->d_small : nullptr,
                ctx->d_small + zoff, n_type, flags, ctx->s_compute, 0, one ? scans : nullptr);
    if (rc) return rc;
    const auto t1 = clk::now();
    // a latency-bound call: poll the stream instead of cudaStreamSynchronize (whose wake-up costs microseconds); bounded,
    // then fall back to the blocking wait
    {
      cudaError_t q = cudaErrorNotReady;
      for (int spin = 0; spin < 200000 && q == cudaErrorNotReady; ++spin) q = cudaStreamQuery(ctx->s_compute);
      if (q == cudaErrorNotReady) q = cudaStreamSynchronize(ctx->s_compute);
      QD_CUDA(ctx, q);
    }
    const auto t2 = clk::now();
    ctx->staged_pending = false;
    if (z_out_host) memcpy(z_out_host, ctx->h_small, zbytes);
    if (nbytes) memcpy(n_out_host, ctx->h_small + zoff, nbytes);
    const auto t3 = clk::now();
    ctx->tr_launch += std::chrono::duration<double, std::micro>(t1 - t0).count();
    ctx->tr_sync += std::chrono::duration<double, std::micro>(t2 - t1).count();
    ctx->tr_copy += std::chrono::duration<double, std::micro>(t3 - t2).count();
    ctx->tr_calls += 1;
    return check_status(ctx);
  }

  rc = grow(ctx, &ctx->d_z, &ctx->z_cap, (size_t)pixels * sizeof(float));
  if (rc) return rc;
  if (esz) {
    rc = grow(ctx, (unsigned char**)&ctx->d_n, &ctx->n_cap, (size_t)pixels * N * esz);
    if (rc) return rc;
  }
  const ChunkPlan P = plan_chunks(ctx, n_scan, scans, 1);
  if (!P.tiled) {
    // the copies below move whole pixel ranges: what lies between the scans must not be stale device memory
    if (z_out_host) QD_CUDA(ctx, cudaMemsetAsync(ctx->d_z, 0, (size_t)pixels * sizeof(float), ctx->s_compute));
    if (esz) QD_CUDA(ctx, cudaMemsetAsync(ctx->d_n, 0, (size_t)pixels * N * esz, ctx->s_compute));
  }
  const int rows_cap = pipe_rows_cap();
  for (int c = 0; c < P.n_chunk; ++c) {
    rc = launch(ctx, P.cut[c + 1] - P.cut[c], ctx->d_scans + P.cut[c], max_ny, nullptr, ctx->d_z, ctx->d_n, n_type, flags,
                ctx->s_compute, P.n_chunk > 1 ? rows_cap : 0);
    if (rc) return rc;
    QD_CUDA(ctx, cudaEventRecord(ctx->chunk_done[c], ctx->s_compute));
    QD_CUDA(ctx, cudaStreamWaitEvent(ctx->s_copy, ctx->chunk_done[c], 0));
    const long long lo = P.lo[c], hi = P.hi[c];
    if (z_out_host)
      QD_CUDA(ctx, cudaMemcpyAsync(z_out_host + lo, ctx->d_z + lo, (size_t)(hi - lo) * sizeof(float),
                                   cudaMemcpyDeviceToHost, ctx->s_copy));
    if (esz)
      QD_CUDA(ctx, cudaMemcpyAsync((char*)n_out_host + (size_t)lo * N * esz, (char*)ctx->d_n + (size_t)lo * N * esz,
                                   (size_t)(hi - lo) * N * esz, cudaMemcpyDeviceToHost, ctx->s_copy));
  }
  QD_CUDA(ctx, cudaStreamSynchronize(ctx->s_copy));
  QD_CUDA(ctx, cudaStreamSynchronize(ctx->s_compute));
  ctx->staged_pending = false;
  return check_status(ctx);
}

extern "C++" {
namespace {
size_t z_elem_size(int z_type) { return z_type == QD_Z_F32 ? 4 : z_type == QD_Z_F16 ? 2 : z_type == QD_Z_U8 ? 1 : 0; }

template <typename OUT>
int normalise_launch(qd_ctx* ctx, const float* z, OUT* out, int64_t per_env, int n_env, double ql, double qh, double* stats,
                     cudaStream_t stream) {
  const size_t need = (size_t)per_env * sizeof(float);
  auto fn = qd::qd_normalise_kernel<OUT, false>;
  size_t smem = 0;
  if (per_env <= 32 * 1024) {        // the env's image fits in the registers of one CTA: one HBM read per pixel
    fn = qd::qd_normalise_reg_kernel<OUT>;
  } else if (need <= 200 * 1024) {   // ... or in its shared memory
    fn = qd::qd_normalise_kernel<OUT, true>;
    smem = need;
  }
  return issue(ctx, fn, n_env, 1024, smem, stream, z, out, per_env, n_env, ql, qh, stats);
}

int normalise_typed(qd_ctx* ctx, const float* z, void* out, int z_type, int64_t per_env, int n_env, double q_low_pct,
                    double q_high_pct, double* stats, cudaStream_t stream) {
  const double ql = q_low_pct / 100.0, qh = q_high_pct / 100.0;
  switch (z_type) {
    case QD_Z_F32: return normalise_launch<float>(ctx, z, (float*)out, per_env, n_env, ql, qh, stats, stream);
    case QD_Z_F16: return normalise_launch<__half>(ctx, z, (__half*)out, per_env, n_env, ql, qh, stats, stream);
    case QD_Z_U8: return normalise_launch<unsigned char>(ctx, z, (unsigned char*)out, per_env, n_env, ql, qh, stats, stream);
    default: return fail(ctx, QD_ERR_INVALID, "bad z_type %d", z_type);
  }
}
}  // namespace
}  // extern "C++"

int qd_scan_obs_host(qd_ctx* ctx, int n_scan, const qd_scan* scans, int scans_per_env, void* out_host, int z_type,
                     int normalise, double q_low_pct, double q_high_pct, double* stats_host, unsigned flags) {
  int rc = validate_launch(ctx, QD_N_NONE, flags, nullptr);
  if (rc) return rc;
  if (!out_host) return fail(ctx, QD_ERR_INVALID, "out_host is NULL");
  const size_t zsz = z_elem_size(z_type);
  if (!zsz) return fail(ctx, QD_ERR_INVALID, "bad z_type %d", z_type);
  if (!normalise && z_type == QD_Z_U8) return fail(ctx, QD_ERR_INVALID, "QD_Z_U8 needs a normalised image (normalise = 1)");
  if (scans_per_env <= 0 || n_scan <= 0 || n_scan % scans_per_env != 0)
    return fail(ctx, QD_ERR_INVALID, "n_scan (%d) must be a positive multiple of scans_per_env (%d)", n_scan, scans_per_env);
  if (normalise && !(q_low_pct >= 0.0 && q_low_pct <= q_high_pct && q_high_pct <= 100.0))
    return fail(ctx, QD_ERR_INVALID, "percentiles must satisfy 0 <= low <= high <= 100");
  if (!scans) return fail(ctx, QD_ERR_INVALID, "scans is NULL");
  const long long per_scan = (long long)scans[0].nx * scans[0].ny;
  for (int i = 0; i < n_scan; ++i)
    if (scans[i].nx != scans[0].nx || scans[i].ny != scans[0].ny || scans[i].pix_offset != (long long)i * per_scan)
      return fail(ctx, QD_ERR_INVALID, "scan %d: the observation path needs equal-size scans with pix_offset = i * nx * ny", i);
  QD_CUDA(ctx, cudaSetDevice(ctx->device));
  *ctx->h_status = 0u;
  int max_ny = 0;
  rc = stage_scans(ctx, n_scan, scans, ctx->s_compute, &max_ny, true);
  if (rc) return rc;
  const long long pixels = ctx->up_pixels;
  const int n_env_b = n_scan / scans_per_env;
  const long long per_env = per_scan * scans_per_env;
  rc = grow(ctx, &ctx->d_z, &ctx->z_cap, (size_t)pixels * sizeof(float));
  if (rc) return rc;
  const bool direct = !normalise && z_type == QD_Z_F32;        // raw fp32: copied straight out of d_z
  if (!direct) {
    rc = grow(ctx, (unsigned char**)&ctx->d_obs, &ctx->obs_cap, (size_t)pixels * zsz);
    if (rc) return rc;
  }
  if (normalise) {
    rc = grow(ctx, &ctx->d_stats, &ctx->stats_cap, (size_t)n_env_b * 2 * sizeof(double));
    if (rc) return rc;
  }
  const ChunkPlan P = plan_chunks(ctx, n_scan, scans, scans_per_env);
  const int rows_cap = pipe_rows_cap();
  for (int c = 0; c < P.n_chunk; ++c) {
    rc = launch(ctx, P.cut[c + 1] - P.cut[c], ctx->d_scans + P.cut[c], max_ny, nullptr, ctx->d_z, nullptr, QD_N_NONE, flags,
                ctx->s_compute, P.n_chunk > 1 ? rows_cap : 0);
    if (rc) return rc;
    const long long lo = P.lo[c], hi = P.hi[c];
    const int env0 = P.cut[c] / scans_per_env, envs = (P.cut[c + 1] - P.cut[c]) / scans_per_env;
    const char* src = (const char*)ctx->d_z + (size_t)lo * 4;
    if (normalise) {
      rc = normalise_typed(ctx, ctx->d_z + lo, (char*)ctx->d_obs + (size_t)lo * zsz, z_type, per_env, envs, q_low_pct,
                           q_high_pct, ctx->d_stats + 2 * (size_t)env0, ctx->s_compute);
      if (rc) return rc;
      src = (const char*)ctx->d_obs + (size_t)lo * zsz;
    } else if (z_type == QD_Z_F16) {
      long long blocks = (hi - lo + 2047) / 2048;
      if (blocks > 8 * (long long)ctx->sm_count) blocks = 8 * (long long)ctx->sm_count;
      rc = issue(ctx, qd::qd_to_half_kernel, blocks, 256, 0, ctx->s_compute, ctx->d_z + lo, (__half*)ctx->d_obs + lo,
                 hi - lo);
      if (rc) return rc;
      src = (const char*)ctx->d_obs + (size_t)lo * zsz;
    }
    QD_CUDA(ctx, cudaEventRecord(ctx->chunk_done[c], ctx->s_compute));
    QD_CUDA(ctx, cudaStreamWaitEvent(ctx->s_copy, ctx->chunk_done[c], 0));
    QD_CUDA(ctx, cudaMemcpyAsync((char*)out_host + (size_t)lo * zsz, src, (size_t)(hi - lo) * zsz, cudaMemcpyDeviceToHost,
                                 ctx->s_copy));
  }
  if (normalise && stats_host) {
    QD_CUDA(ctx, cudaStreamSynchronize(ctx->s_compute));
    QD_CUDA(ctx, cudaMemcpyAsync(stats_host, ctx->d_stats, (size_t)n_env_b * 2 * sizeof(double), cudaMemcpyDeviceToHost,
                                 ctx->s_copy));
  }
  QD_CUDA(ctx, cudaStreamSynchronize(ctx->s_copy));
  QD_CUDA(ctx, cudaStreamSynchronize(ctx->s_compute));
  ctx->staged_pending = false;
  return check_status(ctx);
}

int qd_points_open_host(qd_ctx* ctx, const qd_scan* scan, int ny, int nx, const double* v, float* z_out_host,
                        void* n_out_host, int n_type, unsigned flags) {
  int rc = validate_launch(ctx, n_type, flags, n_out_host);
  if (rc) return rc;
  if (!scan || !v) return fail(ctx, QD_ERR_INVALID, "NULL argument to qd_points_open_host");
  if (nx <= 0 || ny <= 0) return fail(ctx, QD_ERR_INVALID, "nx, ny must be positive");
  QD_CUDA(ctx, cudaSetDevice(ctx->device));
  *ctx->h_status = 0u;
  qd_scan s = *scan;
  s.nx = nx;
  s.ny = ny;
  s.pix_offset = 0;
  int max_ny = 0;
  rc = stage_scans(ctx, 1, &s, nullptr, &max_ny, true);
  if (rc) return rc;
  const long long pixels = (long long)nx * ny;
  const int N = ctx->L.n_dot, NV = ctx->L.n_volt;
  rc = grow(ctx, &ctx->d_pts, &ctx->pts_cap, (size_t)pixels * NV * sizeof(double));
  if (rc) return rc;
  rc = grow(ctx, &ctx->d_z, &ctx->z_cap, (size_t)pixels * sizeof(float));
  if (rc) return rc;
  const size_t nbytes = (size_t)pixels * N * n_elem_size(n_type);
  if (nbytes) {
    rc = grow(ctx, (unsigned char**)&ctx->d_n, &ctx->n_cap, nbytes);
    if (rc) return rc;
  }
  QD_CUDA(ctx, cudaMemcpyAsync(ctx->d_pts, v, (size_t)pixels * NV * sizeof(double), cudaMemcpyHostToDevice, nullptr));
  rc = launch(ctx, 1, ctx->d_scans, max_ny, ctx->d_pts, ctx->d_z, ctx->d_n, n_type, flags, nullptr);
  if (rc) return rc;
  if (z_out_host)
    QD_CUDA(ctx, cudaMemcpyAsync(z_out_host, ctx->d_z, (size_t)pixels * sizeof(float), cudaMemcpyDeviceToHost, nullptr));
  if (nbytes) QD_CUDA(ctx, cudaMemcpyAsync(n_out_host, ctx->d_n, nbytes, cudaMemcpyDeviceToHost, nullptr));
  QD_CUDA(ctx, cudaStreamSynchronize(nullptr));
  ctx->staged_pending = false;
  return check_status(ctx);
}

int qd_normalise_obs_typed(qd_ctx* ctx, const float* z, void* out, int z_type, int64_t per_env, int n_env,
                           double q_low_pct, double q_high_pct, double* stats, void* stream) {
  if (!ctx) return fail(nullptr, QD_ERR_INVALID, "ctx is NULL");
  if (!z || !out) return fail(ctx, QD_ERR_INVALID, "NULL image pointer");
  if (per_env <= 0 || n_env <= 0) return fail(ctx, QD_ERR_INVALID, "per_env and n_env must be positive");
  if (!(q_low_pct >= 0.0 && q_low_pct <= q_high_pct && q_high_pct <= 100.0))
    return fail(ctx, QD_ERR_INVALID, "percentiles must satisfy 0 <= low <= high <= 100");
  QD_CUDA(ctx, cudaSetDevice(ctx->device));
  return normalise_typed(ctx, z, out, z_type, per_env, n_env, q_low_pct, q_high_pct, stats, (cudaStream_t)stream);
}

int qd_normalise_obs(qd_ctx* ctx, const float* z, float* out, int64_t per_env, int n_env, double q_low_pct,
                     double q_high_pct, double* stats, void* stream) {
  return qd_normalise_obs_typed(ctx, z, out, QD_Z_F32, per_env, n_env, q_low_pct, q_high_pct, stats, stream);
}

int qd_status(qd_ctx* ctx, int clear) {
  if (!ctx || !ctx->h_status) return 0;
  const unsigned st = *reinterpret_cast<volatile unsigned*>(ctx->h_status);
  if (clear) *ctx->h_status = 0u;
  return (int)st;
}

int qd_measure_fp64_peak(qd_ctx* ctx, int iters, double* tflops) { return measure_peak<double>(ctx, iters, tflops); }
int qd_measure_fp32_peak(qd_ctx* ctx, int iters, double* tflops) { return measure_peak<float>(ctx, iters, tflops); }

}  // extern "C"
