// qd_normalise.cuh -- K8: per-env percentile normalisation of the observation images (first "next" row of SURVEY 8f).
// Replaces QuantumDeviceEnv._normalise_obs (src/qadapt/environment/env.py:471-509):
//     p_low, p_high = np.percentile(image, 0.5), np.percentile(image, 99.5)      # over ALL channels of the env
//     image = clip((image - p_low) / (p_high - p_low), 0, 1).astype(float32)      # zeros if p_high <= p_low
// One CTA per env.  The four order statistics the two interpolated percentiles need (ranks k, k+1 at both ends) are
// found EXACTLY by a 4-pass 8-bit radix select over the monotone uint32 image of the fp32 values (shared-memory
// histograms, four ranks tracked at once), then one more pass normalises in fp64 and writes fp32 / half / uint8.  The
// env's image (N-1 scans, 112 KB at 8 dots x 64 x 64) is staged in shared memory once: 4 B read + one typed write per pixel.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace qd {

__device__ __forceinline__ uint32_t f32_key(float x) {
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);      // order-preserving map float -> uint32
}
__device__ __forceinline__ float key_f32(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// numpy's _lerp (lib/_function_base_impl.py): a + (b-a) t, or b - (b-a)(1-t) when t >= 0.5
// (explicitly rounded products and sums: an FMA contraction would differ from NumPy in the last bit)
__device__ __forceinline__ double np_lerp(double a, double b, double t) {
  const double d = __dsub_rn(b, a);
  return (t >= 0.5) ? __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, t))) : __dadd_rn(a, __dmul_rn(d, t));
}

// typed store of a normalised value in [0, 1]: fp32, IEEE half, or uint8 = rint(255 v)
__device__ __forceinline__ void store_norm(float* p, double v) { *p = (float)v; }
__device__ __forceinline__ void store_norm(__half* p, double v) { *p = __float2half_rn((float)v); }
__device__ __forceinline__ void store_norm(unsigned char* p, double v) { *p = (unsigned char)__double2int_rn(255.0 * v); }

// Histogram update of one warp: when every participating lane hits the same bin (a plateau of the image -- the common
// case in the leading digits) one lane adds the count; otherwise plain shared-memory atomics.
__device__ __forceinline__ void hist_add(unsigned* hist, uint32_t b, bool on) {
  const unsigned act = __ballot_sync(0xffffffffu, on);
  if (!act) return;
  const uint32_t b0 = __shfl_sync(0xffffffffu, b, __ffs(act) - 1);
  if (__all_sync(0xffffffffu, !on || b == b0)) {
    if ((int)(threadIdx.x & 31) == __ffs(act) - 1) atomicAdd(&hist[b0], (unsigned)__popc(act));
  } else if (on) {
    atomicAdd(&hist[b], 1u);
  }
}

// The production kernel: one CTA of 1024 threads per env, the env's image held in REGISTERS (up to 32 values per thread,
// i.e. 32768 pixels per env: 8 dots x 64 x 64 = 28672), so HBM sees one 4-byte read and one typed write per pixel.
//
// The two percentiles of the reference (0.5 % and 99.5 %) are EXTREME order statistics: ranks k, k+1 with k ~ 143 from the
// bottom and from the top of 28672 values.  So instead of histogramming every pixel, the kernel
//   (1) takes each thread's minimum and maximum; the (k_lo+2)-th smallest of the 1024 thread minima, T_lo, is an upper bound
//       of the value of rank k_lo+1 (the minima alone are k_lo+2 values <= T_lo); likewise T_hi from the maxima.  Both come
//       from one 4-pass radix select over ONE value per thread (passes whose byte is common to all values are skipped);
//   (2) gathers the pixels <= T_lo and >= T_hi into two short shared-memory lists (a few hundred entries: T_lo sits near the
//       k/1024 quantile of minima-of-28, i.e. near the 0.5 % quantile of the image);
//   (3) ranks the list entries by counting ((value, position) order, so ties are exact) and picks ranks k, k+1 from each end.
// Exact for every input.  Inputs that defeat (2) -- more than 1024 pixels tied at an extreme, percentiles that are not
// extreme, envs larger than 1024 x 32 -- take the full MSB-first radix select over the registers (FULL below).
template <typename OUT>
__global__ void __launch_bounds__(1024) qd_normalise_reg_kernel(const float* __restrict__ z, OUT* __restrict__ out,
                                                                long long per_env, int n_env, double q_lo, double q_hi,
                                                                double* __restrict__ stats) {
  constexpr int EPT = 32;
  constexpr int LCAP = 1024;
  __shared__ unsigned hist[4][256];
  __shared__ uint32_t prefix[4];
  __shared__ long long rank[4];
  __shared__ uint32_t red[2][32];
  __shared__ uint32_t list_lo[LCAP], list_hi[LCAP];
  __shared__ unsigned cnt[2];
  const int env = blockIdx.x;
  if (env >= n_env) return;
  const float* __restrict__ src = z + (size_t)env * per_env;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  uint32_t key[EPT];
  uint32_t kmin = 0xffffffffu, kmax = 0u;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const long long i = (long long)e * 1024 + tid;
    key[e] = 0u;
    if (i < per_env) {
      key[e] = f32_key(src[i]);
      kmin = min(kmin, key[e]);
      kmax = max(kmax, key[e]);
    }
  }
  const uint32_t tmin = kmin, tmax = kmax;                 // this thread's own extremes
  const bool has = tid < per_env;                          // the thread holds at least one pixel
  kmin = __reduce_min_sync(0xffffffffu, kmin);
  kmax = __reduce_max_sync(0xffffffffu, kmax);
  if (lane == 0) { red[0][wid] = kmin; red[1][wid] = kmax; }
  // numpy 'linear' percentile: virtual index (n-1) q, neighbours floor / floor+1 (clamped), weight = fractional part
  // (explicitly rounded product: contracted into the subtraction below it would differ from NumPy in the last bit of t)
  const double vi_lo = __dmul_rn((double)(per_env - 1), q_lo), vi_hi = __dmul_rn((double)(per_env - 1), q_hi);
  const long long k_lo = (long long)floor(vi_lo), k_hi = (long long)floor(vi_hi);
  const long long r_lo1 = min(k_lo + 1, per_env - 1), r_hi1 = min(k_hi + 1, per_env - 1);
  const long long M = min(per_env, (long long)1024);        // threads that hold pixels
  // extreme-rank path: enough thread minima / maxima to bound the wanted ranks
  bool fast = (k_lo + 2 <= M) && (per_env - k_hi <= M) && per_env <= (long long)EPT * 1024;
  if (tid == 0) { cnt[0] = 0u; cnt[1] = 0u; }
  __syncthreads();
  kmin = __reduce_min_sync(0xffffffffu, red[0][lane]);
  kmax = __reduce_max_sync(0xffffffffu, red[1][lane]);

  if (fast) {
    // ---- (1) T_lo = ascending rank k_lo+1 of the thread minima, T_hi = ascending rank M - (n - k_hi) of the maxima ----
    if (tid == 0) { rank[0] = k_lo + 1; rank[1] = M - (per_env - k_hi); prefix[0] = prefix[1] = 0u; }
    __syncthreads();
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      if ((kmin >> shift) == (kmax >> shift)) {            // every pixel shares this byte and all above it
        __syncthreads();
        if (tid < 2) prefix[tid] |= ((kmin >> shift) & 0xffu) << shift;
        __syncthreads();
        continue;
      }
      for (int i = tid; i < 2 * 256; i += 1024) (&hist[0][0])[i] = 0u;
      __syncthreads();
      const uint32_t hi_mask = (pass == 0) ? 0u : (0xffffffffu << (shift + 8));
      const uint32_t p0 = prefix[0], p1 = prefix[1];
      hist_add(hist[0], (tmin >> shift) & 0xffu, has && (tmin & hi_mask) == p0);
      hist_add(hist[1], (tmax >> shift) & 0xffu, has && (tmax & hi_mask) == p1);
      __syncthreads();
      if (tid < 2) {
        long long r = rank[tid];
        int bb = 0;
        for (; bb < 255; ++bb) {
          const unsigned c = hist[tid][bb];
          if (r < (long long)c) break;
          r -= c;
        }
        rank[tid] = r;
        prefix[tid] |= (uint32_t)bb << shift;
      }
      __syncthreads();
    }
    const uint32_t T_lo = prefix[0], T_hi = prefix[1];
    // ---- (2) gather the pixels at or beyond the two thresholds ----
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      if ((long long)e * 1024 >= per_env) break;           // (uniform over the CTA)
      const bool in = (long long)e * 1024 + tid < per_env;
      const bool lo = in && key[e] <= T_lo, hi = in && key[e] >= T_hi;
      const unsigned ml = __ballot_sync(0xffffffffu, lo), mh = __ballot_sync(0xffffffffu, hi);
      if (ml) {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(&cnt[0], (unsigned)__popc(ml));
        base = __shfl_sync(0xffffffffu, base, 0);
        const unsigned at = base + __popc(ml & ((1u << lane) - 1u));
        if (lo && at < LCAP) list_lo[at] = key[e];
      }
      if (mh) {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(&cnt[1], (unsigned)__popc(mh));
        base = __shfl_sync(0xffffffffu, base, 0);
        const unsigned at = base + __popc(mh & ((1u << lane) - 1u));
        if (hi && at < LCAP) list_hi[at] = key[e];
      }
    }
    __syncthreads();
    const unsigned L0 = cnt[0], L1 = cnt[1];
    fast = L0 <= (unsigned)LCAP && L1 <= (unsigned)LCAP;   // (uniform) otherwise: massive ties at an extreme -> FULL
    if (fast) {
      // ---- (3) rank by counting.  The gather order is arbitrary, but ties hold EQUAL values: any consistent tie-break
      // (here: list position) yields the same value at every rank ----
      if (tid < (int)L0) {
        const uint32_t v = list_lo[tid];
        unsigned r = 0;
        for (unsigned j = 0; j < L0; ++j) { const uint32_t w = list_lo[j]; r += (w < v || (w == v && j < (unsigned)tid)) ? 1u : 0u; }
        if ((long long)r == k_lo) prefix[0] = v;
        if ((long long)r == r_lo1) prefix[1] = v;
      }
      if (tid < (int)L1) {
        const uint32_t v = list_hi[tid];
        unsigned r = 0;                                     // rank from the TOP
        for (unsigned j = 0; j < L1; ++j) { const uint32_t w = list_hi[j]; r += (w > v || (w == v && j < (unsigned)tid)) ? 1u : 0u; }
        if ((long long)r == per_env - 1 - k_hi) prefix[2] = v;
        if ((long long)r == per_env - 1 - r_hi1) prefix[3] = v;
      }
    }
    __syncthreads();
  }
  if (!fast) {
    // ---- FULL: MSB-first 8-bit radix select of the four ranks over all pixels (in registers) ----
    if (tid == 0) {
      rank[0] = k_lo; rank[1] = r_lo1; rank[2] = k_hi; rank[3] = r_hi1;
      prefix[0] = prefix[1] = prefix[2] = prefix[3] = 0u;
    }
    __syncthreads();
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      if ((kmin >> shift) == (kmax >> shift)) {          // every pixel shares this byte (and all above): nothing to select
        __syncthreads();
        if (tid < 4) prefix[tid] |= ((kmin >> shift) & 0xffu) << shift;
        __syncthreads();
        continue;
      }
      for (int i = tid; i < 4 * 256; i += 1024) (&hist[0][0])[i] = 0u;
      __syncthreads();
      const uint32_t hi_mask = (pass == 0) ? 0u : (0xffffffffu << (shift + 8));
      const uint32_t p0 = prefix[0], p1 = prefix[1], p2 = prefix[2], p3 = prefix[3];
      const bool d1 = p1 != p0, d2 = p2 != p0 && p2 != p1, d3 = p3 != p0 && p3 != p1 && p3 != p2;
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const long long i = (long long)e * 1024 + tid;
        if ((long long)e * 1024 >= per_env) break;       // (uniform over the CTA)
        const bool in = i < per_env;
        const uint32_t k = key[e];
        const uint32_t b = (k >> shift) & 0xffu, top = k & hi_mask;
        hist_add(hist[0], b, in && top == p0);
        if (d1) hist_add(hist[1], b, in && top == p1);
        if (d2) hist_add(hist[2], b, in && top == p2);
        if (d3) hist_add(hist[3], b, in && top == p3);
      }
      __syncthreads();
      if (tid < 256) {
        const int b = tid;
        if (!d1) hist[1][b] = hist[0][b];
        if (!d2) hist[2][b] = (p2 == p0) ? hist[0][b] : hist[1][b];
        if (!d3) hist[3][b] = (p3 == p0) ? hist[0][b] : (p3 == p1) ? hist[1][b] : hist[2][b];
      }
      __syncthreads();
      if (tid < 4) {
        const int t = tid;
        long long r = rank[t];
        int b = 0;
        for (; b < 255; ++b) {
          const unsigned c = hist[t][b];
          if (r < (long long)c) break;
          r -= c;
        }
        rank[t] = r;
        prefix[t] |= (uint32_t)b << shift;
      }
      __syncthreads();
    }
  }
  const double a_lo = (double)key_f32(prefix[0]), b_lo = (double)key_f32(prefix[1]);
  const double a_hi = (double)key_f32(prefix[2]), b_hi = (double)key_f32(prefix[3]);
  const double p_low = np_lerp(a_lo, b_lo, __dsub_rn(vi_lo, (double)k_lo));
  const double p_high = np_lerp(a_hi, b_hi, __dsub_rn(vi_hi, (double)k_hi));
  if (stats && tid == 0) { stats[2 * env] = p_low; stats[2 * env + 1] = p_high; }
  const bool ok = p_high > p_low;
  const double span = p_high - p_low;
  OUT* __restrict__ dst = out + (size_t)env * per_env;
  // The reference's fp64 quotient (x - p_low) / span, correctly rounded, for every output type: the same values as
  // qd_normalise_kernel's division, whichever kernel the env's size picks (tests/test_normalise_gpu.py).  Without a
  // division per pixel: q0 = d * RN(1 / span) is within an ulp and one exact residual step rounds it correctly
  // (Markstein), as long as nothing underflows -- d is 0 or >= ~2^-202 for fp32 pixels.  (An fp32 multiply-add by
  // 1 / span instead loses about log2(p_low / span) bits: 8 LSB of uint8 at p_low / span = 1e6.)
  const double rcp = ok ? 1.0 / span : 0.0;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const long long i = (long long)e * 1024 + tid;
    if (i < per_env) {
      const double d = __dsub_rn((double)key_f32(key[e]), p_low);
      const double q0 = __dmul_rn(d, rcp);
      double v = ok ? __fma_rn(__fma_rn(-q0, span, d), rcp, q0) : 0.0;
      v = fmin(fmax(v, 0.0), 1.0);
      store_norm(dst + i, v);
    }
  }
}

// RESIDENT = true: the env's image is staged in shared memory once (dynamic smem of per_env floats) and the four radix
// passes + the output pass read it from there: 4 B read + sizeof(OUT) written per pixel of HBM traffic.
template <typename OUT, bool RESIDENT>
__global__ void __launch_bounds__(1024) qd_normalise_kernel(const float* __restrict__ z, OUT* __restrict__ out,
                                                            long long per_env, int n_env, double q_lo, double q_hi,
                                                            double* __restrict__ stats) {
  extern __shared__ __align__(16) float zs[];
  __shared__ unsigned hist[4][256];
  __shared__ uint32_t prefix[4];
  __shared__ long long rank[4];
  const int env = blockIdx.x;
  if (env >= n_env) return;
  const float* __restrict__ gsrc = z + (size_t)env * per_env;
  const long long n_round = (per_env + 31) & ~31LL;          // whole warps run every iteration (match / ballot below)
  if (RESIDENT) {
    for (long long i = threadIdx.x; i < per_env; i += blockDim.x) zs[i] = gsrc[i];
    __syncthreads();
  }
  const float* __restrict__ src = RESIDENT ? zs : gsrc;
  // numpy 'linear' percentile: virtual index (n-1) q, neighbours floor / floor+1 (clamped), weight = fractional part
  // (explicitly rounded product: contracted into the subtraction below it would differ from NumPy in the last bit of t)
  const double vi_lo = __dmul_rn((double)(per_env - 1), q_lo), vi_hi = __dmul_rn((double)(per_env - 1), q_hi);
  const long long k_lo = (long long)floor(vi_lo), k_hi = (long long)floor(vi_hi);
  if (threadIdx.x == 0) {
    rank[0] = k_lo; rank[1] = min(k_lo + 1, per_env - 1);
    rank[2] = k_hi; rank[3] = min(k_hi + 1, per_env - 1);
    prefix[0] = prefix[1] = prefix[2] = prefix[3] = 0u;
  }
  __syncthreads();
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int i = threadIdx.x; i < 4 * 256; i += blockDim.x) (&hist[0][0])[i] = 0u;
    __syncthreads();
    const uint32_t hi_mask = (pass == 0) ? 0u : (0xffffffffu << (shift + 8));
    const uint32_t p0 = prefix[0], p1 = prefix[1], p2 = prefix[2], p3 = prefix[3];
    // ranks that still share their prefix share one histogram (all four in the first pass, usually the two of each end
    // afterwards): count once, copy after the pass
    const bool d1 = p1 != p0, d2 = p2 != p0 && p2 != p1, d3 = p3 != p0 && p3 != p1 && p3 != p2;
    for (long long i = threadIdx.x; i < n_round; i += blockDim.x) {
      const bool in = i < per_env;
      const uint32_t k = in ? f32_key(src[i]) : 0u;
      const uint32_t b = (k >> shift) & 0xffu, top = k & hi_mask;
      hist_add(hist[0], b, in && top == p0);
      if (d1) hist_add(hist[1], b, in && top == p1);
      if (d2) hist_add(hist[2], b, in && top == p2);
      if (d3) hist_add(hist[3], b, in && top == p3);
    }
    __syncthreads();
    if (threadIdx.x < 256) {
      const int b = threadIdx.x;
      if (!d1) hist[1][b] = hist[0][b];
      if (!d2) hist[2][b] = (p2 == p0) ? hist[0][b] : hist[1][b];
      if (!d3) hist[3][b] = (p3 == p0) ? hist[0][b] : (p3 == p1) ? hist[1][b] : hist[2][b];
    }
    __syncthreads();
    if (threadIdx.x < 4) {
      const int t = threadIdx.x;
      long long r = rank[t];
      int b = 0;
      for (; b < 255; ++b) {
        const unsigned c = hist[t][b];
        if (r < (long long)c) break;
        r -= c;
      }
      rank[t] = r;
      prefix[t] |= (uint32_t)b << shift;
    }
    __syncthreads();
  }
  const double a_lo = (double)key_f32(prefix[0]), b_lo = (double)key_f32(prefix[1]);
  const double a_hi = (double)key_f32(prefix[2]), b_hi = (double)key_f32(prefix[3]);
  const double p_low = np_lerp(a_lo, b_lo, __dsub_rn(vi_lo, (double)k_lo));
  const double p_high = np_lerp(a_hi, b_hi, __dsub_rn(vi_hi, (double)k_hi));
  if (stats && threadIdx.x == 0) { stats[2 * env] = p_low; stats[2 * env + 1] = p_high; }
  const bool ok = p_high > p_low;
  const double span = p_high - p_low;
  OUT* __restrict__ dst = out + (size_t)env * per_env;
  for (long long i = threadIdx.x; i < per_env; i += blockDim.x) {
    double v = ok ? ((double)src[i] - p_low) / span : 0.0;
    v = fmin(fmax(v, 0.0), 1.0);
    store_norm(dst + i, v);
  }
}

}  // namespace qd

namespace qd {
// raw fp32 -> half conversion of a sensor image (qd_scan_obs_host with normalise = 0, QD_Z_F16)
__global__ void __launch_bounds__(256) qd_to_half_kernel(const float* __restrict__ z, __half* __restrict__ out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = __float2half_rn(z[i]);
}
}  // namespace qd
