// qd_device.cuh -- small device helpers: Philox4x32-10, TMA bulk copy + mbarrier, warp utilities.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace qd {

// ---------------------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11).  Stream contract: see oracle/philox.py (the CPU checker implements the
// same contract).  key = 64-bit scan seed, counter = (index_lo, index_hi, purpose, sensor): c3 is the charge sensor
// whose noise the block feeds (0 for everything else).
// ---------------------------------------------------------------------------------------------------------------
struct Philox4 { uint32_t w0, w1, w2, w3; };

__device__ __forceinline__ Philox4 philox4x32_10(uint64_t seed, uint64_t index, uint32_t purpose, uint32_t sensor = 0u) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  uint32_t c0 = (uint32_t)index, c1 = (uint32_t)(index >> 32), c2 = purpose, c3 = sensor;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
  }
  return Philox4{c0, c1, c2, c3};
}

// uint32 -> uniform in [0,1) on the 2^-24 lattice (exact in fp32 and fp64)
__device__ __forceinline__ float u24(uint32_t w) { return (float)(w >> 8) * (1.0f / 16777216.0f); }

// Box-Muller on (w0, w1): two unit normals.
__device__ __forceinline__ void box_muller(uint32_t w0, uint32_t w1, float& z0, float& z1) {
  const float u1 = ((float)(w0 >> 8) + 1.0f) * (1.0f / 16777216.0f);   // (0, 1]
  const float u2 = u24(w1);
  const float r = sqrtf(-2.0f * logf(u1));
  float s, c;
  sincospif(2.0f * u2, &s, &c);
  z0 = r * c;
  z1 = r * s;
}

// ---------------------------------------------------------------------------------------------------------------
// TMA 1-D bulk copy global -> shared with mbarrier completion (SASS: UBLKCP / SYNCS).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "QD_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra QD_DONE_%=;\n"
      "bra QD_WAIT_%=;\n"
      "QD_DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// bytes must be a multiple of 16; src and dst 16-byte aligned
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// order prior generic-proxy accesses to shared memory before subsequent async-proxy (TMA) writes
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// min by one DSETP.LT + select pair (the C ternary is pattern-matched into DSETP.MIN plus NaN fix-ups: twice the work)
__device__ __forceinline__ double min_lt(double e, double m) {
  double r;
  asm("{\n .reg .pred p;\n setp.lt.f64 p, %1, %2;\n selp.f64 %0, %1, %2, p;\n}" : "=d"(r) : "d"(e), "d"(m));
  return r;
}

// MUFU.RCP, ~1 ulp: the Lorentzian sum tolerates it (DESIGN.md, error budget of the sensor signal)
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double shfl_f64(double v, int src) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_sync(0xffffffffu, lo, src);
  hi = __shfl_sync(0xffffffffu, hi, src);
  return __hiloint2double(hi, lo);
}
__device__ __forceinline__ uint64_t shfl_u64(uint64_t v, int src) {
  uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
  lo = __shfl_sync(0xffffffffu, lo, src);
  hi = __shfl_sync(0xffffffffu, hi, src);
  return ((uint64_t)hi << 32) | lo;
}

}  // namespace qd
