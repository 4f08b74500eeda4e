// Shared device/host helpers for the ctxnerf kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#define CTX_ERR_BAD_ARG (-1)
#define CTX_ERR_UNSUPPORTED (-2)
#define CTX_ERR_NO_NCCL (-3)

#define CTX_FULL_MASK 0xffffffffu

// Launch-check used by every extern "C" launcher: returns the cudaError_t as int.
#define CTX_RETURN_LAST()                              \
  do {                                                 \
    cudaError_t _e = cudaGetLastError();               \
    return (int)_e;                                    \
  } while (0)

namespace ctx {

constexpr int kNumSMs = 148;  // B200 (compile-time sizing of job tables); launch geometry uses num_sms()

// SM count of the current device (cached per device): grids and SM budgets follow the part the code runs on
inline int num_sms() {
  static int cached[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return kNumSMs;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = kNumSMs;
    cached[dev] = n;
  }
  return cached[dev];
}

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(CTX_FULL_MASK, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(CTX_FULL_MASK, v, o);
  return v;
}

// torch.linspace(start, end, n)[i] in fp32: two-sided, one rounding per element
// (SURVEY.md H1; verified against the reference's torch.linspace in
// tests/golden).  step = (end-start)/(n-1) rounded to fp32.
__device__ __forceinline__ float linspace_at(float start, float end, int n, int i) {
  if (n <= 1) return start;
  const float step = __fdiv_rn(__fsub_rn(end, start), (float)(n - 1));
  return (i < n / 2) ? fmaf(step, (float)i, start) : fmaf(-step, (float)(n - 1 - i), end);
}

// Philox4x32-10 counter RNG (own implementation of the published algorithm;
// Salmon et al., SC'11).  Used when the caller does not hand in uniforms.
struct Philox {
  uint32_t k0, k1;
  __device__ Philox(uint64_t seed) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)) {}
  __device__ __forceinline__ uint4 operator()(uint64_t ctr_lo, uint64_t ctr_hi) const {
    uint32_t c0 = (uint32_t)ctr_lo, c1 = (uint32_t)(ctr_lo >> 32);
    uint32_t c2 = (uint32_t)ctr_hi, c3 = (uint32_t)(ctr_hi >> 32);
    uint32_t a = k0, b = k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      c0 = hi1 ^ c1 ^ a; c1 = lo1; c2 = hi0 ^ c3 ^ b; c3 = lo0;
      a += 0x9E3779B9u; b += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};
// 24-bit uniform in [0,1)
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

// one uniform for (stream, row, col): 4 consecutive cols share one Philox call
__device__ __forceinline__ float philox_uniform(uint64_t seed, uint64_t stream, uint64_t row, uint32_t col) {
  Philox ph(seed);
  const uint4 r = ph(row, (stream << 32) | (uint64_t)(col >> 2));
  const uint32_t sel = col & 3u;
  return u01(sel == 0 ? r.x : sel == 1 ? r.y : sel == 2 ? r.z : r.w);
}

// four standard normals for (stream, row, cols 4q .. 4q+3): the Philox call of philox_uniform's layout, then
// Box-Muller on (x, y) and (z, w), cos then sin.  The radius uniform lies in (0, 1] so that log never sees 0 (|n| is
// at most sqrt(48 ln 2) = 5.77).  Explicitly rounded products: callers that inline this keep the same bits whatever
// they do with the result.
__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint64_t stream, uint64_t row, uint32_t quad) {
  Philox ph(seed);
  const uint4 r = ph(row, (stream << 32) | (uint64_t)quad);
  const float ua = (float)((r.x >> 8) + 1u) * (1.0f / 16777216.0f), ta = u01(r.y);
  const float ub = (float)((r.z >> 8) + 1u) * (1.0f / 16777216.0f), tb = u01(r.w);
  const float ra = sqrtf(__fmul_rn(-2.0f, logf(ua))), rb = sqrtf(__fmul_rn(-2.0f, logf(ub)));
  float sa, ca, sb, cb;
  sincospif(__fmul_rn(2.0f, ta), &sa, &ca);
  sincospif(__fmul_rn(2.0f, tb), &sb, &cb);
  return make_float4(__fmul_rn(ra, ca), __fmul_rn(ra, sa), __fmul_rn(rb, cb), __fmul_rn(rb, sb));
}

// cudaFuncSetAttribute is per device: remember which devices a launcher has already prepared (one process may drive
// several GPUs even though the training path uses one process per GPU)
struct DeviceOnce {
  bool done[64] = {};
  bool needed() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
    if (done[dev]) return false;
    done[dev] = true;
    return true;
  }
};

}  // namespace ctx
