// raw2outputs: density -> alpha, exclusive-cumprod transmittance, weighted
// rgb/depth/acc.  One warp per ray (each lane a block of consecutive samples), shuffle scans, 128-bit loads.
//
// Spec: upstream nerf-pytorch raw2outputs as restated in SURVEY.md 8c-S1 (the
// reference tree only carries the pointer comment, src/run_nerf_helpers.py:131-133).
// HBM-bound: fwd moves 24*S+36 B/ray, bwd 40*S+36 B/ray (DESIGN.md).
#include "ctx_common.cuh"
#include <initializer_list>
#include <stdlib.h>

namespace ctx {

constexpr int kCompWarps = 8;  // warps per CTA
// rays longer than this take the chunked kernels (CTXNERF_COMP_SINGLE_MAX overrides it: tests, tuning)
static inline int comp_single_pass_max() {
  static const int v = [] {
    const char* e = getenv("CTXNERF_COMP_SINGLE_MAX");
    const int x = e ? atoi(e) : 512;
    return x < 1 ? 1 : (x > 512 ? 512 : x);
  }();
  return v;
}

struct SampleTerms {
  float alpha, trans_factor, expo;  // expo = exp(-relu(sigma)*dist) ; trans_factor = 1-alpha+1e-10
};

// sigmoid: 1 / (1 + e^-x) with the reciprocal as MUFU.RCP + one Newton step (error < 1 ulp, like the oracle's own
// exp).  The IEEE division the compiler emits for 1.0f / y carries a range check, a branch and a slow-path CALL per
// use -- with three sigmoids per sample that was a quarter of the kernels' instructions, and they are issue-bound.
// y is clamped to <= 1e30 so that the Newton step never sees inf * 0 (sigmoid(x) for x < -69 is then 1e-30, not e^x).
__device__ __forceinline__ float sigmoidf_(float x) {
  const float e = __expf(-x);                          // ex2.approx: |d sigmoid| <= s (1 - s) (2.4e-7 + 6e-8 |x|) < 1 ulp of 0.5
  const float y = 1.0f + ((e > 1e30f) ? 1e30f : e);    // (a comparison, not fminf: a NaN logit must stay NaN)
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(y));
  return fmaf(r, fmaf(-y, r, 1.0f), r);
}

__device__ __forceinline__ SampleTerms sample_terms(float sigma, float dist) {
  SampleTerms t;
  const float dens = (sigma < 0.0f) ? 0.0f : sigma;     // relu that keeps a NaN density a NaN (fmaxf would return 0)
  t.expo = expf(-dens * dist);
  t.alpha = 1.0f - t.expo;
  t.trans_factor = (1.0f - t.alpha) + 1e-10f;
  return t;
}

// inclusive product scan across a group of G consecutive lanes (`lane` = position inside the group)
template <int G>
__device__ __forceinline__ float group_scan_prod(float v, int lane) {
#pragma unroll
  for (int o = 1; o < G; o <<= 1) {
    const float n = __shfl_up_sync(CTX_FULL_MASK, v, o, G);
    if (lane >= o) v *= n;
  }
  return v;
}
template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(CTX_FULL_MASK, v, o, G);
  return v;
}

// Blocked sample-to-lane map: lane l owns the K consecutive samples [l*K, l*K+K) (S <= 32*K), so a ray costs ONE
// warp scan and ONE set of warp reductions whatever its length; the per-sample work is a serial pass over registers.
// K consecutive floats / float4 per lane keep every global access a whole number of 16- or 32-byte pieces.
template <int K>
__device__ __forceinline__ void load_row(const float* __restrict__ p, int64_t base, int s0, int S, int vec,
                                         float (&v)[K + 1]) {
  if ((K & 3) == 0 && vec >= 4) {
#pragma unroll
    for (int k = 0; k < K; k += 4) {
      const float4 q = (s0 + k < S) ? __ldg(reinterpret_cast<const float4*>(p + base + s0 + k))
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
      v[k] = q.x; v[k + 1] = q.y; v[k + 2] = q.z; v[k + 3] = q.w;
    }
  } else if ((K & 1) == 0 && vec >= 2) {
#pragma unroll
    for (int k = 0; k < K; k += 2) {
      const float2 q = (s0 + k < S) ? __ldg(reinterpret_cast<const float2*>(p + base + s0 + k)) : make_float2(0.f, 0.f);
      v[k] = q.x; v[k + 1] = q.y;
    }
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = (s0 + k < S) ? __ldg(p + base + s0 + k) : 0.f;
  }
}
template <int K>
__device__ __forceinline__ void store_row(float* __restrict__ p, int64_t base, int s0, int S, int vec,
                                          const float (&v)[K]) {
  if ((K & 3) == 0 && vec >= 4) {
#pragma unroll
    for (int k = 0; k < K; k += 4)
      if (s0 + k < S) *reinterpret_cast<float4*>(p + base + s0 + k) = make_float4(v[k], v[k + 1], v[k + 2], v[k + 3]);
  } else if ((K & 1) == 0 && vec >= 2) {
#pragma unroll
    for (int k = 0; k < K; k += 2)
      if (s0 + k < S) *reinterpret_cast<float2*>(p + base + s0 + k) = make_float2(v[k], v[k + 1]);
  } else {
#pragma unroll
    for (int k = 0; k < K; ++k)
      if (s0 + k < S) p[base + s0 + k] = v[k];
  }
}

// Density noise drawn inside the fused training pass (upstream raw2outputs: sigma + randn * raw_noise_std): sample s
// of ray r gets std * n, n the standard normal philox_normal4 gives for (key, stream, row r, col s), with
// key = seed + *seed_dev.  ctx_density_noise writes the same values as an [R,S] tensor.
struct NoiseRng {
  float std;
  uint64_t seed;
  const unsigned long long* seed_dev;   // nullable device counter added to seed (fresh numbers on every graph replay)
  uint32_t stream;
  __device__ __forceinline__ uint64_t key() const { return seed + (seed_dev ? *seed_dev : 0ull); }
};

// nz[k] = noise of samples s0 + k (k < K) of `ray`.  One Philox call serves a quad of samples; a lane whose K is a
// multiple of 4 starts on a quad (s0 = multiple of K), a lane of 3 or 6 samples straddles quads and picks its samples
// out of each quad it touches.
template <int K>
__device__ __forceinline__ void noise_row(const NoiseRng& g, uint64_t key, int64_t ray, int s0, float (&nz)[K + 1]) {
  const uint32_t q0 = (uint32_t)s0 >> 2;
  if constexpr ((K & 3) == 0) {
#pragma unroll
    for (int q = 0; q < K / 4; ++q) {
      const float4 n = philox_normal4(key, g.stream, (uint64_t)ray, q0 + q);
      nz[4 * q + 0] = __fmul_rn(g.std, n.x); nz[4 * q + 1] = __fmul_rn(g.std, n.y);
      nz[4 * q + 2] = __fmul_rn(g.std, n.z); nz[4 * q + 3] = __fmul_rn(g.std, n.w);
    }
  } else {
    const int off = s0 & 3;
    constexpr int NQ = (K + 6) / 4;              // most quads K consecutive samples can touch
#pragma unroll
    for (int j = 0; j < NQ; ++j) {
      if (4 * j < off + K) {
        const float4 n = philox_normal4(key, g.stream, (uint64_t)ray, q0 + j);
        const float v[4] = {n.x, n.y, n.z, n.w};
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (4 * j + e == off + k) nz[k] = __fmul_rn(g.std, v[e]);
      }
    }
  }
}

// G lanes share a ray (32 / G rays per warp): short rays use 8- or 16-lane groups so that the scan and the five
// reductions, the part of the work that does not shrink with S, are paid once per 4 or 2 rays.
template <int K, int G>
__global__ void __launch_bounds__(kCompWarps * 32, K <= 4 ? 4 : (K <= 8 ? 3 : (K <= 12 ? 2 : 1)))
composite_fwd_kernel(const float4* __restrict__ raw, const float* __restrict__ z,
                     const float* __restrict__ rays_d, const float* __restrict__ noise,
                     int64_t R, int S_all, int vec, int white_bkgd,
                     float* __restrict__ rgb_map, float* __restrict__ disp_map,
                     float* __restrict__ acc_map, float* __restrict__ weights,
                     float* __restrict__ depth_map) {
  constexpr int RPW = 32 / G;                        // rays per warp
  const int lane = threadIdx.x & (G - 1), sub = (threadIdx.x & 31) / G;
  const int64_t warp0 = (int64_t)blockIdx.x * kCompWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kCompWarps;
  const int s0 = lane * K;
  for (int64_t rb = warp0 * RPW; rb < R; rb += nwarps * RPW) {
    const bool live = rb + sub < R;                  // lane groups past the last ray only take part in the shuffles
    const int64_t ray = live ? rb + sub : R - 1;
    const int S = live ? S_all : 0;
    const float dx = rays_d[ray * 3 + 0], dy = rays_d[ray * 3 + 1], dz = rays_d[ray * 3 + 2];
    const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
    const int64_t base = ray * S_all;
    float4 rw[K];
    float zl[K + 1], nz[K + 1];
    // every load of the ray is issued up front
#pragma unroll
    for (int k = 0; k < K; ++k)
      rw[k] = (s0 + k < S) ? __ldg(raw + base + s0 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    load_row<K>(z, base, s0, S, vec, zl);
    if (noise != nullptr) load_row<K>(noise, base, s0, S, vec, nz);
    else {
#pragma unroll
      for (int k = 0; k < K; ++k) nz[k] = 0.f;
    }
    zl[K] = __shfl_down_sync(CTX_FULL_MASK, zl[0], 1, G);   // first depth of the next lane
    // serial pass: alpha and the transmittance prefix inside the lane
    float al[K], pref[K];
    float run = 1.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int s = s0 + k;
      const bool ok = s < S;
      const float dist = ((s == S - 1) ? 1e10f : (zl[k + 1] - zl[k])) * dnorm;
      const SampleTerms t = sample_terms(rw[k].w + nz[k], dist);
      al[k] = ok ? t.alpha : 0.f;
      pref[k] = run;
      run *= ok ? t.trans_factor : 1.0f;
    }
    const float incl = group_scan_prod<G>(run, lane);
    float excl = __shfl_up_sync(CTX_FULL_MASK, incl, 1, G);
    if (lane == 0) excl = 1.0f;
    float w[K];
    float sr = 0.f, sg = 0.f, sb = 0.f, sd = 0.f, sa = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      w[k] = al[k] * (excl * pref[k]);
      if (s0 + k < S) {
        sr += w[k] * sigmoidf_(rw[k].x);
        sg += w[k] * sigmoidf_(rw[k].y);
        sb += w[k] * sigmoidf_(rw[k].z);
        sd += w[k] * zl[k];
        sa += w[k];
      }
    }
    store_row<K>(weights, base, s0, S, vec, w);
    sr = group_sum<G>(sr); sg = group_sum<G>(sg); sb = group_sum<G>(sb); sd = group_sum<G>(sd); sa = group_sum<G>(sa);
    if (lane == 0 && live) {
      const float bg = white_bkgd ? (1.0f - sa) : 0.0f;
      rgb_map[ray * 3 + 0] = sr + bg;
      rgb_map[ray * 3 + 1] = sg + bg;
      rgb_map[ray * 3 + 2] = sb + bg;
      depth_map[ray] = sd;
      acc_map[ray] = sa;
      // 1/max(1e-10, depth/acc); NaN when acc == 0 (0/0 propagates through max in torch)
      const float q = sd / sa;
      disp_map[ray] = (q != q) ? q : 1.0f / fmaxf(1e-10f, q);
    }
  }
}

// Backward.  With t_k = 1-alpha_k+1e-10, T_i = prod_{k<i} t_k, w_i = alpha_i T_i and
// G_i = dL/dw_i:   dL/dalpha_i = T_i * (G_i - S_i),
//   S_i = sum_{j>i} G_j alpha_j prod_{i<k<j} t_k      (suffix affine scan; no division
// by t_i, which is 1e-10 at an opaque sample -- SURVEY.md H5).  S_i = U_{i+1} with
// U_j = b_j + a_j U_{j+1}, a_j = t_j, b_j = G_j alpha_j: composed inside the lane, scanned across lanes, and
// substituted back.
//
// TRAIN = true is the fused training form (NerfTrainer.step): the forward the backward has to recompute anyway
// also yields rgb_map, so the photometric loss img2mse(rgb_map, target) (src/run_nerf_helpers.py:9) and its
// gradient g_rgb = 2 (rgb_map - target) * loss_scale are formed in place -- one pass over raw replaces
// composite_fwd + mse + composite_bwd.  It writes g_raw, optionally weights (the coarse pass feeds sample_pdf) and
// rgb_map; the loss itself is summed from rgb_map by loss_sum_kernel, in a fixed order.
// RNG = true (TRAIN only): the density noise comes from `rng` instead of the `noise` rows.
template <int K, int G, bool TRAIN, bool RNG>
__global__ void __launch_bounds__(kCompWarps * 32, K <= 4 ? 4 : (K <= 8 ? 2 : 1))
composite_bwd_kernel(const float4* __restrict__ raw, const float* __restrict__ z,
                     const float* __restrict__ rays_d, const float* __restrict__ noise,
                     int64_t R, int S_all, int vec, int white_bkgd,
                     const float* __restrict__ g_rgb, const float* __restrict__ g_disp,
                     const float* __restrict__ g_acc, const float* __restrict__ g_weights,
                     const float* __restrict__ g_depth, float4* __restrict__ g_raw,
                     const float* __restrict__ target, float loss_scale, float* __restrict__ loss,
                     float* __restrict__ weights_out, float* __restrict__ rgb_out, NoiseRng rng) {
  constexpr int RPW = 32 / G;
  const int lane = threadIdx.x & (G - 1), sub = (threadIdx.x & 31) / G;
  const int64_t warp0 = (int64_t)blockIdx.x * kCompWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kCompWarps;
  const int s0 = lane * K;
  uint64_t key = 0;
  if constexpr (RNG) key = rng.key();
  for (int64_t rb = warp0 * RPW; rb < R; rb += nwarps * RPW) {
    const bool live = rb + sub < R;
    const int64_t ray = live ? rb + sub : R - 1;
    const int S = live ? S_all : 0;
    const float dx = rays_d[ray * 3 + 0], dy = rays_d[ray * 3 + 1], dz = rays_d[ray * 3 + 2];
    const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
    const int64_t base = ray * S_all;
    float4 rw[K];
    float zl[K + 1], nz[K + 1], gw[K + 1];
#pragma unroll
    for (int k = 0; k < K; ++k)
      rw[k] = (s0 + k < S) ? __ldg(raw + base + s0 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    load_row<K>(z, base, s0, S, vec, zl);
    if constexpr (RNG) noise_row<K>(rng, key, ray, s0, nz);
    else if (noise != nullptr) load_row<K>(noise, base, s0, S, vec, nz);
    else {
#pragma unroll
      for (int k = 0; k < K; ++k) nz[k] = 0.f;
    }
    if (!TRAIN && g_weights != nullptr) load_row<K>(g_weights, base, s0, S, vec, gw);
    else {
#pragma unroll
      for (int k = 0; k < K; ++k) gw[k] = 0.f;
    }
    zl[K] = __shfl_down_sync(CTX_FULL_MASK, zl[0], 1, G);
    // forward recompute: expo (alpha, t follow from it), the in-lane transmittance prefix, the ray totals
    float ex[K], dist[K], pref[K];
    float run = 1.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int s = s0 + k;
      const bool ok = s < S;
      dist[k] = ((s == S - 1) ? 1e10f : (zl[k + 1] - zl[k])) * dnorm;
      const SampleTerms t = sample_terms(rw[k].w + nz[k], dist[k]);
      ex[k] = ok ? t.expo : 1.0f;            // padded samples: alpha = 0, t = 1 + 1e-10 ~ identity (masked below)
      pref[k] = run;
      run *= ok ? t.trans_factor : 1.0f;
      // the colour logits are only ever used through their sigmoid: replace them in place, once (the forward sums,
      // G_k and the final gradients below then cost no further exp / division)
      rw[k].x = sigmoidf_(rw[k].x); rw[k].y = sigmoidf_(rw[k].y); rw[k].z = sigmoidf_(rw[k].z);
    }
    const float incl = group_scan_prod<G>(run, lane);
    float excl = __shfl_up_sync(CTX_FULL_MASK, incl, 1, G);
    if (lane == 0) excl = 1.0f;
    float sd = 0.f, sa = 0.f;
    float gr, gg, gb, gd, ga, gdisp;
    if constexpr (TRAIN) {
      float sr = 0.f, sg = 0.f, sb = 0.f;
      float wk[K];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        wk[k] = (1.0f - ex[k]) * (excl * pref[k]);
        if (s0 + k < S) {
          sr += wk[k] * rw[k].x;
          sg += wk[k] * rw[k].y;
          sb += wk[k] * rw[k].z;
          sa += wk[k];
        } else {
          wk[k] = 0.f;
        }
      }
      if (weights_out != nullptr) store_row<K>(weights_out, base, s0, S, vec, wk);
      sr = group_sum<G>(sr); sg = group_sum<G>(sg); sb = group_sum<G>(sb); sa = group_sum<G>(sa);
      const float bg = white_bkgd ? (1.0f - sa) : 0.0f;
      const float er = sr + bg - target[ray * 3 + 0], eg = sg + bg - target[ray * 3 + 1],
                  eb = sb + bg - target[ray * 3 + 2];
      gr = 2.0f * er * loss_scale; gg = 2.0f * eg * loss_scale; gb = 2.0f * eb * loss_scale;
      gd = 0.f; ga = 0.f; gdisp = 0.f;
      if (lane == 0 && live) {
        if (rgb_out != nullptr) { rgb_out[ray * 3 + 0] = sr + bg; rgb_out[ray * 3 + 1] = sg + bg; rgb_out[ray * 3 + 2] = sb + bg; }
      }
    } else {
#pragma unroll
      for (int k = 0; k < K; ++k) {
        if (s0 + k < S) {
          const float w = (1.0f - ex[k]) * (excl * pref[k]);
          sd += w * zl[k];
          sa += w;
        }
      }
      sd = group_sum<G>(sd); sa = group_sum<G>(sa);
      gr = g_rgb ? g_rgb[ray * 3 + 0] : 0.f;
      gg = g_rgb ? g_rgb[ray * 3 + 1] : 0.f;
      gb = g_rgb ? g_rgb[ray * 3 + 2] : 0.f;
      gd = g_depth ? g_depth[ray] : 0.f;
      ga = g_acc ? g_acc[ray] : 0.f;
      gdisp = g_disp ? g_disp[ray] : 0.f;
    }
    if (gdisp != 0.f) {  // disp = 1/max(1e-10, q), q = depth/acc
      const float q = sd / sa;
      if (q > 1e-10f) {
        const float dq = -gdisp / (q * q);
        gd += dq / sa;
        ga += -dq * sd / (sa * sa);
      } else if (q != q) {
        gd = q; ga = q;
      }
    }
    if (white_bkgd) ga -= (gr + gg + gb);
    // G_k, and the lane's composed map U_first = Bc + A * U_(first sample of the next lane)
    float Gs[K];
    float A = 1.0f, Bc = 0.f;
#pragma unroll
    for (int k = K - 1; k >= 0; --k) {
      const bool ok = s0 + k < S;
      const float cr = rw[k].x, cg = rw[k].y, cb = rw[k].z;
      Gs[k] = gw[k] + gr * cr + gg * cg + gb * cb + gd * zl[k] + ga;
      const float alpha = 1.0f - ex[k];
      const float a = ok ? ((1.0f - alpha) + 1e-10f) : 1.0f;
      const float b = ok ? Gs[k] * alpha : 0.f;
      Bc = b + a * Bc;
      A = a * A;
    }
    {
      float a = A, b = Bc;   // inclusive suffix scan over the lanes: (a, b) <- map of lanes [lane, 32)
#pragma unroll
      for (int o = 1; o < G; o <<= 1) {
        const float a2 = __shfl_down_sync(CTX_FULL_MASK, a, o, G);
        const float b2 = __shfl_down_sync(CTX_FULL_MASK, b, o, G);
        if (lane + o < G) { b = b + a * b2; a = a * a2; }
      }
      Bc = b;                // = U of this lane's first sample (U past the end of the ray is 0)
    }
    float U = __shfl_down_sync(CTX_FULL_MASK, Bc, 1, G);
    if (lane == G - 1) U = 0.f;
#pragma unroll
    for (int k = K - 1; k >= 0; --k) {
      const bool ok = s0 + k < S;
      const float alpha = 1.0f - ex[k];
      const float T = excl * pref[k];
      if (ok) {
        const float cr = rw[k].x, cg = rw[k].y, cb = rw[k].z;
        const float g_alpha = T * (Gs[k] - U);
        const float sig = rw[k].w + nz[k];
        const float g_sigma = (sig > 0.f) ? g_alpha * ex[k] * dist[k] : 0.f;
        const float w = alpha * T;
        float4 o4;
        o4.x = w * gr * cr * (1.0f - cr);
        o4.y = w * gg * cg * (1.0f - cg);
        o4.z = w * gb * cb * (1.0f - cb);
        o4.w = g_sigma;
        g_raw[base + s0 + k] = o4;
        U = Gs[k] * alpha + ((1.0f - alpha) + 1e-10f) * U;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Any number of samples per ray: the same blocked scheme run over CHUNKS of 32*K samples with carries -- the
// transmittance that enters a chunk on the way forward, the value of the reverse recurrence U that enters it on the
// way back.  Used beyond 512 samples per ray (the single-pass kernels keep a whole ray in registers) and for 257-512,
// where 16 samples per lane cost more registers than the second pass over a chunk costs time.
constexpr int kCompMaxChunks = 64;      // per-chunk entry transmittances kept in shared memory by the backward

// widest aligned vector access (floats) for rows of S floats behind the given pointers (device-side twin of comp_vec)
__device__ __forceinline__ int dev_vec(int S, const void* a, const void* b, const void* c) {
  const uintptr_t bits = reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c);
  return ((S & 3) == 0 && (bits & 15) == 0) ? 4 : 1;
}

template <int K, bool RNG = false>
__device__ __forceinline__ void chunk_load(const float4* __restrict__ raw, const float* __restrict__ z,
                                           const float* __restrict__ noise, int64_t base, int c0, int lane, int S,
                                           int vec, float dnorm, float4 (&rw)[K], float (&zl)[K + 1], float (&sig)[K],
                                           float (&dist)[K], const NoiseRng* rng = nullptr, uint64_t key = 0,
                                           int64_t ray = 0) {
  const int s0 = c0 + lane * K;
#pragma unroll
  for (int k = 0; k < K; ++k)
    rw[k] = (s0 + k < S) ? __ldg(raw + base + s0 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
  load_row<K>(z, base, s0, S, vec, zl);                        // 16-byte pieces when the rows allow it
  float nz[K + 1];
  if constexpr (RNG) {
    noise_row<K>(*rng, key, ray, s0, nz);
#pragma unroll
    for (int k = 0; k < K; ++k) sig[k] = rw[k].w + nz[k];
  } else {
    if (noise != nullptr) load_row<K>(noise, base, s0, S, vec, nz);
#pragma unroll
    for (int k = 0; k < K; ++k) sig[k] = rw[k].w + (noise != nullptr ? nz[k] : 0.f);
  }
  zl[K] = (s0 + K < S) ? __ldg(z + base + s0 + K) : 0.f;     // first depth of the next lane / next chunk
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int s = s0 + k;
    dist[k] = ((s == S - 1) ? 1e10f : (zl[k + 1] - zl[k])) * dnorm;
  }
}

template <int K>
__global__ void __launch_bounds__(kCompWarps * 32)
composite_chunked_fwd_kernel(const float4* __restrict__ raw, const float* __restrict__ z,
                             const float* __restrict__ rays_d, const float* __restrict__ noise, int64_t R, int S,
                             int white_bkgd, float* __restrict__ rgb_map, float* __restrict__ disp_map,
                             float* __restrict__ acc_map, float* __restrict__ weights, float* __restrict__ depth_map) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kCompWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kCompWarps;
  const int vec = dev_vec(S, z, noise, weights);
  for (int64_t ray = warp0; ray < R; ray += nwarps) {
    const float dx = rays_d[ray * 3 + 0], dy = rays_d[ray * 3 + 1], dz = rays_d[ray * 3 + 2];
    const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
    const int64_t base = ray * S;
    float carry = 1.0f, sr = 0.f, sg = 0.f, sb = 0.f, sd = 0.f, sa = 0.f;
    for (int c0 = 0; c0 < S; c0 += 32 * K) {
      float4 rw[K];
      float zl[K + 1], sig[K], dist[K];
      chunk_load<K>(raw, z, noise, base, c0, lane, S, vec, dnorm, rw, zl, sig, dist);
      float al[K], pref[K];
      float run = 1.0f;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const bool ok = c0 + lane * K + k < S;
        const SampleTerms t = sample_terms(sig[k], dist[k]);
        al[k] = ok ? t.alpha : 0.f;
        pref[k] = run;
        run *= ok ? t.trans_factor : 1.0f;
      }
      const float incl = group_scan_prod<32>(run, lane);
      float excl = __shfl_up_sync(CTX_FULL_MASK, incl, 1);
      if (lane == 0) excl = 1.0f;
      float wv[K];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const int s = c0 + lane * K + k;
        wv[k] = 0.f;
        if (s < S) {
          const float w = al[k] * ((carry * excl) * pref[k]);
          wv[k] = w;
          sr += w * sigmoidf_(rw[k].x); sg += w * sigmoidf_(rw[k].y); sb += w * sigmoidf_(rw[k].z);
          sd += w * zl[k]; sa += w;
        }
      }
      store_row<K>(weights, base, c0 + lane * K, S, vec, wv);
      carry *= __shfl_sync(CTX_FULL_MASK, incl, 31);
    }
    sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb); sd = warp_sum(sd); sa = warp_sum(sa);
    if (lane == 0) {
      const float bg = white_bkgd ? (1.0f - sa) : 0.0f;
      rgb_map[ray * 3 + 0] = sr + bg; rgb_map[ray * 3 + 1] = sg + bg; rgb_map[ray * 3 + 2] = sb + bg;
      depth_map[ray] = sd; acc_map[ray] = sa;
      const float q = sd / sa;
      disp_map[ray] = (q != q) ? q : 1.0f / fmaxf(1e-10f, q);
    }
  }
}

// backward / fused training form over chunks: pass 1 walks forward (entry transmittance of every chunk, ray totals),
// pass 2 walks the chunks in reverse with the incoming value of U (see composite_bwd_kernel for the recurrence).
template <int K, bool TRAIN, bool RNG>
__global__ void __launch_bounds__(kCompWarps * 32)
composite_chunked_bwd_kernel(const float4* __restrict__ raw, const float* __restrict__ z,
                             const float* __restrict__ rays_d, const float* __restrict__ noise, int64_t R, int S,
                             int white_bkgd, const float* __restrict__ g_rgb, const float* __restrict__ g_disp,
                             const float* __restrict__ g_acc, const float* __restrict__ g_weights,
                             const float* __restrict__ g_depth, float4* __restrict__ g_raw,
                             const float* __restrict__ target, float loss_scale, float* __restrict__ loss,
                             float* __restrict__ weights_out, float* __restrict__ rgb_out, NoiseRng rng) {
  __shared__ float s_carry[kCompWarps][kCompMaxChunks];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp0 = (int64_t)blockIdx.x * kCompWarps + wib;
  const int64_t nwarps = (int64_t)gridDim.x * kCompWarps;
  const int n_chunks = (S + 32 * K - 1) / (32 * K);
  const int vec = dev_vec(S, z, noise, TRAIN ? (const void*)weights_out : (const void*)g_weights);
  uint64_t key = 0;
  if constexpr (RNG) key = rng.key();
  for (int64_t ray = warp0; ray < R; ray += nwarps) {
    const float dx = rays_d[ray * 3 + 0], dy = rays_d[ray * 3 + 1], dz = rays_d[ray * 3 + 2];
    const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
    const int64_t base = ray * S;
    // ---- pass 1: forward ----
    float carry = 1.0f, sr = 0.f, sg = 0.f, sb = 0.f, sd = 0.f, sa = 0.f;
    for (int ci = 0; ci < n_chunks; ++ci) {
      const int c0 = ci * 32 * K;
      float4 rw[K];
      float zl[K + 1], sig[K], dist[K];
      chunk_load<K, RNG>(raw, z, noise, base, c0, lane, S, vec, dnorm, rw, zl, sig, dist, &rng, key, ray);
      if (lane == 0) s_carry[wib][ci] = carry;
      float al[K], pref[K];
      float run = 1.0f;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const bool ok = c0 + lane * K + k < S;
        const SampleTerms t = sample_terms(sig[k], dist[k]);
        al[k] = ok ? t.alpha : 0.f;
        pref[k] = run;
        run *= ok ? t.trans_factor : 1.0f;
      }
      const float incl = group_scan_prod<32>(run, lane);
      float excl = __shfl_up_sync(CTX_FULL_MASK, incl, 1);
      if (lane == 0) excl = 1.0f;
      float wv[K];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const int s = c0 + lane * K + k;
        wv[k] = 0.f;
        if (s < S) {
          const float w = al[k] * ((carry * excl) * pref[k]);
          wv[k] = w;
          if (TRAIN) { sr += w * sigmoidf_(rw[k].x); sg += w * sigmoidf_(rw[k].y); sb += w * sigmoidf_(rw[k].z); }
          sd += w * zl[k]; sa += w;
        }
      }
      if (TRAIN && weights_out != nullptr) store_row<K>(weights_out, base, c0 + lane * K, S, vec, wv);
      carry *= __shfl_sync(CTX_FULL_MASK, incl, 31);
    }
    sd = warp_sum(sd); sa = warp_sum(sa);
    float gr, gg, gb, gd, ga;
    if constexpr (TRAIN) {
      sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
      const float bg = white_bkgd ? (1.0f - sa) : 0.0f;
      const float er = sr + bg - target[ray * 3 + 0], eg = sg + bg - target[ray * 3 + 1], eb = sb + bg - target[ray * 3 + 2];
      gr = 2.0f * er * loss_scale; gg = 2.0f * eg * loss_scale; gb = 2.0f * eb * loss_scale;
      gd = 0.f; ga = 0.f;
      if (lane == 0 && rgb_out != nullptr) {
        rgb_out[ray * 3 + 0] = sr + bg; rgb_out[ray * 3 + 1] = sg + bg; rgb_out[ray * 3 + 2] = sb + bg;
      }
    } else {
      gr = g_rgb ? g_rgb[ray * 3 + 0] : 0.f; gg = g_rgb ? g_rgb[ray * 3 + 1] : 0.f; gb = g_rgb ? g_rgb[ray * 3 + 2] : 0.f;
      gd = g_depth ? g_depth[ray] : 0.f;
      ga = g_acc ? g_acc[ray] : 0.f;
      const float gdisp = g_disp ? g_disp[ray] : 0.f;
      if (gdisp != 0.f) {
        const float q = sd / sa;
        if (q > 1e-10f) {
          const float dq = -gdisp / (q * q);
          gd += dq / sa;
          ga += -dq * sd / (sa * sa);
        } else if (q != q) {
          gd = q; ga = q;
        }
      }
    }
    if (white_bkgd) ga -= (gr + gg + gb);
    __syncwarp();
    // ---- pass 2: reverse ----
    float carryU = 0.f;                         // U just past the end of the chunk being processed
    for (int ci = n_chunks - 1; ci >= 0; --ci) {
      const int c0 = ci * 32 * K;
      float4 rw[K];
      float zl[K + 1], sig[K], dist[K];
      chunk_load<K, RNG>(raw, z, noise, base, c0, lane, S, vec, dnorm, rw, zl, sig, dist, &rng, key, ray);
      const float cin = s_carry[wib][ci];
      float ex[K], pref[K], Gs[K];
      float run = 1.0f;
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const bool ok = c0 + lane * K + k < S;
        const SampleTerms t = sample_terms(sig[k], dist[k]);
        ex[k] = ok ? t.expo : 1.0f;
        pref[k] = run;
        run *= ok ? t.trans_factor : 1.0f;
      }
      const float incl = group_scan_prod<32>(run, lane);
      float excl = __shfl_up_sync(CTX_FULL_MASK, incl, 1);
      if (lane == 0) excl = 1.0f;
      // the lane's composed map  U_first = Bc + A * U_(first sample of the next lane)
      float A = 1.0f, Bc = 0.f;
      float gwv[K + 1];
      if (!TRAIN && g_weights != nullptr) load_row<K>(g_weights, base, c0 + lane * K, S, vec, gwv);
#pragma unroll
      for (int k = K - 1; k >= 0; --k) {
        const int s = c0 + lane * K + k;
        const bool ok = s < S;
        const float cr = sigmoidf_(rw[k].x), cg = sigmoidf_(rw[k].y), cb = sigmoidf_(rw[k].z);
        const float gw = (!TRAIN && g_weights != nullptr && ok) ? gwv[k] : 0.f;
        Gs[k] = gw + gr * cr + gg * cg + gb * cb + gd * zl[k] + ga;
        const float alpha = 1.0f - ex[k];
        const float a = ok ? ((1.0f - alpha) + 1e-10f) : 1.0f;
        const float b = ok ? Gs[k] * alpha : 0.f;
        Bc = b + a * Bc;
        A = a * A;
      }
      float a = A, b = Bc;                      // inclusive suffix composition over the lanes [lane, 32)
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float a2 = __shfl_down_sync(CTX_FULL_MASK, a, o);
        const float b2 = __shfl_down_sync(CTX_FULL_MASK, b, o);
        if (lane + o < 32) { b = b + a * b2; a = a * a2; }
      }
      // U at the first sample of the NEXT lane = map of lanes (lane, 32) applied to carryU
      float an = __shfl_down_sync(CTX_FULL_MASK, a, 1), bn = __shfl_down_sync(CTX_FULL_MASK, b, 1);
      if (lane == 31) { an = 1.0f; bn = 0.f; }
      float U = bn + an * carryU;
#pragma unroll
      for (int k = K - 1; k >= 0; --k) {
        const int s = c0 + lane * K + k;
        if (s < S) {
          const float alpha = 1.0f - ex[k];
          const float T = (cin * excl) * pref[k];
          const float cr = sigmoidf_(rw[k].x), cg = sigmoidf_(rw[k].y), cb = sigmoidf_(rw[k].z);
          const float g_alpha = T * (Gs[k] - U);
          const float g_sigma = (sig[k] > 0.f) ? g_alpha * ex[k] * dist[k] : 0.f;
          const float w = alpha * T;
          g_raw[base + s] = make_float4(w * gr * cr * (1.0f - cr), w * gg * cg * (1.0f - cg), w * gb * cb * (1.0f - cb), g_sigma);
          U = Gs[k] * alpha + ((1.0f - alpha) + 1e-10f) * U;
        }
      }
      // U at the first sample of this chunk = whole-chunk map applied to the incoming value
      const float a0 = __shfl_sync(CTX_FULL_MASK, a, 0), b0 = __shfl_sync(CTX_FULL_MASK, b, 0);
      carryU = b0 + a0 * carryU;
    }
    __syncwarp();
  }
}

// widest vector access (floats) that is aligned for every [R,S] row of the given pointers
static inline int comp_vec(int S, std::initializer_list<const void*> ptrs) {
  int vec = (S % 4 == 0) ? 4 : (S % 2 == 0 ? 2 : 1);
  for (const void* p : ptrs) {
    if (!p) continue;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    while (vec > 1 && (a % (vec * sizeof(float))) != 0) vec >>= 1;
  }
  return vec;
}

static inline int comp_grid(int64_t R, int S) {
  const int rpw = S <= 32 ? 4 : (S <= 64 ? 2 : 1);   // rays per warp of the dispatch below
  int64_t blocks = ceil_div(R, (int64_t)kCompWarps * rpw);
  const int64_t cap = (int64_t)num_sms() * 8;  // 8 CTAs of 8 warps = 64 warps/SM, grid-stride beyond
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace ctx

// K = samples per lane, G = lanes per ray (S <= G K)
#define CTX_COMP_DISPATCH(KERNEL, ...)                                                      \
  if (S <= 32) KERNEL<4, 8><<<grid, block, 0, st>>>(__VA_ARGS__);                          \
  else if (S <= 64) KERNEL<4, 16><<<grid, block, 0, st>>>(__VA_ARGS__);                    \
  else if (S <= 96) KERNEL<3, 32><<<grid, block, 0, st>>>(__VA_ARGS__);                    \
  else if (S <= 128) KERNEL<4, 32><<<grid, block, 0, st>>>(__VA_ARGS__);                   \
  else if (S <= 192) KERNEL<6, 32><<<grid, block, 0, st>>>(__VA_ARGS__);                   \
  else if (S <= 256) KERNEL<8, 32><<<grid, block, 0, st>>>(__VA_ARGS__);                   \
  else if (S <= 384) KERNEL<12, 32><<<grid, block, 0, st>>>(__VA_ARGS__);                  \
  else KERNEL<16, 32><<<grid, block, 0, st>>>(__VA_ARGS__);

#define CTX_COMP_DISPATCH_BWD(TRAIN, RNG, ...)                                                                   \
  if (S <= 32) ctx::composite_bwd_kernel<4, 8, TRAIN, RNG><<<grid, block, 0, st>>>(__VA_ARGS__);                    \
  else if (S <= 64) ctx::composite_bwd_kernel<4, 16, TRAIN, RNG><<<grid, block, 0, st>>>(__VA_ARGS__);              \
  else if (S <= 96) ctx::composite_bwd_kernel<3, 32, TRAIN, RNG><<<grid, block, 0, st>>>(__VA_ARGS__);              \
  else if (S <= 128) ctx::composite_bwd_kernel<4, 32, TRAIN, RNG><<<grid, block, 0, st>>>(__VA_ARGS__);             \
  else if (S <= 192) ctx::composite_bwd_kernel<6, 32, TRAIN, RNG><<<grid, block, 0, st>>>(__VA_ARGS__);             \
  else if (S <= 256) ctx::composite_bwd_kernel<8, 32, TRAIN, RNG><<<grid, block, 0, st>>>(__VA_ARGS__);             \
  else if (S <= 384) ctx::composite_bwd_kernel<12, 32, TRAIN, RNG><<<grid, block, 0, st>>>(__VA_ARGS__);            \
  else ctx::composite_bwd_kernel<16, 32, TRAIN, RNG><<<grid, block, 0, st>>>(__VA_ARGS__);

extern "C" int ctx_composite_fwd(const float* raw, const float* z_vals, const float* rays_d,
                                 const float* noise, int64_t R, int S, int white_bkgd,
                                 float* rgb_map, float* disp_map, float* acc_map, float* weights,
                                 float* depth_map, void* stream) {
  if (R < 0 || S < 1 || S > 256 * ctx::kCompMaxChunks) return CTX_ERR_BAD_ARG;
  if (R == 0) return 0;
  if (!raw || !z_vals || !rays_d || !rgb_map || !disp_map || !acc_map || !weights || !depth_map)
    return CTX_ERR_BAD_ARG;
  if (reinterpret_cast<uintptr_t>(raw) % 16 != 0) return CTX_ERR_BAD_ARG;   // raw is read as float4 (128-bit loads)
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = ctx::comp_grid(R, S), block = ctx::kCompWarps * 32;
  // (forward: beyond 384 samples the 16-samples-per-lane single pass is slower than two chunks of 8 per lane --
  //  36 % vs 52 % of the copy bandwidth at S = 512; the backward keeps its single pass up to 512: 41 % vs 36 %)
  if (S > (ctx::comp_single_pass_max() < 384 ? ctx::comp_single_pass_max() : 384)) {
    ctx::composite_chunked_fwd_kernel<8><<<grid, block, 0, st>>>((const float4*)raw, z_vals, rays_d, noise, R, S,
                                                                white_bkgd, rgb_map, disp_map, acc_map, weights, depth_map);
    CTX_RETURN_LAST();
  }
  const int vec = ctx::comp_vec(S, {z_vals, noise, weights});
  CTX_COMP_DISPATCH(ctx::composite_fwd_kernel, (const float4*)raw, z_vals, rays_d, noise, R, S, vec,
                    white_bkgd, rgb_map, disp_map, acc_map, weights, depth_map)
  CTX_RETURN_LAST();
}

extern "C" int ctx_composite_bwd(const float* raw, const float* z_vals, const float* rays_d,
                                 const float* noise, int64_t R, int S, int white_bkgd,
                                 const float* g_rgb, const float* g_disp, const float* g_acc,
                                 const float* g_weights, const float* g_depth, float* g_raw,
                                 void* stream) {
  if (R < 0 || S < 1 || S > 256 * ctx::kCompMaxChunks) return CTX_ERR_BAD_ARG;
  if (R == 0) return 0;
  if (!raw || !z_vals || !rays_d || !g_raw) return CTX_ERR_BAD_ARG;
  if (reinterpret_cast<uintptr_t>(raw) % 16 != 0 || reinterpret_cast<uintptr_t>(g_raw) % 16 != 0)
    return CTX_ERR_BAD_ARG;                                                  // float4 loads / stores
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = ctx::comp_grid(R, S), block = ctx::kCompWarps * 32;
  if (S > ctx::comp_single_pass_max()) {
    ctx::composite_chunked_bwd_kernel<8, false, false><<<grid, block, 0, st>>>(
        (const float4*)raw, z_vals, rays_d, noise, R, S, white_bkgd, g_rgb, g_disp, g_acc, g_weights, g_depth,
        (float4*)g_raw, nullptr, 0.f, nullptr, nullptr, nullptr, ctx::NoiseRng{});
    CTX_RETURN_LAST();
  }
  const int vec = ctx::comp_vec(S, {z_vals, noise, g_weights});
  CTX_COMP_DISPATCH_BWD(false, false, (const float4*)raw, z_vals, rays_d, noise, R, S, vec, white_bkgd, g_rgb,
                        g_disp, g_acc, g_weights, g_depth, (float4*)g_raw, nullptr, 0.f, nullptr, nullptr, nullptr,
                        ctx::NoiseRng{})
  CTX_RETURN_LAST();
}

namespace ctx {
// loss[0] += loss_scale * sum over rays of |rgb - target|^2: one block, every thread a fixed strided set of rays, then
// a fixed reduction tree, so the loss is the same on every run (atomics from many blocks would sum in arrival order).
__global__ void __launch_bounds__(1024) loss_sum_kernel(const float* __restrict__ rgb, const float* __restrict__ target,
                                                        int64_t R, float loss_scale, float* __restrict__ loss) {
  __shared__ float s_part[32];
  float acc = 0.f;
  for (int64_t r = threadIdx.x; r < R; r += blockDim.x) {
    const float er = rgb[r * 3 + 0] - target[r * 3 + 0], eg = rgb[r * 3 + 1] - target[r * 3 + 1],
                eb = rgb[r * 3 + 2] - target[r * 3 + 2];
    acc += (er * er + eg * eg + eb * eb) * loss_scale;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? s_part[threadIdx.x] : 0.f;
    acc = warp_sum(acc);
    if (threadIdx.x == 0) loss[0] += acc;
  }
}
}  // namespace ctx

namespace ctx {
// the launches behind ctx_composite_train (RNG = false: the `noise` rows, if any) and ctx_composite_train_noise
// (RNG = true: noise drawn in-kernel from `rng`)
template <bool RNG>
static int composite_train_launch(const float* raw, const float* z_vals, const float* rays_d, const float* noise,
                                  int64_t R, int S, int white_bkgd, const float* target, float loss_scale, float* loss,
                                  float* g_raw, float* weights, float* rgb_map, NoiseRng rng, cudaStream_t st) {
  const int grid = comp_grid(R, S), block = kCompWarps * 32;
  if (S > comp_single_pass_max()) {
    composite_chunked_bwd_kernel<8, true, RNG><<<grid, block, 0, st>>>(
        (const float4*)raw, z_vals, rays_d, noise, R, S, white_bkgd, nullptr, nullptr, nullptr, nullptr, nullptr,
        (float4*)g_raw, target, loss_scale, nullptr, weights, rgb_map, rng);
  } else {
    const int vec = comp_vec(S, {z_vals, noise, weights});
    CTX_COMP_DISPATCH_BWD(true, RNG, (const float4*)raw, z_vals, rays_d, noise, R, S, vec, white_bkgd, nullptr,
                          nullptr, nullptr, nullptr, nullptr, (float4*)g_raw, target, loss_scale, nullptr, weights,
                          rgb_map, rng)
  }
  loss_sum_kernel<<<1, 1024, 0, st>>>(rgb_map, target, R, loss_scale, loss);
  CTX_RETURN_LAST();
}

// [R,S] rows of the in-kernel density noise: one thread per quad of samples, the Philox call the fused pass makes
__global__ void density_noise_kernel(float* __restrict__ out, int64_t R, int S, NoiseRng g) {
  const uint64_t key = g.key();
  const int nq = (S + 3) >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < R * nq; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / nq;
    const int q = (int)(i - r * nq);
    const float4 n = philox_normal4(key, g.stream, (uint64_t)r, (uint32_t)q);
    const float v[4] = {n.x, n.y, n.z, n.w};
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (4 * q + e < S) out[r * S + 4 * q + e] = __fmul_rn(g.std, v[e]);
  }
}

// streams 0 and 1 of the step's key are the stratified jitter and the sample_pdf uniforms
static inline bool noise_args_ok(float noise_std, int stream_id) { return noise_std >= 0.f && stream_id >= 2; }
}  // namespace ctx

// Fused training form of raw2outputs: forward + img2mse(rgb_map, target) + backward in one pass (see the kernel),
// then the loss from rgb_map (loss_sum_kernel).  loss_scale = 1 / (3 R) for the mean over the rgb image; loss[0] is
// ADDED to (zero it once per step: the coarse and the fine pass accumulate into the same scalar).  weights is an
// optional output.
extern "C" int ctx_composite_train(const float* raw, const float* z_vals, const float* rays_d, const float* noise,
                                   int64_t R, int S, int white_bkgd, const float* target, float loss_scale,
                                   float* loss, float* g_raw, float* weights, float* rgb_map, void* stream) {
  if (R < 0 || S < 1 || S > 256 * ctx::kCompMaxChunks) return CTX_ERR_BAD_ARG;
  if (R == 0) return 0;
  if (!raw || !z_vals || !rays_d || !target || !loss || !g_raw || !rgb_map) return CTX_ERR_BAD_ARG;
  if (reinterpret_cast<uintptr_t>(raw) % 16 != 0 || reinterpret_cast<uintptr_t>(g_raw) % 16 != 0)
    return CTX_ERR_BAD_ARG;
  return ctx::composite_train_launch<false>(raw, z_vals, rays_d, noise, R, S, white_bkgd, target, loss_scale, loss,
                                            g_raw, weights, rgb_map, ctx::NoiseRng{}, (cudaStream_t)stream);
}

// ctx_composite_train with the density noise noise_std * n drawn inside the kernel (the values ctx_density_noise
// writes), so that a captured training step needs no noise tensor made before each replay.  noise_std == 0 runs
// exactly the launches of ctx_composite_train without noise.
extern "C" int ctx_composite_train_noise(const float* raw, const float* z_vals, const float* rays_d, int64_t R, int S,
                                         int white_bkgd, const float* target, float loss_scale, float* loss,
                                         float* g_raw, float* weights, float* rgb_map, float noise_std, uint64_t seed,
                                         const uint64_t* seed_dev, int stream_id, void* stream) {
  if (R < 0 || S < 1 || S > 256 * ctx::kCompMaxChunks || !ctx::noise_args_ok(noise_std, stream_id))
    return CTX_ERR_BAD_ARG;
  if (!raw || !z_vals || !rays_d || !target || !loss || !g_raw || !rgb_map) return CTX_ERR_BAD_ARG;
  if (reinterpret_cast<uintptr_t>(raw) % 16 != 0 || reinterpret_cast<uintptr_t>(g_raw) % 16 != 0)
    return CTX_ERR_BAD_ARG;
  if (R == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (noise_std == 0.f)
    return ctx::composite_train_launch<false>(raw, z_vals, rays_d, nullptr, R, S, white_bkgd, target, loss_scale,
                                              loss, g_raw, weights, rgb_map, ctx::NoiseRng{}, st);
  const ctx::NoiseRng rng{noise_std, seed, reinterpret_cast<const unsigned long long*>(seed_dev), (uint32_t)stream_id};
  return ctx::composite_train_launch<true>(raw, z_vals, rays_d, nullptr, R, S, white_bkgd, target, loss_scale, loss,
                                           g_raw, weights, rgb_map, rng, st);
}

extern "C" int ctx_density_noise(float* noise, int64_t R, int S, float noise_std, uint64_t seed,
                                 const uint64_t* seed_dev, int stream_id, void* stream) {
  if (R < 0 || S < 1 || !noise || !ctx::noise_args_ok(noise_std, stream_id)) return CTX_ERR_BAD_ARG;
  if (R == 0) return 0;
  int64_t blocks = ctx::ceil_div(R * ((S + 3) / 4), 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  const ctx::NoiseRng rng{noise_std, seed, reinterpret_cast<const unsigned long long*>(seed_dev), (uint32_t)stream_id};
  ctx::density_noise_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(noise, R, S, rng);
  CTX_RETURN_LAST();
}
