// Per-image reconstruction metrics of a batch of rendered images against their targets: the MSE behind upstream's
// img2mse / mse2psnr (src/run_nerf_helpers.py:9-10), and SSIM as the compute_ssim of Google's mip-NeRF / MultiNeRF
// defines it with max_val = 1 (restated in oracle/image_metrics.py):
//   window: 11 taps g_i = exp(-0.5 ((i - 5) / 1.5)^2), normalised to sum 1, applied along x then along y, valid mode
//   per channel: mu_x = f(x), mu_y = f(y), s_xx = max(0, f(x^2) - mu_x^2), s_yy likewise,
//                s_xy = f(xy) - mu_x mu_y clipped to sign(s_xy) min(sqrt(s_xx s_yy), |s_xy|)
//   map = ((2 mu_x mu_y + c1)(2 s_xy + c2)) / ((mu_x^2 + mu_y^2 + c1)(s_xx + s_yy + c2)), c1 = 0.01^2, c2 = 0.03^2
//   ssim = mean of the map over the three channels and the (H-10) x (W-10) valid positions.
//
// One CTA per (image, 32 x 32 tile).  The tile owns the pixels [y0, y0+32) x [x0, x0+32) for the squared error and the
// map positions with the same coordinates (position m filters pixels m .. m+10), so it stages 42 x 42 pixels of both
// images in shared memory once; the horizontal pass and then the vertical pass run out of shared memory.  Every pixel
// belongs to exactly one tile, so the SSE counts each pixel once, the 5-pixel border included.
//
// The moments are formed in fp64: f(x^2) - mu_x^2 cancels, and in fp32 its rounding error (~1e-7) is not small
// against c2 = 9e-4 in flat regions.  x^2 and xy of fp32 inputs are exact in fp64, so the only roundings are the
// weighted sums.  The squared differences are formed in fp32 (pred - target) and squared and summed in fp64.
//
// Deterministic, without floating-point atomics: each CTA writes its two fp64 sums to `partials`, and a second launch
// adds each image's partials with one warp (lane l takes tiles l, l+32, ..., then a fixed shuffle tree).  Nothing
// depends on B or on the other images of the batch.
#include "ctx_common.cuh"

#include <climits>
#include <cmath>

namespace ctx {

constexpr int kMetTile = 32;                        // pixels (and map positions) per tile side
constexpr int kMetWin = 11;                         // SSIM window taps
constexpr int kMetStage = kMetTile + kMetWin - 1;   // staged rows / cols: the tile and its 10-pixel halo
constexpr int kMetThreads = 256;
// horizontal sums [5][kMetStage][kMetTile] fp64, then the staged pixels [2 images][3 channels][kMetStage][kMetStage]
constexpr int kMetSmem = 5 * kMetStage * kMetTile * 8 + 2 * 3 * kMetStage * kMetStage * 4;

struct MetricParams {
  const float* pred;
  const void* target;
  int target_u8;
  int H, W, tiles_x, tiles;     // tiles per image
  int want_ssim;
  double g[kMetWin];            // normalised Gaussian taps
  double* partials;             // [B * tiles][2]: SSE, sum of the SSIM map over the tile's positions and channels
};

__global__ void __launch_bounds__(kMetThreads) image_metrics_kernel(MetricParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  double* hs = reinterpret_cast<double*>(smem);                 // [5][kMetStage][kMetTile]
  float* sp = reinterpret_cast<float*>(hs + 5 * kMetStage * kMetTile);   // pred   [3][kMetStage][kMetStage]
  float* st = sp + 3 * kMetStage * kMetStage;                              // target [3][kMetStage][kMetStage]
  __shared__ double red[2][kMetThreads / 32];

  const int64_t b = blockIdx.x / p.tiles;
  const int tile = (int)(blockIdx.x - b * p.tiles);
  const int ty = tile / p.tiles_x, tx = tile - ty * p.tiles_x;
  const int y0 = ty * kMetTile, x0 = tx * kMetTile;
  const int rows = min(kMetStage, p.H - y0), cols = min(kMetStage, p.W - x0);   // staged pixels inside the image
  const int64_t base = b * (int64_t)p.H * p.W * 3;

  // stage: consecutive threads read consecutive floats of an image row; pixels outside the image read as 0 (they
  // feed only map positions outside the valid map)
  for (int i = threadIdx.x; i < kMetStage * kMetStage * 3; i += kMetThreads) {
    const int sy = i / (kMetStage * 3), r = i - sy * (kMetStage * 3);
    const int sx = r / 3, c = r - sx * 3;
    float a = 0.0f, t = 0.0f;
    if (sy < rows && sx < cols) {
      const int64_t gi = base + ((int64_t)(y0 + sy) * p.W + (x0 + sx)) * 3 + c;
      a = __ldg(p.pred + gi);
      t = p.target_u8 ? __fdiv_rn((float)__ldg(static_cast<const unsigned char*>(p.target) + gi), 255.0f)
                      : __ldg(static_cast<const float*>(p.target) + gi);
    }
    sp[(c * kMetStage + sy) * kMetStage + sx] = a;
    st[(c * kMetStage + sy) * kMetStage + sx] = t;
  }
  __syncthreads();

  // squared error of the pixels the tile owns
  double sse = 0.0;
  for (int i = threadIdx.x; i < kMetTile * kMetTile; i += kMetThreads) {
    const int sy = i / kMetTile, sx = i - sy * kMetTile;
    if (sy < rows && sx < cols) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int s = (c * kMetStage + sy) * kMetStage + sx;
        const double d = (double)__fsub_rn(sp[s], st[s]);
        sse = fma(d, d, sse);
      }
    }
  }

  // SSIM map over the tile's valid positions, one channel at a time
  double ssum = 0.0;
  const int my = min(kMetTile, p.H - (kMetWin - 1) - y0), mx = min(kMetTile, p.W - (kMetWin - 1) - x0);
  if (p.want_ssim && my > 0 && mx > 0) {
    for (int c = 0; c < 3; ++c) {
      const float* a = sp + c * kMetStage * kMetStage;
      const float* t = st + c * kMetStage * kMetStage;
      for (int i = threadIdx.x; i < kMetStage * kMetTile; i += kMetThreads) {   // along x
        const int sy = i / kMetTile, ox = i - sy * kMetTile;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0, s4 = 0.0;
#pragma unroll
        for (int k = 0; k < kMetWin; ++k) {
          const double x = a[sy * kMetStage + ox + k], y = t[sy * kMetStage + ox + k], w = p.g[k];
          s0 = fma(w, x, s0);
          s1 = fma(w, y, s1);
          s2 = fma(w, x * x, s2);
          s3 = fma(w, y * y, s3);
          s4 = fma(w, x * y, s4);
        }
        double* h = hs + sy * kMetTile + ox;
        h[0] = s0;
        h[kMetStage * kMetTile] = s1;
        h[2 * kMetStage * kMetTile] = s2;
        h[3 * kMetStage * kMetTile] = s3;
        h[4 * kMetStage * kMetTile] = s4;
      }
      __syncthreads();
      for (int i = threadIdx.x; i < kMetTile * kMetTile; i += kMetThreads) {     // along y
        const int oy = i / kMetTile, ox = i - oy * kMetTile;
        if (oy < my && ox < mx) {
          double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
          const double* h = hs + oy * kMetTile + ox;
#pragma unroll
          for (int k = 0; k < kMetWin; ++k) {
            const double w = p.g[k];
            m0 = fma(w, h[k * kMetTile], m0);
            m1 = fma(w, h[kMetStage * kMetTile + k * kMetTile], m1);
            m2 = fma(w, h[2 * kMetStage * kMetTile + k * kMetTile], m2);
            m3 = fma(w, h[3 * kMetStage * kMetTile + k * kMetTile], m3);
            m4 = fma(w, h[4 * kMetStage * kMetTile + k * kMetTile], m4);
          }
          const double sxx = fmax(0.0, m2 - m0 * m0), syy = fmax(0.0, m3 - m1 * m1);
          double sxy = m4 - m0 * m1;
          sxy = copysign(fmin(sqrt(sxx * syy), fabs(sxy)), sxy);
          const double c1 = 0.01 * 0.01, c2 = 0.03 * 0.03;
          ssum += ((2.0 * m0 * m1 + c1) * (2.0 * sxy + c2)) / ((m0 * m0 + m1 * m1 + c1) * (sxx + syy + c2));
        }
      }
      __syncthreads();      // the next channel overwrites hs
    }
  }

  // block sums in a fixed order
  sse = warp_sum(sse);
  ssum = warp_sum(ssum);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    red[0][warp] = sse;
    red[1][warp] = ssum;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double e = 0.0, s = 0.0;
#pragma unroll
    for (int w = 0; w < kMetThreads / 32; ++w) {
      e += red[0][w];
      s += red[1][w];
    }
    p.partials[2 * (int64_t)blockIdx.x] = e;
    p.partials[2 * (int64_t)blockIdx.x + 1] = s;
  }
}

// one warp per image: its tiles' partials, lane l summing tiles l, l+32, ... in order, then a fixed shuffle tree
__global__ void __launch_bounds__(kMetThreads) image_metrics_finish_kernel(const double* partials, int B, int tiles,
                                                                           double n_px, double n_map, double* mse,
                                                                           double* ssim) {
  const int64_t img = ((int64_t)blockIdx.x * kMetThreads + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (img >= B) return;                     // whole warps only
  const double* pp = partials + img * tiles * 2;
  double e = 0.0, s = 0.0;
  for (int t = lane; t < tiles; t += 32) {
    e += pp[2 * t];
    s += pp[2 * t + 1];
  }
  e = warp_sum(e);
  s = warp_sum(s);
  if (lane == 0) {
    if (mse) mse[img] = e / n_px;
    if (ssim) ssim[img] = s / n_map;
  }
}

}  // namespace ctx

extern "C" int64_t ctx_image_metrics_partials(int B, int H, int W) {
  if (B < 0 || H < 1 || W < 1) return CTX_ERR_BAD_ARG;
  return 2 * (int64_t)B * ctx::ceil_div(H, ctx::kMetTile) * ctx::ceil_div(W, ctx::kMetTile);
}

extern "C" int ctx_image_metrics(const float* pred, const void* target, int target_u8, int B, int H, int W,
                                 double* mse, double* ssim, double* partials, void* stream) {
  if (B < 0 || H < 1 || W < 1 || (target_u8 != 0 && target_u8 != 1)) return CTX_ERR_BAD_ARG;
  if (ssim && (H < ctx::kMetWin || W < ctx::kMetWin)) return CTX_ERR_BAD_ARG;   // no valid SSIM position
  if (B == 0) return 0;
  if (!pred || !target || !partials) return CTX_ERR_BAD_ARG;
  const int tiles_x = (int)ctx::ceil_div(W, ctx::kMetTile);
  const int64_t tiles = tiles_x * ctx::ceil_div(H, ctx::kMetTile);
  if ((int64_t)B * tiles > INT_MAX) return CTX_ERR_BAD_ARG;
  ctx::MetricParams p;
  p.pred = pred; p.target = target; p.target_u8 = target_u8;
  p.H = H; p.W = W; p.tiles_x = tiles_x; p.tiles = (int)tiles;
  p.want_ssim = ssim != nullptr;
  double gsum = 0.0;
  for (int i = 0; i < ctx::kMetWin; ++i) {
    const double u = (i - 5) / 1.5;
    p.g[i] = std::exp(-0.5 * u * u);
    gsum += p.g[i];
  }
  for (int i = 0; i < ctx::kMetWin; ++i) p.g[i] /= gsum;
  p.partials = partials;
  static ctx::DeviceOnce once;
  if (once.needed()) {
    cudaError_t e = cudaFuncSetAttribute(ctx::image_metrics_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         ctx::kMetSmem);
    if (e != cudaSuccess) return (int)e;
  }
  cudaStream_t s = (cudaStream_t)stream;
  ctx::image_metrics_kernel<<<(int)(B * tiles), ctx::kMetThreads, ctx::kMetSmem, s>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  const double n_map = 3.0 * (double)(H - (ctx::kMetWin - 1)) * (double)(W - (ctx::kMetWin - 1));
  ctx::image_metrics_finish_kernel<<<(int)ctx::ceil_div(B, ctx::kMetThreads / 32), ctx::kMetThreads, 0, s>>>(
      partials, B, (int)tiles, 3.0 * (double)H * W, n_map, mse, ssim);
  CTX_RETURN_LAST();
}
