// Training ray batches drawn on the device: the batch samplers of upstream nerf-pytorch's train() loop
// (run_nerf.py: `no_batching` picks one image per step and N_rand of its pixels, with the centre crop for the first
// precrop_iters steps; otherwise the loop walks a shuffled stream over every ray of every image), evaluated inside the
// captured training step so that no host work runs between replays.
//
// Ray ids are global: view * H*W + y * W + x, the order of upstream's rays_rgb flatten over [N_train, H, W].
//
// Both modes sample without replacement through a keyed pseudo-random permutation pi of [0, n), evaluated pointwise
// (no state in memory):
//   b = the smallest even number >= 2 with 2^b >= n, h = b / 2, m = 2^h - 1
//   feistel(x):  L = x >> h, R = x & m;  for i = 0..3: (L, R) = (R, L ^ (F_i(R) & m));  return (L << h) | R
//   F_i(v) = word x of Philox4x32-10 (ctx::Philox) with key `key` and counter words
//            (c0, c1, c2, c3) = (v, tweak, i + 1, 4)       [ph(lo = (tweak << 32) | v, hi = (4 << 32) | (i + 1))]
//   pi(x) = feistel(x), applied again while the result is >= n (cycle-walking: 2^b < 4n, so fewer than 4 rounds of
//           the network are expected; x < n lies on a cycle of feistel that returns to [0, n), so the walk ends)
// Counter word c3 = 4 is Philox stream 4: streams 0-3 of the raygen key are the stratified jitter, the sample_pdf
// uniforms and the density noise of the coarse and the fine pass.
//
// mode 0 (upstream no_batching=True, the Blender recipe), t = counters[1] (the step count, 1 on the first step):
//   key = seed + counters[0] (the step's raygen key), tweak = rank
//   view = (x * n_views) >> 32, x = word x of Philox(key) at counter words (0, rank, 0, 4)
//   domain: if t < precrop_iters, rows [H/2 - dH, H/2 + dH) x cols [W/2 - dW, W/2 + dW) (upstream's centre crop,
//   dH = int(H//2 * precrop_frac)), else the whole image; ch x cw pixels, origin (y0, x0)
//   ray r: q = pi(r) over n = ch * cw, y = y0 + q / cw, x = x0 + q % cw
// mode 1 (upstream no_batching=False, the LLFF recipe): n = n_views * H * W
//   p = ((t - 1) * world + rank) * R + r, epoch e = p / n, key = seed (the same on every rank), tweak = e mod 2^32
//   ray r: id = pi(p mod n)
//   Every ray is drawn exactly once per epoch across the ranks, and every epoch is reshuffled.  Unlike upstream, a
//   batch that straddles the end of an epoch takes the tail of that epoch and the head of the next (upstream's
//   batch is short there, which a captured step of static shape cannot be).
// The target colours are gathered as target[r] = images[v, y, x, :].
#include "ctx_common.cuh"

namespace ctx {

struct DrawParams {
  const float* images;   // nullable [n_views, H, W, 3]
  int n_views, H, W;
  int64_t R;
  int mode;
  int precrop_iters, crop_dh, crop_dw;
  int rank, world;
  uint64_t seed;
  const unsigned long long* counters;
  int64_t* ray_idx;
  float* target;         // nullable [R, 3]
};

struct FeistelPerm {
  Philox ph;
  uint32_t tweak, half, mask, n;
  __device__ FeistelPerm(uint64_t key, uint32_t tweak_, uint32_t n_) : ph(key), tweak(tweak_), n(n_) {
    uint32_t b = 2;
    while (b < 32 && (1ull << b) < (uint64_t)n_) b += 2;
    half = b / 2;
    mask = (1u << half) - 1u;
  }
  __device__ __forceinline__ uint32_t feistel(uint32_t x) const {
    uint32_t L = x >> half, R = x & mask;
#pragma unroll
    for (uint32_t i = 0; i < 4; ++i) {
      const uint32_t f = ph(((uint64_t)tweak << 32) | R, (4ull << 32) | (uint64_t)(i + 1)).x & mask;
      const uint32_t nl = R;
      R = L ^ f;
      L = nl;
    }
    return (L << half) | R;
  }
  __device__ __forceinline__ uint32_t operator()(uint32_t x) const {
    uint32_t y = feistel(x);
    while (y >= n) y = feistel(y);
    return y;
  }
};

__global__ void __launch_bounds__(256) draw_rays_kernel(DrawParams p) {
  const uint64_t t = p.counters[1];
  const uint32_t hw = (uint32_t)p.H * (uint32_t)p.W;
  uint64_t key = p.seed;
  uint32_t view = 0, ch = p.H, cw = p.W, y0 = 0, x0 = 0;
  if (p.mode == 0) {
    key = p.seed + p.counters[0];
    const uint32_t x = Philox(key)((uint64_t)(uint32_t)p.rank << 32, 4ull << 32).x;
    view = (uint32_t)(((uint64_t)x * (uint64_t)p.n_views) >> 32);
    if ((int64_t)t < (int64_t)p.precrop_iters) {
      ch = 2 * p.crop_dh; cw = 2 * p.crop_dw;
      y0 = p.H / 2 - p.crop_dh; x0 = p.W / 2 - p.crop_dw;
    }
  }
  const uint32_t n = p.mode == 0 ? ch * cw : hw * (uint32_t)p.n_views;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < p.R; r += (int64_t)gridDim.x * blockDim.x) {
    uint32_t id;
    if (p.mode == 0) {
      const uint32_t q = FeistelPerm(key, (uint32_t)p.rank, n)((uint32_t)r);
      const uint32_t qy = q / cw;
      id = view * hw + (y0 + qy) * (uint32_t)p.W + x0 + (q - qy * cw);
    } else {
      const uint64_t pos = ((t - 1ull) * (uint64_t)p.world + (uint64_t)p.rank) * (uint64_t)p.R + (uint64_t)r;
      const uint64_t e = pos / n;
      id = FeistelPerm(key, (uint32_t)e, n)((uint32_t)(pos - e * n));
    }
    p.ray_idx[r] = (int64_t)id;
    if (p.target) {
      const float* src = p.images + (int64_t)id * 3;
      float* dst = p.target + r * 3;
      dst[0] = __ldg(src); dst[1] = __ldg(src + 1); dst[2] = __ldg(src + 2);
    }
  }
}

}  // namespace ctx

extern "C" int ctx_draw_rays(const float* images, int n_views, int H, int W, int64_t R, int mode, int precrop_iters,
                             int crop_dh, int crop_dw, int rank, int world, uint64_t seed, const void* counters,
                             int64_t* ray_idx, float* target, void* stream) {
  if (!ray_idx || !counters || R < 0 || n_views < 1 || H < 1 || W < 1) return CTX_ERR_BAD_ARG;
  if (target && !images) return CTX_ERR_BAD_ARG;
  if (world < 1 || rank < 0 || rank >= world) return CTX_ERR_BAD_ARG;
  if ((int64_t)n_views * H * W >= ((int64_t)1 << 31)) return CTX_ERR_BAD_ARG;   // ids are split in 32 bits
  if (mode == 0) {
    if (R > (int64_t)H * W) return CTX_ERR_BAD_ARG;                              // distinct pixels of one image
    if (precrop_iters < 0) return CTX_ERR_BAD_ARG;
    if (precrop_iters > 0) {
      if (crop_dh < 1 || crop_dw < 1 || crop_dh > H / 2 || crop_dw > W / 2) return CTX_ERR_BAD_ARG;   // empty crop
      if (R > (int64_t)4 * crop_dh * crop_dw) return CTX_ERR_BAD_ARG;
    }
  } else if (mode == 1) {
    if (precrop_iters != 0) return CTX_ERR_BAD_ARG;          // upstream crops only when it batches from one image
  } else {
    return CTX_ERR_BAD_ARG;
  }
  if (R == 0) return 0;
  ctx::DrawParams p;
  p.images = images; p.n_views = n_views; p.H = H; p.W = W; p.R = R; p.mode = mode;
  p.precrop_iters = precrop_iters; p.crop_dh = crop_dh; p.crop_dw = crop_dw; p.rank = rank; p.world = world;
  p.seed = seed; p.counters = (const unsigned long long*)counters; p.ray_idx = ray_idx; p.target = target;
  int64_t blocks = ctx::ceil_div(R, 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  ctx::draw_rays_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  CTX_RETURN_LAST();
}
