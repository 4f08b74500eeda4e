// Ray generation fused with stratified depth sampling, the NDC warp, and the
// stand-alone stratified sampler used by render_rays.
//
// get_rays:  /root/reference/src/run_nerf_helpers.py:139-148
// ndc_rays:  /root/reference/src/run_nerf_helpers.py:161-178
// stratified depths: upstream render_rays (SURVEY.md 8c-S2)
// Built with -fmad=false: every mul/add is a separate fp32 op as in eager
// PyTorch, so rays_d / z_vals (given the same uniforms) are bit-identical.
// HBM-bound, write-only: 24 + 12[viewdirs] + 4*S bytes per ray.
#include "ctx_common.cuh"

namespace ctx {

constexpr int kRayWarps = 8;

struct RaygenParams {
  int H, W;
  float fx, fy, cx, cy;
  const float* c2w;        // device, row-major [3,4] (or the top of a [4,4])
  int c2w_ld;              // 4
  const int64_t* ray_idx;  // optional gather list of flat pixel ids (y*W + x)
  int64_t n_rays;
  // optional ndc warp
  int use_ndc;
  float ndc_focal, ndc_near;
  // depth sampling
  int n_samples;  // 0: no z output
  float near, far;
  int lindisp;
  int perturb;            // 0: none, 1: jitter
  const float* jitter;    // optional uniforms [n_rays, n_samples]; else Philox(seed)
  uint64_t seed;
  const uint64_t* seed_dev;   // optional device counter ADDED to seed (a captured CUDA graph replays with fresh numbers)
  // optional bounding sphere: per-ray near/far = sphere entry/exit (cfg 4)
  int use_sphere;
  float sph_cx, sph_cy, sph_cz, sph_r;
  // outputs
  float* rays_o;    // [n,3]
  float* rays_d;    // [n,3]
  float* viewdirs;  // optional [n,3]
  float* z_vals;    // optional [n, n_samples]
  float* near_far;  // optional [n,2]
  int rays_per_iter;  // rays a warp builds per iteration (power of two, >= rows per pass, <= 32; set by the launcher)
  // pose stack (raygen_kernel<true>): c2w holds n_views poses pose_stride floats apart, ray_idx global ray ids
  int n_views, pose_stride;
};

// z(s) before jitter
__device__ __forceinline__ float base_depth(float near, float far, int S, int s, int lindisp) {
  const float t = linspace_at(0.0f, 1.0f, S, s);
  if (lindisp) return 1.0f / ((1.0f / near) * (1.0f - t) + (1.0f / far) * t);
  return near * (1.0f - t) + far * t;
}

__device__ __forceinline__ float stratified_depth(float near, float far, int S, int s, int lindisp,
                                                  bool jit, float u) {
  const float zc = base_depth(near, far, S, s, lindisp);
  if (!jit) return zc;
  const float lower = (s == 0) ? zc : 0.5f * (zc + base_depth(near, far, S, s - 1, lindisp));
  const float upper = (s == S - 1) ? zc : 0.5f * (base_depth(near, far, S, s + 1, lindisp) + zc);
  return lower + (upper - lower) * u;
}

// One warp writes the S depths of a ray: each lane produces QUADS of consecutive samples (one Philox call =
// 4 uniforms, one 16-byte store), the linspace step and the reciprocals are hoisted.  Values are bit-identical
// to stratified_depth() sample by sample.
// `lane` / `nl`: position in and size of the lane group that shares this ray (8, 16 or 32 lanes).
__device__ __forceinline__ void write_z_row(float* __restrict__ zrow, float near, float far, int S, int lindisp,
                                            int perturb, const float* __restrict__ jrow, uint64_t seed,
                                            uint64_t ray, int lane, int nl = 32, float step_in = -1.0f) {
  if ((S & 3) != 0 || S < 4) {   // ragged sample counts: element-wise path
    for (int s = lane; s < S; s += nl) {
      float u = 0.f;
      if (perturb) u = jrow ? jrow[s] : philox_uniform(seed, 0, ray, (uint32_t)s);
      zrow[s] = stratified_depth(near, far, S, s, lindisp, perturb != 0, u);
    }
    return;
  }
  const float step = step_in >= 0.0f ? step_in : __fdiv_rn(1.0f, (float)(S - 1));   // (callers in a loop pass it in)
  float inear = 0.f, ifar = 0.f;
  if (lindisp) { inear = 1.0f / near; ifar = 1.0f / far; }
  const int half = S / 2;
  const float fS1 = (float)(S - 1), fhalf = (float)half;
  // base depth of sample index `fi` (an integer held in fp32: one int->float conversion per quad instead of one or two
  // per depth -- the conversions run on the quarter-rate pipe and this kernel is issue-bound); same values as
  // linspace_at: lower half step*i, upper half 1 - step*(S-1-i), one rounding each
  auto base = [&](float fi) -> float {
    const float t = (fi < fhalf) ? fmaf(step, fi, 0.0f) : fmaf(-step, fS1 - fi, 1.0f);
    if (lindisp) return 1.0f / (inear * (1.0f - t) + ifar * t);
    return near * (1.0f - t) + far * t;
  };
  for (int q = lane; q < (S >> 2); q += nl) {
    const int s0 = q << 2;
    float4 out;
    if (!perturb) {
      const float f0 = (float)s0;
      out = make_float4(base(f0), base(f0 + 1.0f), base(f0 + 2.0f), base(f0 + 3.0f));
    } else {
      float zb[6];
      const float fm1 = (float)(s0 - 1);
#pragma unroll
      for (int i = 0; i < 6; ++i) zb[i] = base(fminf(fmaxf(fm1 + (float)i, 0.0f), fS1));   // neighbours, clamped to the row
      float u[4];
      if (jrow) {
        const float4 j4 = *reinterpret_cast<const float4*>(jrow + s0);
        u[0] = j4.x; u[1] = j4.y; u[2] = j4.z; u[3] = j4.w;
      } else {
        Philox ph(seed);
        const uint4 rr = ph(ray, (uint64_t)q);   // stream 0: same numbers as philox_uniform(seed, 0, ray, s)
        u[0] = u01(rr.x); u[1] = u01(rr.y); u[2] = u01(rr.z); u[3] = u01(rr.w);
      }
      float o[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int s = s0 + i;
        const float zc = zb[i + 1];
        const float lower = (s == 0) ? zc : 0.5f * (zc + zb[i]);
        const float upper = (s == S - 1) ? zc : 0.5f * (zb[i + 2] + zc);
        o[i] = lower + (upper - lower) * u[i];
      }
      out = make_float4(o[0], o[1], o[2], o[3]);
    }
    *reinterpret_cast<float4*>(zrow + s0) = out;
  }
}

__device__ __forceinline__ void ndc_warp(int H, int W, float focal, float near, float& ox,
                                         float& oy, float& oz, float& dx, float& dy, float& dz) {
  const float t = -(near + oz) / dz;
  ox = ox + t * dx; oy = oy + t * dy; oz = oz + t * dz;
  // -1./(W/(2.*focal)) is evaluated in Python doubles, then applied as an fp32 scalar
  const float sx = (float)(-1.0 / ((double)W / (2.0 * (double)focal)));
  const float sy = (float)(-1.0 / ((double)H / (2.0 * (double)focal)));
  const float two_near = (float)(2.0 * (double)near);
  const float n0 = sx * ox / oz, n1 = sy * oy / oz, n2 = 1.0f + two_near / oz;
  const float e0 = sx * (dx / dz - ox / oz), e1 = sy * (dy / dz - oy / oz);
  const float e2 = (float)(-2.0 * (double)near) / oz;
  ox = n0; oy = n1; oz = n2; dx = e0; dy = e1; dz = e2;
}

// rotation and origin of a camera-to-world pose, row-major with leading dimension ld
__device__ __forceinline__ void load_pose(const float* c2w, int ld, float (&rot)[3][3], float (&org)[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int j = 0; j < 3; ++j) rot[k][j] = __ldg(c2w + k * ld + j);
    org[k] = __ldg(c2w + k * ld + 3);
  }
}

// kPoseStack = false: one camera (p.c2w), ray ids are pixel ids y*W + x.  kPoseStack = true: ray ids are global ids
// view*H*W + y*W + x (upstream's rays_rgb order over [N_train, H, W]) and each lane loads the pose of its own view;
// everything after the pose load is the one-camera code, so a ray of view v is the ray the one-camera kernel makes
// with pose v on the same batch row.
template <bool kPoseStack>
__global__ void __launch_bounds__(kRayWarps * 32) raygen_kernel(RaygenParams p) {
  // A warp takes 32 rays per iteration.  Phase 1: lane l builds ray r0 + l ONCE (pixel split, the two intrinsics
  // divisions, rotation, norm, view direction, sphere interval) and stores its origin / direction / view direction.
  // Phase 2: the depth rows, a group of `nl` lanes (8/16/32, chosen so that one pass of quads covers the S depths)
  // per ray, near / far handed over by shuffle.  (Before: every lane of a group redid the whole per-ray setup --
  // a third of the kernel's instructions in the ncu source page, and the kernel is issue-bound.)
  const int nl = p.n_samples > 64 ? 32 : (p.n_samples > 32 ? 16 : 8);
  const int gpw = 32 / nl;                                   // depth rows written per pass
  const int l32 = threadIdx.x & 31;
  const int lane = l32 & (nl - 1), sub = l32 / nl;
  const int64_t warp0 = (int64_t)blockIdx.x * kRayWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kRayWarps;
  // camera (uniform loads)
  float rot[3][3], org[3];
  if constexpr (!kPoseStack) load_pose(p.c2w, p.c2w_ld, rot, org);
  const uint64_t seed = p.seed + (p.seed_dev ? *p.seed_dev : 0ull);
  const float zstep = p.n_samples > 1 ? __fdiv_rn(1.0f, (float)(p.n_samples - 1)) : 0.0f;
  const int rpi = p.rays_per_iter;                           // 32 for large launches; fewer so that a small batch
  for (int64_t r0 = warp0 * rpi; r0 < p.n_rays; r0 += nwarps * rpi) {   // (a 4096-ray training step) still covers the SMs
    const int64_t r = r0 + l32;
    float near = p.near, far = p.far;
    if (l32 < rpi && r < p.n_rays) {
      const int64_t pix = p.ray_idx ? p.ray_idx[r] : r;
      uint32_t pix32 = (uint32_t)pix;                             // (n_views*)H*W < 2^31 is checked by the launcher
      if constexpr (kPoseStack) {
        const uint32_t hw = (uint32_t)p.H * (uint32_t)p.W;
        const uint32_t view = min(pix32 / hw, (uint32_t)(p.n_views - 1));   // (clamped: an id past the stack reads no
        pix32 -= view * hw;                                                   //  memory beyond it)
        load_pose(p.c2w + (int64_t)view * p.pose_stride, p.c2w_ld, rot, org);
      }
      const int py = (int)(pix32 / (uint32_t)p.W), px = (int)(pix32 - (uint32_t)py * (uint32_t)p.W);
      const float a = ((float)px - p.cx) / p.fx;
      const float b = -((float)py - p.cy) / p.fy;
      const float c = -1.0f;
      float dx = (a * rot[0][0] + b * rot[0][1]) + c * rot[0][2];
      float dy = (a * rot[1][0] + b * rot[1][1]) + c * rot[1][2];
      float dz = (a * rot[2][0] + b * rot[2][1]) + c * rot[2][2];
      float ox = org[0], oy = org[1], oz = org[2];
      // viewdirs are taken before the NDC warp (upstream render())
      const float inv = sqrtf(dx * dx + dy * dy + dz * dz);
      const float vx = dx / inv, vy = dy / inv, vz = dz / inv;
      if (p.use_ndc) ndc_warp(p.H, p.W, p.ndc_focal, p.ndc_near, ox, oy, oz, dx, dy, dz);
      if (p.use_sphere) {
        // |o + t d - c|^2 = r^2 ; rays that miss get near = far = |o - c| projected distance
        const float lx = ox - p.sph_cx, ly = oy - p.sph_cy, lz = oz - p.sph_cz;
        const float A = dx * dx + dy * dy + dz * dz;
        const float Bq = lx * dx + ly * dy + lz * dz;
        const float Cq = lx * lx + ly * ly + lz * lz - p.sph_r * p.sph_r;
        const float disc = Bq * Bq - A * Cq;
        if (disc > 0.f) {
          const float sq = sqrtf(disc);
          near = fmaxf((-Bq - sq) / A, 0.f);
          far = fmaxf((-Bq + sq) / A, near);
        } else {
          near = far = fmaxf(-Bq / A, 0.f);
        }
      }
      // three consecutive floats per lane: the warp's 32 rays fill one contiguous 384-byte span per array
      float* po = p.rays_o + r * 3;
      po[0] = ox; po[1] = oy; po[2] = oz;
      float* pd = p.rays_d + r * 3;
      pd[0] = dx; pd[1] = dy; pd[2] = dz;
      if (p.viewdirs) {
        float* pv = p.viewdirs + r * 3;
        pv[0] = vx; pv[1] = vy; pv[2] = vz;
      }
      if (p.near_far) { p.near_far[r * 2] = near; p.near_far[r * 2 + 1] = far; }
    }
    if (p.z_vals) {
      const int64_t left = p.n_rays - r0;
      const int cnt = left < rpi ? (int)left : rpi;             // warp-uniform
      for (int j = 0; j < cnt; j += gpw) {
        const int owner = j + sub;                               // lane that built this group's ray (< 32)
        float nr = p.near, fr = p.far;
        if (p.use_sphere) {
          nr = __shfl_sync(CTX_FULL_MASK, near, owner);
          fr = __shfl_sync(CTX_FULL_MASK, far, owner);
        }
        const int64_t rr = r0 + owner;
        if (rr < p.n_rays)
          write_z_row(p.z_vals + rr * p.n_samples, nr, fr, p.n_samples, p.lindisp, p.perturb,
                      p.jitter ? p.jitter + rr * p.n_samples : nullptr, seed, (uint64_t)rr, lane, nl, zstep);
      }
    }
  }
}

// z_vals from per-ray near/far (columns 6,7 of upstream's ray_batch)
__global__ void __launch_bounds__(kRayWarps * 32)
stratified_kernel(const float* __restrict__ near, int64_t near_stride, const float* __restrict__ far,
                  int64_t far_stride, int64_t R, int S, int lindisp, int perturb,
                  const float* __restrict__ jitter, uint64_t seed, float* __restrict__ z_vals) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kRayWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kRayWarps;
  for (int64_t r = warp0; r < R; r += nwarps) {
    const float n = near[r * near_stride], f = far[r * far_stride];
    write_z_row(z_vals + r * S, n, f, S, lindisp, perturb, jitter ? jitter + r * S : nullptr, seed, (uint64_t)r, lane);
  }
}

__global__ void ndc_fwd_kernel(int H, int W, float focal, float near, const float* __restrict__ o_in,
                               const float* __restrict__ d_in, int64_t n, float* __restrict__ o_out,
                               float* __restrict__ d_out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    float ox = o_in[i * 3], oy = o_in[i * 3 + 1], oz = o_in[i * 3 + 2];
    float dx = d_in[i * 3], dy = d_in[i * 3 + 1], dz = d_in[i * 3 + 2];
    ndc_warp(H, W, focal, near, ox, oy, oz, dx, dy, dz);
    o_out[i * 3] = ox; o_out[i * 3 + 1] = oy; o_out[i * 3 + 2] = oz;
    d_out[i * 3] = dx; d_out[i * 3 + 1] = dy; d_out[i * 3 + 2] = dz;
  }
}

// Backward of the NDC warp w.r.t. rays_o / rays_d (hand-derived; the warp is a
// per-ray rational map).  Inputs are the ORIGINAL rays.
__global__ void ndc_bwd_kernel(int H, int W, float focal, float near, const float* __restrict__ o_in,
                               const float* __restrict__ d_in, const float* __restrict__ g_o,
                               const float* __restrict__ g_d, int64_t n, float* __restrict__ go_in,
                               float* __restrict__ gd_in) {
  const float sx = (float)(-1.0 / ((double)W / (2.0 * (double)focal)));
  const float sy = (float)(-1.0 / ((double)H / (2.0 * (double)focal)));
  const float tn = 2.0f * near;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float ox = o_in[i * 3], oy = o_in[i * 3 + 1], oz = o_in[i * 3 + 2];
    const float dx = d_in[i * 3], dy = d_in[i * 3 + 1], dz = d_in[i * 3 + 2];
    const float t = -(near + oz) / dz;
    const float px = ox + t * dx, py = oy + t * dy, pz = oz + t * dz;  // shifted origin
    const float a0 = g_o ? g_o[i * 3] : 0.f, a1 = g_o ? g_o[i * 3 + 1] : 0.f, a2 = g_o ? g_o[i * 3 + 2] : 0.f;
    const float b0 = g_d ? g_d[i * 3] : 0.f, b1 = g_d ? g_d[i * 3 + 1] : 0.f, b2 = g_d ? g_d[i * 3 + 2] : 0.f;
    // outputs: n0 = sx px/pz, n1 = sy py/pz, n2 = 1 + tn/pz
    //          e0 = sx (dx/dz - px/pz), e1 = sy (dy/dz - py/pz), e2 = -tn/pz
    const float ipz = 1.0f / pz, idz = 1.0f / dz;
    float gpx = sx * ipz * (a0 - b0);
    float gpy = sy * ipz * (a1 - b1);
    float gpz = -sx * px * ipz * ipz * (a0 - b0) - sy * py * ipz * ipz * (a1 - b1) +
                tn * ipz * ipz * (b2 - a2);
    float gdx = sx * idz * b0, gdy = sy * idz * b1;
    float gdz = -sx * dx * idz * idz * b0 - sy * dy * idz * idz * b1;
    // p = o + t d, t = -(near+oz)/dz
    const float gt = gpx * dx + gpy * dy + gpz * dz;
    gdx += gpx * t; gdy += gpy * t; gdz += gpz * t;
    float gox = gpx, goy = gpy, goz = gpz;
    goz += gt * (-idz);
    gdz += gt * ((near + oz) * idz * idz);
    go_in[i * 3] = gox; go_in[i * 3 + 1] = goy; go_in[i * 3 + 2] = goz;
    gd_in[i * 3] = gdx; gd_in[i * 3 + 1] = gdy; gd_in[i * 3 + 2] = gdz;
  }
}

static inline int warp_grid(int64_t rows, int warps_per_cta) {
  int64_t blocks = ceil_div(rows, warps_per_cta);
  const int64_t cap = (int64_t)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace ctx

namespace ctx {

// the one-camera and the pose-stack launch: same checks, same geometry
static int launch_raygen(bool pose_stack, int H, int W, float fx, float fy, float cx, float cy, const float* c2w,
                         int c2w_ld, const int64_t* ray_idx, int64_t n_rays, int use_ndc, float ndc_focal,
                         float ndc_near, int n_samples, float near, float far, int lindisp, int perturb,
                         const float* jitter, uint64_t seed, const uint64_t* seed_dev, int use_sphere,
                         const float* sphere, float* rays_o, float* rays_d, float* viewdirs, float* z_vals,
                         float* near_far, int n_views, int pose_stride, cudaStream_t stream) {
  if (H < 1 || W < 1 || n_rays < 0 || !c2w || c2w_ld < 4 || n_samples < 0) return CTX_ERR_BAD_ARG;
  if (n_views < 1 || pose_stride < 3 * c2w_ld) return CTX_ERR_BAD_ARG;
  // ray ids are split with 32-bit arithmetic (view, then row and column)
  if ((int64_t)n_views * H * W >= ((int64_t)1 << 31)) return CTX_ERR_BAD_ARG;
  if (pose_stack && !ray_idx && n_rays > (int64_t)n_views * H * W) return CTX_ERR_BAD_ARG;
  if (n_rays == 0) return 0;
  if (!rays_o || !rays_d) return CTX_ERR_BAD_ARG;
  if (use_sphere && !sphere) return CTX_ERR_BAD_ARG;
  RaygenParams p;
  p.H = H; p.W = W; p.fx = fx; p.fy = fy; p.cx = cx; p.cy = cy; p.c2w = c2w; p.c2w_ld = c2w_ld;
  p.ray_idx = ray_idx; p.n_rays = n_rays; p.use_ndc = use_ndc; p.ndc_focal = ndc_focal;
  p.ndc_near = ndc_near; p.n_samples = n_samples; p.near = near; p.far = far; p.lindisp = lindisp;
  p.perturb = perturb; p.jitter = jitter; p.seed = seed; p.seed_dev = seed_dev; p.use_sphere = use_sphere;
  p.sph_cx = use_sphere ? sphere[0] : 0.f; p.sph_cy = use_sphere ? sphere[1] : 0.f;
  p.sph_cz = use_sphere ? sphere[2] : 0.f; p.sph_r = use_sphere ? sphere[3] : 0.f;
  p.rays_o = rays_o; p.rays_d = rays_d; p.viewdirs = viewdirs;
  p.z_vals = n_samples > 0 ? z_vals : nullptr; p.near_far = near_far;
  p.n_views = n_views; p.pose_stride = pose_stride;
  {
    const int nl = n_samples > 64 ? 32 : (n_samples > 32 ? 16 : 8);
    int rpi = 32;                                       // halve while the launch would leave SMs without a warp
    while (rpi > 32 / nl && n_rays < (int64_t)rpi * kRayWarps * num_sms() * 2) rpi >>= 1;
    p.rays_per_iter = rpi;
  }
  const int grid = warp_grid(ceil_div(n_rays, p.rays_per_iter), kRayWarps);
  if (pose_stack)
    raygen_kernel<true><<<grid, kRayWarps * 32, 0, stream>>>(p);
  else
    raygen_kernel<false><<<grid, kRayWarps * 32, 0, stream>>>(p);
  CTX_RETURN_LAST();
}

}  // namespace ctx

extern "C" int ctx_raygen_fwd(int H, int W, float fx, float fy, float cx, float cy, const float* c2w,
                              int c2w_ld, const int64_t* ray_idx, int64_t n_rays, int use_ndc,
                              float ndc_focal, float ndc_near, int n_samples, float near, float far,
                              int lindisp, int perturb, const float* jitter, uint64_t seed,
                              const uint64_t* seed_dev, int use_sphere, const float* sphere /*host: cx,cy,cz,r*/,
                              float* rays_o, float* rays_d, float* viewdirs, float* z_vals,
                              float* near_far, void* stream) {
  return ctx::launch_raygen(false, H, W, fx, fy, cx, cy, c2w, c2w_ld, ray_idx, n_rays, use_ndc, ndc_focal, ndc_near,
                            n_samples, near, far, lindisp, perturb, jitter, seed, seed_dev, use_sphere, sphere, rays_o,
                            rays_d, viewdirs, z_vals, near_far, 1, 3 * c2w_ld, (cudaStream_t)stream);
}

extern "C" int ctx_raygen_views(int H, int W, float fx, float fy, float cx, float cy, const float* poses,
                                int c2w_ld, const int64_t* ray_idx, int64_t n_rays, int use_ndc,
                                float ndc_focal, float ndc_near, int n_samples, float near, float far,
                                int lindisp, int perturb, const float* jitter, uint64_t seed,
                                const uint64_t* seed_dev, int use_sphere, const float* sphere /*host: cx,cy,cz,r*/,
                                float* rays_o, float* rays_d, float* viewdirs, float* z_vals,
                                float* near_far, int n_views, int pose_stride, void* stream) {
  return ctx::launch_raygen(true, H, W, fx, fy, cx, cy, poses, c2w_ld, ray_idx, n_rays, use_ndc, ndc_focal, ndc_near,
                            n_samples, near, far, lindisp, perturb, jitter, seed, seed_dev, use_sphere, sphere, rays_o,
                            rays_d, viewdirs, z_vals, near_far, n_views, pose_stride, (cudaStream_t)stream);
}

extern "C" int ctx_stratified_fwd(const float* near, int64_t near_stride, const float* far,
                                  int64_t far_stride, int64_t R, int S, int lindisp, int perturb,
                                  const float* jitter, uint64_t seed, float* z_vals, void* stream) {
  if (R < 0 || S < 1 || !near || !far || !z_vals) return CTX_ERR_BAD_ARG;
  if (R == 0) return 0;
  ctx::stratified_kernel<<<ctx::warp_grid(R, ctx::kRayWarps), ctx::kRayWarps * 32, 0,
                           (cudaStream_t)stream>>>(near, near_stride, far, far_stride, R, S, lindisp,
                                                   perturb, jitter, seed, z_vals);
  CTX_RETURN_LAST();
}

extern "C" int ctx_ndc_fwd(int H, int W, float focal, float near, const float* rays_o,
                           const float* rays_d, int64_t n, float* o_out, float* d_out, void* stream) {
  if (n < 0 || !rays_o || !rays_d || !o_out || !d_out) return CTX_ERR_BAD_ARG;
  if (n == 0) return 0;
  int64_t blocks = ctx::ceil_div(n, 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  ctx::ndc_fwd_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(H, W, focal, near, rays_o, rays_d,
                                                                    n, o_out, d_out);
  CTX_RETURN_LAST();
}

extern "C" int ctx_ndc_bwd(int H, int W, float focal, float near, const float* rays_o,
                           const float* rays_d, const float* g_o, const float* g_d, int64_t n,
                           float* g_rays_o, float* g_rays_d, void* stream) {
  if (n < 0 || !rays_o || !rays_d || !g_rays_o || !g_rays_d) return CTX_ERR_BAD_ARG;
  if (n == 0) return 0;
  int64_t blocks = ctx::ceil_div(n, 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  ctx::ndc_bwd_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(H, W, focal, near, rays_o, rays_d,
                                                                    g_o, g_d, n, g_rays_o, g_rays_d);
  CTX_RETURN_LAST();
}
