// Fused Adam over the flat parameter / gradient buckets of the two NeRF MLPs
// (the reference trains with torch.optim.Adam, src/training/trainer.py:603),
// and the fused photometric loss: img2mse(rgb, t) + img2mse(rgb0, t)
// (src/run_nerf_helpers.py:9) with its gradient in one pass.
#include "ctx_common.cuh"

namespace ctx {

// torch.optim.Adam semantics (no amsgrad, optional L2 weight decay), bias-corrected.
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, float lr, float b1, float b2, float eps,
                            float bc1, float bc2_sqrt, float wd, float grad_scale) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i] * grad_scale;
    if (wd != 0.f) gi += wd * p[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

// Device-side step state of the captured training step: ctr[0] = Philox seed offset (raygen / resample add it to their
// seed), ctr[1] = Adam step count.  The tick runs first in every step: it advances both and zeroes the loss scalar
// the fused compositing kernels accumulate into, so a CUDA-graph replay needs no host-side argument to change.
__global__ void step_tick_kernel(unsigned long long* __restrict__ ctr, float* __restrict__ loss) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    ctr[0] += 2ull;
    ctr[1] += 1ull;
    if (loss) loss[0] = 0.f;
  }
}

// Adam with the step count read from the device counter (bias corrections formed per thread: two powf).
// DECAY: update t uses lr * 0.1^(max(t-2, 0) / decay_steps), the rate upstream's loop has set when its t-th
// optimizer.step() runs (it sets lrate * 0.1^(global_step / decay_steps) after each step, then counts global_step
// up from 0).
template <bool DECAY>
__global__ void adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                float* __restrict__ v, int64_t n, float lr, float b1, float b2, float eps,
                                const unsigned long long* __restrict__ ctr, float wd, float grad_scale,
                                float decay_steps) {
  const float step = (float)ctr[1];
  if constexpr (DECAY) lr *= powf(0.1f, fmaxf(step - 2.f, 0.f) / decay_steps);
  const float bc1 = 1.f - powf(b1, step);
  const float bc2_sqrt = sqrtf(1.f - powf(b2, step));
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i] * grad_scale;
    if (wd != 0.f) gi += wd * p[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

// loss = mean((a-t)^2) [+ mean((b-t)^2)]; g_a = 2(a-t)/n * scale, g_b likewise.  One CTA.
__global__ void mse_pair_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                const float* __restrict__ t, int64_t n, float scale, float* __restrict__ loss,
                                float* __restrict__ g_a, float* __restrict__ g_b) {
  __shared__ float red[32];
  float acc = 0.f;
  const float inv = 1.0f / (float)n;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const float ti = t[i];
    const float da = a[i] - ti;
    acc += da * da;
    if (g_a) g_a[i] = 2.f * da * inv * scale;
    if (b) {
      const float db = b[i] - ti;
      acc += db * db;
      if (g_b) g_b[i] = 2.f * db * inv * scale;
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) loss[0] = v * inv;
  }
}

// texture activation of the reference: (tanh(x)+1)/2 (src/models/textured_mesh.py:299), fused with the
// [P,C] -> [C,P] (NCHW) transpose of `.reshape(1,res,res,3).permute(0,3,1,2)`.
__global__ void tanh01_fwd_kernel(const float* __restrict__ raw, float* __restrict__ out, int64_t P, int C) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (int64_t)gridDim.x * blockDim.x)
    for (int c = 0; c < C; ++c) out[(int64_t)c * P + i] = (tanhf(raw[i * C + c]) + 1.0f) * 0.5f;
}
// g_raw[p,c] = g_raw_in[p,c] (optional) + g_tex[c,p] * 0.5 * (1 - tanh(raw)^2)
__global__ void tanh01_bwd_kernel(const float* __restrict__ raw, const float* __restrict__ g_tex,
                                  const float* __restrict__ g_raw_in, float* __restrict__ g_raw, int64_t P, int C) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (int64_t)gridDim.x * blockDim.x)
    for (int c = 0; c < C; ++c) {
      const float t = tanhf(raw[i * C + c]);
      float g = g_tex ? g_tex[(int64_t)c * P + i] * 0.5f * (1.0f - t * t) : 0.f;
      if (g_raw_in) g += g_raw_in[i * C + c];
      g_raw[i * C + c] = g;
    }
}

}  // namespace ctx

extern "C" int ctx_tanh01_fwd(const float* raw, float* out, int64_t P, int C, void* stream) {
  if (P < 0 || C < 1 || !raw || !out) return CTX_ERR_BAD_ARG;
  if (P == 0) return 0;
  int64_t blocks = ctx::ceil_div(P, 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  ctx::tanh01_fwd_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(raw, out, P, C);
  CTX_RETURN_LAST();
}

extern "C" int ctx_tanh01_bwd(const float* raw, const float* g_tex, const float* g_raw_in, float* g_raw, int64_t P,
                              int C, void* stream) {
  if (P < 0 || C < 1 || !raw || !g_raw) return CTX_ERR_BAD_ARG;
  if (P == 0) return 0;
  int64_t blocks = ctx::ceil_div(P, 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  ctx::tanh01_bwd_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(raw, g_tex, g_raw_in, g_raw, P, C);
  CTX_RETURN_LAST();
}

extern "C" int ctx_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                             float lr, float beta1, float beta2, float eps, int step, float weight_decay,
                             float grad_scale, void* stream) {
  if (n < 0 || step < 1 || !params || !grads || !exp_avg || !exp_avg_sq) return CTX_ERR_BAD_ARG;
  if (n == 0) return 0;
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2 = sqrtf(1.f - powf(beta2, (float)step));
  int64_t blocks = ctx::ceil_div(n, 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  ctx::adam_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(params, grads, exp_avg, exp_avg_sq, n, lr, beta1,
                                                                  beta2, eps, bc1, bc2, weight_decay, grad_scale);
  CTX_RETURN_LAST();
}

extern "C" int ctx_step_tick(void* counters, float* loss, void* stream) {
  if (!counters) return CTX_ERR_BAD_ARG;
  ctx::step_tick_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((unsigned long long*)counters, loss);
  CTX_RETURN_LAST();
}

extern "C" int ctx_adam_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                                 float lr, float beta1, float beta2, float eps, const void* counters,
                                 float weight_decay, float grad_scale, void* stream) {
  if (n < 0 || !params || !grads || !exp_avg || !exp_avg_sq || !counters) return CTX_ERR_BAD_ARG;
  if (n == 0) return 0;
  int64_t blocks = ctx::ceil_div(n, 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  ctx::adam_dev_kernel<false><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
      params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, (const unsigned long long*)counters, weight_decay,
      grad_scale, 0.f);
  CTX_RETURN_LAST();
}

extern "C" int ctx_adam_step_dev_decay(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                                       int64_t n, float lr, float beta1, float beta2, float eps, const void* counters,
                                       float weight_decay, float grad_scale, float decay_steps, void* stream) {
  if (n < 0 || !params || !grads || !exp_avg || !exp_avg_sq || !counters || !(decay_steps > 0.f))
    return CTX_ERR_BAD_ARG;
  if (n == 0) return 0;
  int64_t blocks = ctx::ceil_div(n, 256);
  if (blocks > ctx::num_sms() * 8) blocks = ctx::num_sms() * 8;
  ctx::adam_dev_kernel<true><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
      params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, (const unsigned long long*)counters, weight_decay,
      grad_scale, decay_steps);
  CTX_RETURN_LAST();
}

extern "C" int ctx_mse_fwd_bwd(const float* a, const float* b, const float* target, int64_t n, float scale,
                               float* loss, float* g_a, float* g_b, void* stream) {
  if (n < 1 || !a || !target || !loss) return CTX_ERR_BAD_ARG;
  ctx::mse_pair_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(a, b, target, n, scale, loss, g_a, g_b);
  CTX_RETURN_LAST();
}
