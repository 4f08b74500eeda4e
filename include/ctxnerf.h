/* ctxnerf.h -- C-ABI of libctxnerf.so: the B200 (sm_100a) NeRF ray-march path.
 *
 * The reference (zaiisao/ConTEXTure-NeRF) has no FFI: its boundary for this
 * path is the Python surface of src/run_nerf_helpers.py.  Each entry point
 * below is what a ctypes binding placed in that module calls instead of the
 * eager-PyTorch body it replaces (file:line given per function; INTEGRATION.md
 * shows the binding).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless marked "host"; tensors are
 *    contiguous row-major fp32 unless a stride argument is given;
 *  - the library never allocates, frees or synchronises; work is enqueued on
 *    `stream` (a cudaStream_t passed as void*), launchers are re-entrant;
 *  - return 0 on success, a positive cudaError_t on a CUDA failure, a negative
 *    CTX_ERR_* on a bad argument.  Nothing throws across the ABI;
 *  - "nullable" arguments may be NULL.
 */
#ifndef CTXNERF_H
#define CTXNERF_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTXNERF_ABI_VERSION 3
#define CTX_ERR_BAD_ARG (-1)
#define CTX_ERR_UNSUPPORTED (-2)
#define CTX_ERR_NO_NCCL (-3)

int ctx_abi_version(void);
/* static string for a code returned by any ctx_* call */
const char* ctx_error_string(int code);

/* ---- positional encoding: Embedder.embed, src/run_nerf_helpers.py:44-45 ----
 * x [n,d] -> out [n, d*(include_input + 2L)], channel order of :24-39.        */
int ctx_posenc_fwd(const float* x, float* out, int64_t n, int d, int L, int include_input,
                   int log_sampling, void* stream);
int ctx_posenc_bwd(const float* x, const float* g_out, float* g_x, int64_t n, int d, int L,
                   int include_input, int log_sampling, void* stream);

/* ---- ray generation fused with stratified sampling --------------------------
 * get_rays, src/run_nerf_helpers.py:139-148 (+ optional ndc_rays :161-178 and
 * upstream render_rays' depth sampling).  c2w: device [3,4] row-major with
 * leading dimension c2w_ld.  ray_idx (nullable): flat pixel ids y*W+x to
 * generate (training batches); NULL = all H*W pixels in row-major order.
 * n_samples == 0 skips z_vals.  perturb != 0 jitters with `jitter`
 * [n_rays,n_samples] if given, else with Philox(seed).  sphere (host,
 * nullable: cx,cy,cz,r) replaces near/far by the ray/sphere interval.
 * viewdirs, z_vals, near_far ([n,2]) are nullable outputs.                     */
int ctx_raygen_fwd(int H, int W, float fx, float fy, float cx, float cy, const float* c2w,
                   int c2w_ld, const int64_t* ray_idx, int64_t n_rays, int use_ndc,
                   float ndc_focal, float ndc_near, int n_samples, float near, float far,
                   int lindisp, int perturb, const float* jitter, uint64_t seed,
                   const uint64_t* seed_dev, int use_sphere, const float* sphere, float* rays_o,
                   float* rays_d, float* viewdirs, float* z_vals, float* near_far, void* stream);
/* seed_dev (nullable, here and in ctx_resample_fwd): a DEVICE counter added to `seed` inside the kernel, so that a
 * captured CUDA graph of the training step draws fresh Philox numbers on every replay (ctx_adam_step_dev bumps it). */

/* The same over a stack of poses (multi-view training): poses = n_views camera-to-world matrices pose_stride floats
 * apart (12 for [N,3,4], 16 for [N,4,4]), rows c2w_ld apart; ray_idx holds GLOBAL ray ids view*H*W + y*W + x
 * (upstream's rays_rgb order over [N_train, H, W]; NULL = ids 0..n_rays-1), n_views*H*W < 2^31.  Each ray takes the
 * pose of its view; a ray of view v is the ray ctx_raygen_fwd makes with pose v on the same batch row, bit for bit
 * (jitter included: it is keyed by the batch row).  One K for every view.                                        */
int ctx_raygen_views(int H, int W, float fx, float fy, float cx, float cy, const float* poses,
                     int c2w_ld, const int64_t* ray_idx, int64_t n_rays, int use_ndc,
                     float ndc_focal, float ndc_near, int n_samples, float near, float far,
                     int lindisp, int perturb, const float* jitter, uint64_t seed,
                     const uint64_t* seed_dev, int use_sphere, const float* sphere, float* rays_o,
                     float* rays_d, float* viewdirs, float* z_vals, float* near_far, int n_views, int pose_stride,
                     void* stream);

/* ---- training ray batches drawn on the device: upstream run_nerf.py train()'s samplers -------------------------
 * ray_idx [R] int64 <- R global ray ids; target (nullable, [R,3]) <- images[v, y, x, :] (images [n_views,H,W,3] fp32,
 * nullable when target is NULL).  Both modes sample without replacement through a keyed Feistel permutation
 * evaluated pointwise (construction in csrc/raybatch.cu).  counters = ctx_step_tick's pair ([0] Philox offset, [1]
 * step count t, 1 on the first step).
 * mode 0 (no_batching=True): one view per step, drawn uniformly with key seed + counters[0] on Philox stream 4 (rank
 *   in the counter), and R distinct pixels of it; while t < precrop_iters only from upstream's centre crop, rows
 *   [H/2 - crop_dh, H/2 + crop_dh) x cols [W/2 - crop_dw, W/2 + crop_dw) (crop_dh = int(H//2 * precrop_frac)).
 * mode 1 (no_batching=False): position ((t-1)*world + rank)*R + r of an epoch stream over all n_views*H*W rays, each
 *   epoch a permutation keyed by (seed, epoch): seed must be the same on every rank.  A batch that straddles an epoch
 *   boundary takes the tail of one epoch and the head of the next.  precrop_iters must be 0.
 * Bad arguments (before any launch): null ray_idx / counters, R < 0, mode 0 with R above the (cropped) pixel count,
 * an empty crop, rank outside [0, world), n_views*H*W >= 2^31.                                                  */
int ctx_draw_rays(const float* images, int n_views, int H, int W, int64_t R, int mode, int precrop_iters,
                  int crop_dh, int crop_dw, int rank, int world, uint64_t seed, const void* counters,
                  int64_t* ray_idx, float* target, void* stream);

/* z_vals [R,S] from per-ray near/far (ray_batch[:,6], ray_batch[:,7] upstream) */
int ctx_stratified_fwd(const float* near, int64_t near_stride, const float* far,
                       int64_t far_stride, int64_t R, int S, int lindisp, int perturb,
                       const float* jitter, uint64_t seed, float* z_vals, void* stream);

/* ---- ndc_rays, src/run_nerf_helpers.py:161-178 ------------------------------ */
int ctx_ndc_fwd(int H, int W, float focal, float near, const float* rays_o, const float* rays_d,
                int64_t n, float* o_out, float* d_out, void* stream);
int ctx_ndc_bwd(int H, int W, float focal, float near, const float* rays_o, const float* rays_d,
                const float* g_o, const float* g_d, int64_t n, float* g_rays_o, float* g_rays_d,
                void* stream);

/* ---- raw2outputs (absent from the reference; pointer comment at
 * src/run_nerf_helpers.py:131-133; spec SURVEY.md 8c-S1) -----------------------
 * raw [R,S,4], z_vals [R,S], rays_d [R,3], noise (nullable, [R,S], already
 * scaled by raw_noise_std) -> rgb [R,3], disp [R], acc [R], weights [R,S],
 * depth [R].  Any S up to 16384 (rays longer than 512 samples run a chunked variant
 * of the same scan).                                                             */
int ctx_composite_fwd(const float* raw, const float* z_vals, const float* rays_d,
                      const float* noise, int64_t R, int S, int white_bkgd, float* rgb_map,
                      float* disp_map, float* acc_map, float* weights, float* depth_map,
                      void* stream);
/* g_* inputs nullable (treated as zero); writes g_raw [R,S,4] */
int ctx_composite_bwd(const float* raw, const float* z_vals, const float* rays_d,
                      const float* noise, int64_t R, int S, int white_bkgd, const float* g_rgb,
                      const float* g_disp, const float* g_acc, const float* g_weights,
                      const float* g_depth, float* g_raw, void* stream);

/* ---- sample_pdf, src/run_nerf_helpers.py:182-225 ----------------------------
 * bins [R,B] with row stride bins_stride (mid_bins != 0: `bins` is z [R,B+1]
 * and the mid-points .5*(z[i+1]+z[i]) are formed in-kernel), weights [R,B-1]
 * with row stride w_stride (the reference passes the view weights[...,1:-1]).
 * cdf_in (nullable [R,B]) injects stage 1.  u (nullable [R,N]) injects the
 * uniforms; else det -> linspace(0,1,N), otherwise Philox(seed).
 * Outputs: samples [R,N]; inds (nullable, int64 [R,N]) = searchsorted result;
 * z_all (nullable [R,Sm+N]) = sort(cat[z_merge[R,Sm], samples]).               */
int ctx_resample_fwd(const float* bins, int64_t bins_stride, int mid_bins, const float* weights,
                     int64_t w_stride, const float* cdf_in, const float* u, int det,
                     uint64_t seed, const uint64_t* seed_dev, int64_t R, int B, int N, float* samples,
                     int64_t* inds, const float* z_merge, int64_t zm_stride, int Sm, float* z_all,
                     void* stream);
/* d samples / d weights -> g_weights [R,B-1] (contiguous) */
int ctx_resample_bwd(const float* bins, int64_t bins_stride, int mid_bins, const float* weights,
                     int64_t w_stride, const float* u, int det, uint64_t seed, int64_t R, int B,
                     int N, const float* g_samples, float* g_weights, void* stream);

/* Fused training form of raw2outputs (NerfTrainer.step): forward + img2mse(rgb_map, target)
 * (src/run_nerf_helpers.py:9) + backward in ONE pass over raw.  g_raw [R,S,4] = d loss / d raw with
 * loss = sum((rgb_map - target)^2) * loss_scale (loss_scale = 1/(3R) for the image mean); loss[0] += that value
 * (zero it once per step; the coarse and the fine pass add into the same scalar), summed from rgb_map [R,3] in a
 * fixed order so that it is the same on every run.  weights [R,S] is an optional output (the coarse pass feeds
 * sample_pdf with its weights).                                                                    */
int ctx_composite_train(const float* raw, const float* z_vals, const float* rays_d, const float* noise,
                        int64_t R, int S, int white_bkgd, const float* target, float loss_scale, float* loss,
                        float* g_raw, float* weights, float* rgb_map, void* stream);
/* The same with upstream's density noise (raw2outputs: sigma + randn * raw_noise_std) drawn inside the kernel, so
 * that a captured training step draws fresh noise on every replay without a noise tensor: sample s of ray r gets
 * noise_std * n, n a standard normal by Box-Muller from Philox4x32-10 with key seed + *seed_dev (seed_dev nullable)
 * and counter (r, (stream_id << 32) | (s >> 2)), one call for the four samples 4q .. 4q+3 (cos, sin of the first
 * pair, then of the second).  stream_id >= 2: streams 0 and 1 of a key are the stratified jitter and the
 * sample_pdf uniforms.  noise_std == 0 runs ctx_composite_train without noise.  ctx_density_noise writes the same
 * values as a tensor noise [R,S] (a reference for tests; reproduces a step's noise on any host).              */
int ctx_composite_train_noise(const float* raw, const float* z_vals, const float* rays_d, int64_t R, int S,
                              int white_bkgd, const float* target, float loss_scale, float* loss, float* g_raw,
                              float* weights, float* rgb_map, float noise_std, uint64_t seed,
                              const uint64_t* seed_dev, int stream_id, void* stream);
int ctx_density_noise(float* noise, int64_t R, int S, float noise_std, uint64_t seed, const uint64_t* seed_dev,
                      int stream_id, void* stream);

/* ---- coordinate MLP: NeRF2D, src/run_nerf_helpers.py:68-135 (+ the upstream
 * view-direction head kept as comments :86-95, :117-127) ----------------------
 * tcgen05/TMEM kernel, bf16 operands, fp32 accumulation, hidden width 256.
 * `net` is a HOST blob of ctx_mlp_net_bytes() bytes filled by ctx_mlp_describe:
 * D pts layers, skip_mask bit i set <=> "i in skips" (input re-concatenated
 * after layer i, :114-115), in_pts/in_views real encoding widths (63|42 / 27|0),
 * out_ch 4|3 (must be 4 with views).                                            */
int ctx_mlp_net_bytes(void);
int ctx_mlp_describe(int D, uint32_t skip_mask, int in_pts, int in_views, int out_ch, void* net);
/* params: HOST array of n_params DEVICE pointers (fp32, nn.Linear [out,in]) in
 * module order: pts_linears.{0..D-1}.{weight,bias}, then output_linear.{w,b}
 * or feature_linear, alpha_linear, views_linears.0, rgb_linear {w,b}.
 * wpacked [w_bytes], wtpacked [wt_bytes] (nullable), fparams [n_fparams]: device
 * buffers sized from the net blob (see contexture-nerf_b200/csrc/mlp_desc.h).   */
int ctx_mlp_pack(const void* net, const float* const* params, int n_params, void* wpacked,
                 void* wtpacked, float* fparams, void* stream);
/* mode 2: UV-grid texture query, see ctx_tanh01_fwd below.
 * mode 0: x [P,x_ld] holds the already-encoded input [pts_enc | view_enc];
 * mode 1: the P = R*S points o + d*z (z [R,S]) and the view directions are
 * encoded in-kernel straight into shared memory (Embedder.embed :44-45, L_pts
 * / L_dirs frequencies).  out [P,out_ch] raw network output (no activation,
 * :129).  acts (nullable): activation records for ctx_mlp_bwd, sized for a
 * multiple of 4 tiles of 128 points (the kernel works on 512 points per SM pair).*/
int ctx_mlp_fwd(const void* net, const void* wpacked, const float* fparams, int mode, const float* x,
                int x_ld, const float* rays_o, const float* rays_d, const float* viewdirs,
                const float* z, int S, int L_pts, int L_dirs, int64_t P, float* out, void* acts,
                void* stream);

/* same with an SM budget (max_sms > 0: at most that many SMs, 0 = the whole GPU), see ctx_mlp_dgrad_ex, and with
 * mode 3: x holds RAW coordinates [*, x_ld] (x_ld = 2 or 3, nets without views), encoded in-kernel with L_pts
 * frequencies; gather (nullable, int64 [P]): point p reads row gather[p] of x -- the MLP evaluated only at the
 * texels a mesh uses (get_texture_map_only_valid_areas, src/models/textured_mesh.py:303-347).                  */
int ctx_mlp_fwd_ex(const void* net, const void* wpacked, const float* fparams, int mode, const float* x,
                   int x_ld, const float* rays_o, const float* rays_d, const float* viewdirs,
                   const float* z, int S, int L_pts, int L_dirs, int64_t P, float* out, void* acts,
                   const int64_t* gather, int max_sms, void* stream);

/* Backward of ctx_mlp_fwd w.r.t. the parameters (hand-written dgrad + wgrad
 * tcgen05 kernels; the encoded inputs are data and get no gradient).  g_out
 * [P,out_ch]; acts = records written by ctx_mlp_fwd; dacts = scratch of the same
 * size; grads = HOST array of DEVICE pointers in the order of ctx_mlp_pack's
 * params; gradients are ACCUMULATED (+=) into them.                              */
int ctx_mlp_bwd(const void* net, const void* wtpacked, const float* fparams, const float* g_out,
                const void* acts, void* dacts, int64_t P, float* const* grads, int n_grads,
                const float* const* params, float* scratch, void* stream);
/* the two halves of ctx_mlp_bwd, separately launchable (and separately timed by bench.py):
 * dgrad fills the dZ records from g_out, wgrad reduces records + dZ records into the gradients. */
int ctx_mlp_dgrad(const void* net, const void* wtpacked, const float* fparams, const float* g_out,
                  const void* acts, void* dacts, int64_t P, void* stream);
/* scratch (device, ctx_mlp_wgrad_scratch_floats() floats) holds the per-CTA partial sums, which a second kernel
 * adds in a fixed order, so the gradients are the same on every run.  params (HOST array of DEVICE pointers, order
 * of ctx_mlp_pack) are read only for a view-direction net, and may be NULL for a net without views: the feature
 * layer is linear, so its weight gradients and those of views_linears.0[:, :256] are rebuilt from
 * G = [dZ_views | g_out]^T h (in scratch) and the weights instead of from records of the feature activations
 * (which are never written).                                                                                    */
int ctx_mlp_wgrad_scratch_floats(void);
int ctx_mlp_wgrad(const void* net, const void* acts, const void* dacts, int64_t P, float* const* grads,
                  int n_grads, const float* const* params, float* scratch, void* stream);
/* the same with an SM budget (max_sms > 0: at most that many SMs are occupied; 0 = the whole GPU), so that the
 * tensor-bound dgrad of one network can run beside the HBM-bound wgrad of the other on disjoint SM pairs
 * (NerfTrainer.step: dgrad_coarse || wgrad_fine).  dgrad accepts any budget >= 2 (one cluster); wgrad needs two
 * SMs per (layer, segment) job -- 28 for the view-direction net -- and returns CTX_ERR_UNSUPPORTED below that.  */
int ctx_mlp_dgrad_ex(const void* net, const void* wtpacked, const float* fparams, const float* g_out,
                     const void* acts, void* dacts, int64_t P, int max_sms, void* stream);
int ctx_mlp_wgrad_ex(const void* net, const void* acts, const void* dacts, int64_t P, float* const* grads,
                     int n_grads, const float* const* params, float* scratch, int max_sms, void* stream);

/* ---- fused texture map: get_texture_map, src/models/textured_mesh.py:266-301 -----------------------
 * ctx_mlp_fwd mode 2 generates the res x res UV grid (meshgrid of linspace(0,1,res), 'xy' indexing, :269-272),
 * encodes it (L_pts frequencies, 2-D) in shared memory and runs the 42->3 texture MLP: pass x = NULL, S = res,
 * P = res*res.  ctx_tanh01_fwd then applies (tanh+1)/2 (:299) and writes the NCHW layout [C, P] of
 * `.reshape(1,res,res,3).permute(0,3,1,2)`; ctx_tanh01_bwd is its backward (g_raw_in nullable: extra gradient
 * arriving directly on mlp_output).                                                                      */
int ctx_tanh01_fwd(const float* raw, float* out, int64_t P, int C, void* stream);
int ctx_tanh01_bwd(const float* raw, const float* g_tex, const float* g_raw_in, float* g_raw, int64_t P, int C,
                   void* stream);

/* ---- texture lookup of the rasterised mesh: kal.render.mesh.texture_mapping + mask / background composite,
 * src/models/render.py:133-140 (SURVEY.md 8f row 2).  uv [B,N,2] in [0,1] (v up), tex [tex_batch,C,H,W] with
 * tex_batch == B or 1 (one atlas shared by every view: its gradient is the sum over the views), mode 0 = nearest,
 * 1 = bilinear (grid_sample, align_corners=False, padding border).  mask (nullable, [B,N]): out = sample*mask +
 * bg*(1-mask), bg (nullable) = C background values.  Only the texture receives a gradient (upstream detaches uv);
 * ctx_texmap_bwd ACCUMULATES into g_tex.                                                                      */
int ctx_texmap_fwd(const float* uv, const float* tex, const float* mask, const float* bg, float* out, int64_t B,
                   int64_t N, int tex_batch, int C, int H, int W, int mode, void* stream);
int ctx_texmap_bwd(const float* uv, const float* mask, const float* g_out, float* g_tex, int64_t B, int64_t N,
                   int tex_batch, int C, int H, int W, int mode, void* stream);

/* dst [n,C] = 0 ; dst[idx[m]] = src[m] * scale (m < M)  -- `final_image[mask] = colors` of
 * get_texture_map_only_valid_areas (:345) -- and its backward g_src[m] = g_dst[idx[m]] * scale.                  */
int ctx_rows_scatter(const float* src, const int64_t* idx, float scale, float* dst, int64_t M, int64_t n, int C,
                     void* stream);
int ctx_rows_gather(const float* g_dst, const int64_t* idx, float scale, float* g_src, int64_t M, int C,
                    void* stream);

/* ---- training-step glue ------------------------------------------------------
 * img2mse(a,t) + img2mse(b,t) (src/run_nerf_helpers.py:9) and its gradient in one
 * pass: loss[0] = mean((a-t)^2) [+ mean((b-t)^2)], g_a = 2(a-t)/n*scale (b, g_*
 * nullable).  n = number of elements.                                            */
int ctx_mse_fwd_bwd(const float* a, const float* b, const float* target, int64_t n, float scale,
                    float* loss, float* g_a, float* g_b, void* stream);
/* torch.optim.Adam update (src/training/trainer.py:603) over flat fp32 buckets;
 * step >= 1 is the bias-correction step, grad_scale multiplies the gradient
 * (1/world_size after a sum all-reduce).                                         */
int ctx_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                  float lr, float beta1, float beta2, float eps, int step, float weight_decay,
                  float grad_scale, void* stream);

/* Device-resident step state for a CUDA-graph-captured training step (SURVEY.md 8f row 3): counters = two
 * uint64 on the device, [0] Philox seed offset (see seed_dev above), [1] Adam step count.  ctx_step_tick runs first
 * in a step: counters[0] += 2, counters[1] += 1, loss[0] = 0 (loss nullable).  ctx_adam_step_dev is ctx_adam_step
 * with the step count read from counters[1].                                                                  */
int ctx_step_tick(void* counters, float* loss, void* stream);
int ctx_adam_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                      float lr, float beta1, float beta2, float eps, const void* counters, float weight_decay,
                      float grad_scale, void* stream);
/* ctx_adam_step_dev with upstream's learning-rate decay (lrate_decay; decay_steps = lrate_decay * 1000 > 0): update
 * t = counters[1] uses lr * 0.1^(max(t - 2, 0) / decay_steps), the rate upstream's loop has set when its t-th
 * optimizer.step() runs (the loop sets lrate * 0.1^(global_step / decay_steps) after each step, global_step from 0). */
int ctx_adam_step_dev_decay(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                            float lr, float beta1, float beta2, float eps, const void* counters, float weight_decay,
                            float grad_scale, float decay_steps, void* stream);

/* ---- view-weight masks (SURVEY.md 8f row 4): ConTEXTure.create_face_view_map / compare_face_normals_between_views,
 * src/training/trainer.py:155-249 (the reference uses torch_scatter.scatter_max, :227).  face_idx [V,H,W] int64
 * (< 0 = background), face_normals [V,3,F] fp32.  mask [V,H,W] bytes: 1 unless the pixel's face has a larger
 * z-normal in another view that shows it.  visible [V*F] bytes / maxz [F] floats: caller-owned scratch.            */
int ctx_view_weight_masks(const float* face_normals, const int64_t* face_idx, int V, int F, int H, int W,
                          unsigned char* visible, float* maxz, unsigned char* mask, void* stream);
/* rows (face, view, i, j) of the covered pixels in (view, pixel) order: pass 0 fills block_counts
 * [ctx_face_view_map_blocks(V*H*W) + 1] (exclusive offsets; the last entry = number of rows N), pass 1 writes
 * rows [N,4] int64.                                                                                              */
int64_t ctx_face_view_map_blocks(int64_t n_pixels);
int ctx_face_view_map(const int64_t* face_idx, int V, int H, int W, int64_t* block_counts, int64_t* rows, int pass,
                      void* stream);

/* ---- render_rays, the coarse + fine driver (SURVEY.md 8b "fused driver", 8c S2; upstream run_nerf.py, to which
 * src/run_nerf_helpers.py:131-133 points): rays + stratified depths -> network on n_samples points -> raw2outputs ->
 * sample_pdf(z_mid, weights[...,1:-1], n_importance, det = !perturb) -> sort(cat[z, z_samples]) -> network_fine on
 * n_samples + n_importance points -> raw2outputs, as six launches on `stream`.  Inference form (no records, no
 * density noise).  Every buffer is the caller's; R = n_rays, S = n_samples, Ni = n_importance.                    */
typedef struct CtxNet {
  const void* desc;      /* host blob of ctx_mlp_describe */
  const void* wpacked;   /* device, ctx_mlp_pack */
  const float* fparams;  /* device, ctx_mlp_pack */
} CtxNet;
typedef struct CtxRenderArgs {
  int H, W;                          /* get_rays(H, W, K, c2w): K = [[fx,0,cx],[0,fy,cy],[0,0,1]] */
  float fx, fy, cx, cy;
  const float* c2w;                  /* device [3,4], leading dimension c2w_ld */
  int c2w_ld;
  const int64_t* ray_idx;            /* nullable: flat pixel ids y*W+x; NULL = pixels 0..n_rays-1 */
  int64_t n_rays;
  float near, far;
  int lindisp, perturb;              /* perturb != 0: jittered depths and random u (Philox(seed [+ *seed_dev])) */
  uint64_t seed;
  const uint64_t* seed_dev;          /* nullable device counter added to seed */
  const float* sphere;               /* HOST, nullable: (cx,cy,cz,r) -> per-ray near/far from the ray/sphere interval */
  int n_samples, n_importance;       /* n_importance == 0: single pass, results in the final maps */
  int white_bkgd;
  int L_pts, L_dirs;                 /* encoding frequencies (10 / 4); L_dirs == 0 for a net without view directions */
  int max_sms;                       /* SM budget of the MLP launches (0 = whole GPU) */
  CtxNet coarse, fine;               /* fine.desc == NULL: the coarse network serves both passes */
  /* workspace (device) */
  float *rays_o, *rays_d, *viewdirs; /* [R,3] each; viewdirs nullable when L_dirs == 0 */
  float *z_coarse, *raw_coarse, *weights_coarse;            /* [R,S], [R,S,4], [R,S] */
  float *z_samples, *z_fine, *raw_fine, *weights_fine;      /* [R,Ni], [R,S+Ni], [R,S+Ni,4], [R,S+Ni] */
  /* outputs (device): coarse maps (used when n_importance > 0) and final maps */
  float *rgb0, *disp0, *acc0, *depth0;                      /* [R,3], [R], [R], [R] */
  float *rgb_map, *disp_map, *acc_map, *depth_map;
} CtxRenderArgs;
int ctx_render_rays(const CtxRenderArgs* args, void* stream);
/* the same for forward-facing scenes: the rays are warped to NDC (ndc_rays(H, W, ndc_focal, ndc_near, ...), upstream
 * uses focal = K[0][0], near = 1) after the view directions are taken from the metric rays; near / far are NDC
 * depths (upstream: 0 and 1).  sphere must be NULL.                                                              */
int ctx_render_rays_ndc(const CtxRenderArgs* args, float ndc_focal, float ndc_near, void* stream);
int ctx_render_args_bytes(void);   /* sizeof(CtxRenderArgs) in the library (layout check for bindings) */

/* ---- evaluation metrics of a test split: upstream img2mse / mse2psnr (src/run_nerf_helpers.py:9-10) and SSIM as
 * the compute_ssim of mip-NeRF / MultiNeRF (max_val = 1; restated in csrc/metrics.cu and oracle/image_metrics.py).
 * Per-image reconstruction metrics of a batch of B images.
 * pred: [B,H,W,3] fp32 device.
 * target: [B,H,W,3] device, fp32 (target_u8 == 0) or uint8 (target_u8 == 1, read as u8 / 255.0f, IEEE division).
 * mse (nullable, [B] double): mean over H*W*3 of (pred - target)^2.  The difference is formed in fp32; squares and
 *   sums are in fp64.
 * ssim (nullable, [B] double): mean of the SSIM map (11-tap Gaussian window, sigma 1.5, valid mode) over the three
 *   channels and the (H-10) x (W-10) positions.  Neither image is clamped.
 * partials: caller-owned device workspace of ctx_image_metrics_partials(B, H, W) doubles.
 * Deterministic (no floating-point atomics), and an image gives the same bits whatever the batch around it.
 * Bad arguments: B < 0, H < 1, W < 1, target_u8 outside {0, 1}, ssim != NULL with min(H, W) < 11, a null pred /
 * target / partials when B > 0.  B == 0 returns 0.                                                               */
int ctx_image_metrics(const float* pred, const void* target, int target_u8, int B, int H, int W,
                      double* mse, double* ssim, double* partials, void* stream);
int64_t ctx_image_metrics_partials(int B, int H, int W);   /* -1 for B < 0, H < 1 or W < 1 */

/* ---- mesh extraction: the original NeRF release's extract_mesh.ipynb (density of the fine network on a regular
 * lattice with zero view directions, relu, PyMCubes marching_cubes(sigma, threshold), index -> world coordinates) and
 * a colour per vertex.  Lattice: (nx+1) x (ny+1) x (nz+1) points in C order, point (i, j, k) at
 * (ox + hx*i, oy + hy*j, oz + hz*k) formed in fp32 as __fadd_rn(o, __fmul_rn(h, (float)i)).
 *
 * ctx_density_grid: sigma [nx+1, ny+1, nz+1] fp32 = relu(raw[..., 3]) of `net` (a 4-channel net; L_pts / L_dirs its
 * encoding frequencies).  Lattice column (i, j) runs through ctx_mlp_fwd_ex mode 1 as the ray o = (x_i, y_j, 0),
 * d = (0, 0, 1) with the depth row z_k and a zero view direction; the view head is computed and discarded.  The work
 * goes in slabs of x-planes through the caller's workspace (256-byte aligned) of at least
 * ctx_density_grid_workspace(nx, ny, nz) bytes (one plane); a larger one takes bigger slabs.  The result is the same
 * bit for bit whatever the workspace size.  Bad arguments (before any launch): a cell count per axis outside
 * [1, 1024], a lattice of 2^31 points or more, a null / unsuitable net, a short or misaligned workspace.           */
int64_t ctx_density_grid_workspace(int nx, int ny, int nz);   /* -1 for sizes outside the limits above */
int ctx_density_grid(const CtxNet* net, int L_pts, int L_dirs, int nx, int ny, int nz, float ox, float oy, float oz,
                     float hx, float hy, float hz, void* workspace, int64_t workspace_bytes, float* sigma,
                     void* stream);
/* ctx_marching_cubes: the iso-surface sigma == iso of the lattice sigma [nx+1, ny+1, nz+1] (nx, ny, nz >= 1, fewer than
 * 2^31 points) placed as above.  Case table and rule: csrc/mc_tables.cuh (generated by oracle/mc_tables.py; corner c
 * at offset (c & 1, c >> 1 & 1, c >> 2 & 1), inside iff sigma >= iso, ambiguous faces separate the inside corners, so
 * neighbouring cells agree and the mesh has no cracks; triangle normals point towards decreasing density).
 * pass 0 counts: counts[0] = V (vertices), counts[1] = F (triangles), int64 on the device; read them back and allocate.
 * pass 1 writes vertices [V,3] fp32 (world coordinates), normals [V,3] fp32 (nullable) and faces [F,3] int32 (the
 *   caller checks V < 2^31).
 * Order: one vertex per lattice edge whose ends straddle iso, numbered by (linear index of the lower endpoint, then
 * axis x < y < z); position t = (iso - s0) / (s1 - s0) (IEEE division), then o + h * (idx + t) with one rounding per
 * operation.  The normal is the normalised negative density gradient (central differences, one-sided on the lattice
 * border, divided by the spacing), linearly interpolated along the edge; a zero gradient gives (0, 0, 0).  Faces come
 * in cell order, then in table order.  oracle/marching_cubes.py restates all of it bit for bit.
 * workspace: caller-owned, 256-byte aligned, ctx_marching_cubes_workspace(nx, ny, nz) bytes (about 2.5 bytes per
 * lattice point), the same buffer for both passes.  No atomics: the output is the same on every run.             */
int64_t ctx_marching_cubes_workspace(int nx, int ny, int nz);   /* -1 for sizes outside the limits above */
int ctx_marching_cubes(const float* sigma, int nx, int ny, int nz, float ox, float oy, float oz, float hx, float hy,
                       float hz, float iso, void* workspace, int64_t workspace_bytes, int64_t* counts, float* vertices,
                       float* normals, int* faces, int pass, void* stream);
/* ctx_vertex_colors: rgb [V,3] = sigmoid(raw[:, :3]) of `net` at each vertex [V,3] seen along -normal (normals
 * nullable: a zero view direction), through ctx_mlp_fwd_ex mode 1 with S = 1, o = vertex, d = 0, z = 0.  Chunks of
 * vertices go through the caller's workspace (256-byte aligned, at least ctx_vertex_colors_workspace(1) bytes;
 * ctx_vertex_colors_workspace(n) holds a chunk of n); the result is the same whatever its size.                    */
int64_t ctx_vertex_colors_workspace(int64_t n_vertices);   /* -1 for n_vertices < 1 */
int ctx_vertex_colors(const CtxNet* net, int L_pts, int L_dirs, const float* vertices, const float* normals,
                      int64_t V, void* workspace, int64_t workspace_bytes, float* rgb, void* stream);

/* ---- gradient all-reduce (SURVEY.md 8b / 8e): the one exchange step of the ray-sharded training step, replacing the
 * reduce-add of nn.DataParallel (src/training/trainer.py:134-135).  NCCL is opened at run time (dlopen; `path`
 * nullable = "libnccl.so.2" by soname), so the library has no link-time dependency on it; every call below returns
 * CTX_ERR_NO_NCCL (text in ctx_comm_last_error) when NCCL is absent or reports an error.  The communicator is an
 * opaque handle owned by the caller.  Rendezvous: one rank makes the 128-byte token with ctx_comm_unique_id and the
 * host passes it to the others; ctx_comm_init is collective and binds to the CURRENT device.  ctx_allreduce sums
 * bucket[0..n) in place on `stream`; it can be captured into a CUDA graph (all ranks capture the same sequence).  */
#define CTX_COMM_ID_BYTES 128
int ctx_comm_load(const char* path);
int ctx_comm_version(void);
const char* ctx_comm_last_error(void);
int ctx_comm_unique_id(void* id_out_host);
int ctx_comm_init(void** comm_out, int n_ranks, const void* id_host, int rank);
int ctx_comm_destroy(void* comm);
int ctx_allreduce(void* comm, float* bucket, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CTXNERF_H */
