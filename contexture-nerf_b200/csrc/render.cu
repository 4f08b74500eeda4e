// ctx_render_rays: the coarse + fine render_rays driver behind one C-ABI call (SURVEY.md 8b "fused driver", 8c S2).
//
// The reference tree has no render_rays (only the pointer at /root/reference/src/run_nerf_helpers.py:131-133 to
// upstream's run_nerf.py); the sequence restated in oracle/nerf_oracle.py is: rays + stratified depths -> network on the
// N_samples points -> raw2outputs -> sample_pdf on the mid-points with weights[..., 1:-1] -> sort(cat[z, z_samples]) ->
// network_fine on the N_samples + N_importance points -> raw2outputs.  Here that is six launches enqueued back to back
// on the caller's stream: raygen (fused with the stratified depths), MLP forward (encoding fused), compositing,
// resample fused with the merge, MLP forward, compositing.  Host-only code: every kernel lives in its own file and is
// reached through the same extern "C" launchers a host could call one by one; buffers are the caller's.
#include "ctx_common.cuh"
#include "ctxnerf.h"

// sizeof(CtxRenderArgs) as this library was compiled: lets a binding check its own struct layout
extern "C" int ctx_render_args_bytes(void) { return (int)sizeof(CtxRenderArgs); }

// use_ndc: the raygen launch warps the rays to NDC (ndc_rays(H, W, ndc_focal, ndc_near, ...)) after taking the view
// directions, as upstream render() does for forward-facing scenes; near / far are then NDC depths.
static int render_rays(const CtxRenderArgs* a, int use_ndc, float ndc_focal, float ndc_near, void* stream) {
  if (!a || a->n_rays < 0 || a->n_samples < 2 || a->n_importance < 0) return CTX_ERR_BAD_ARG;
  if (a->n_rays == 0) return 0;
  const int S = a->n_samples, Ni = a->n_importance, Sf = S + Ni;
  const int64_t R = a->n_rays;
  const bool hier = Ni > 0;
  if (!a->coarse.desc || !a->coarse.wpacked || !a->coarse.fparams) return CTX_ERR_BAD_ARG;
  if (!a->rays_o || !a->rays_d || !a->z_coarse || !a->raw_coarse || !a->weights_coarse) return CTX_ERR_BAD_ARG;
  if (!a->rgb_map || !a->disp_map || !a->acc_map || !a->depth_map) return CTX_ERR_BAD_ARG;
  if (hier && (!a->z_samples || !a->z_fine || !a->raw_fine || !a->weights_fine || !a->rgb0 || !a->disp0 || !a->acc0 ||
               !a->depth0 || S < 3))
    return CTX_ERR_BAD_ARG;
  if (a->L_dirs > 0 && !a->viewdirs) return CTX_ERR_BAD_ARG;
  const CtxNet& fine = a->fine.desc ? a->fine : a->coarse;        // network_fine or network_fn
  if (!fine.wpacked || !fine.fparams) return CTX_ERR_BAD_ARG;

  int rc = ctx_raygen_fwd(a->H, a->W, a->fx, a->fy, a->cx, a->cy, a->c2w, a->c2w_ld, a->ray_idx, R, use_ndc,
                          ndc_focal, ndc_near, S, a->near, a->far, a->lindisp, a->perturb, nullptr, a->seed, a->seed_dev,
                          a->sphere != nullptr, a->sphere, a->rays_o, a->rays_d, a->viewdirs, a->z_coarse, nullptr,
                          stream);
  if (rc) return rc;
  rc = ctx_mlp_fwd_ex(a->coarse.desc, a->coarse.wpacked, a->coarse.fparams, 1, nullptr, 0, a->rays_o, a->rays_d,
                      a->viewdirs, a->z_coarse, S, a->L_pts, a->L_dirs, R * S, a->raw_coarse, nullptr, nullptr,
                      a->max_sms, stream);
  if (rc) return rc;
  // without a fine pass the coarse maps are the result
  rc = ctx_composite_fwd(a->raw_coarse, a->z_coarse, a->rays_d, nullptr, R, S, a->white_bkgd,
                         hier ? a->rgb0 : a->rgb_map, hier ? a->disp0 : a->disp_map, hier ? a->acc0 : a->acc_map,
                         a->weights_coarse, hier ? a->depth0 : a->depth_map, stream);
  if (rc || !hier) return rc;
  // sample_pdf(z_mid, weights[..., 1:-1], Ni, det = (perturb == 0)) + sort(cat[z, z_samples]) in one launch: the bins
  // are formed in-kernel from z, the weights view is the row pointer + 1 with stride S
  rc = ctx_resample_fwd(a->z_coarse, S, 1, a->weights_coarse + 1, S, nullptr, nullptr, a->perturb == 0, a->seed + 1,
                        a->seed_dev, R, S - 1, Ni, a->z_samples, nullptr, a->z_coarse, S, S, a->z_fine, stream);
  if (rc) return rc;
  rc = ctx_mlp_fwd_ex(fine.desc, fine.wpacked, fine.fparams, 1, nullptr, 0, a->rays_o, a->rays_d, a->viewdirs,
                      a->z_fine, Sf, a->L_pts, a->L_dirs, R * Sf, a->raw_fine, nullptr, nullptr, a->max_sms, stream);
  if (rc) return rc;
  return ctx_composite_fwd(a->raw_fine, a->z_fine, a->rays_d, nullptr, R, Sf, a->white_bkgd, a->rgb_map, a->disp_map,
                           a->acc_map, a->weights_fine, a->depth_map, stream);
}

extern "C" int ctx_render_rays(const CtxRenderArgs* a, void* stream) { return render_rays(a, 0, 0.f, 0.f, stream); }

extern "C" int ctx_render_rays_ndc(const CtxRenderArgs* a, float ndc_focal, float ndc_near, void* stream) {
  // the bounding-sphere interval is metric: it has no meaning for NDC rays
  if (!a || !(ndc_focal > 0.f) || !(ndc_near > 0.f) || a->sphere) return CTX_ERR_BAD_ARG;
  return render_rays(a, 1, ndc_focal, ndc_near, stream);
}
