// Weight gradients of the coordinate MLP on tcgen05 / TMEM, and the ctx_mlp_bwd entry point.
//
//   dgrad (mlp_dgrad.cu) leaves dZ of every GEMM layer in the dZ records; the forward left the layer
//   inputs in the activation records.  wgrad: dW = dZ^T * A summed over all points -- a split-K GEMM whose
//   K dimension is the point index.  Both operands are [points x features] tile images consumed as
//   MN-major operands, so no transposition pass exists anywhere.  Each CTA owns one (layer, segment) job
//   and a slice of the point tiles, accumulates in TMEM, and stores its partial sums to scratch; bias
//   gradients are column sums of dZ taken from the shared-memory tile while the MMAs run.  A second
//   kernel adds the partials of each job in CTA order into the gradients, so that they are the same on
//   every run (fp32 atomics would sum in arrival order).  The kernel is HBM-bound (1 KB read per point
//   per layer).
//
// Gradients flow to the parameters only (the encoded inputs are data).
// Reference semantics: autograd through NeRF2D.forward,
// /root/reference/src/run_nerf_helpers.py:106-135.
#include "mlp_common.cuh"
#include <string.h>
#include <stdlib.h>

// dgrad kernel launcher (mlp_dgrad.cu)
int ctx_launch_dgrad(const CtxMlpNet& net, const void* wtpacked, const float* fparams, const float* g_out,
                      const void* acts, void* dacts, int64_t P, int max_sms, cudaStream_t st);

namespace ctx {

// ============================== wgrad ======================================
// Units of the operand ring are HALF tiles (64 points x channels, <= 32 KB, contiguous in the record);
// a group = {A half, B half} feeds 4 K16 MMAs per 128-wide M half.  The ring holds as many GROUP slots of exactly
// (A bytes + B bytes) as fit into 224 KB (at most kWgMaxGroups): 3 for a 256 x 256 layer job (64 KB per group),
// 12 for the 18 KB groups of the rgb head.  Small-operand jobs are latency-bound, not bandwidth-bound: with a fixed
// number of slots they were the stragglers of the whole kernel (the rgb job at ~1.75 groups/us set its duration);
// with the bytes in flight per SM equalised every job runs at its share of the HBM bandwidth.
constexpr int kWgRingBytes = 7 * 32768;
constexpr int kWgMaxGroups = 12;
constexpr int kWgThreads = 192;     // warp 0 producer, warp 1 MMA, warps 2-5 column sums + flush
constexpr int kWgMaxJobs = 48;
constexpr size_t kWgSmemBytes = (size_t)kWgRingBytes + 512;

struct WgJob {
  int a_slot, a_ch, a_dz;       // A operand tile: record offset, channels (M, multiple of 128), from dZ records?
  int b_slot, b_ch, b_dz;       // B operand tile: channels = N (multiple of 16)
  int a_hstride, b_hstride;     // bytes between the two 64-point halves of the slot (= slot width x 128; a job may
                                // read a channel sub-range of a wider slot: any 8-aligned range of a half is contiguous)
  float* out; int ld_out; int col_off;
  int transposed;               // 1: out[(n-n_lo)*ld + col_off + m]   0: out[m*ld + col_off + (n-n_lo)]
  int m_valid, n_lo, n_hi;
  float* bias_out; int bias_from_b; int bias_lo, bias_hi;   // column sums of the dZ operand -> bias_out[c - bias_lo]
  int cta_begin, cta_count;
  float* part;        // per-CTA partials [cta][n - n_lo][m] (m < m_valid), then the bias partials [cta][c - bias_lo]
  int64_t red_begin;  // first element of this job in the reduction's index space
};
struct WgradArgs {
  int n_jobs;
  WgJob job[kWgMaxJobs];
  const uint8_t* acts; const uint8_t* dacts;
  int tile_bytes;
  int64_t n_tiles;
};
struct __align__(8) WgCtl {
  uint64_t full[kWgMaxGroups], empty[kWgMaxGroups], done;
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(kWgThreads, 1) mlp_wgrad_kernel(const __grid_constant__ WgradArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  WgCtl* ctl = reinterpret_cast<WgCtl*>(smem + kWgRingBytes);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // which job does this CTA serve?
  int ji = 0;
  for (int j = 0; j < a.n_jobs; ++j)
    if ((int)blockIdx.x >= a.job[j].cta_begin && (int)blockIdx.x < a.job[j].cta_begin + a.job[j].cta_count) ji = j;
  const WgJob& J = a.job[ji];
  const int split = blockIdx.x - J.cta_begin, cta_count = J.cta_count;
  const int a_ch = J.a_ch, b_ch = J.b_ch;
  const int m_halves = a_ch / 128;
  const uint32_t a_bytes = 64u * a_ch * 2, b_bytes = 64u * b_ch * 2;   // one 64-point half of each operand
  int64_t my_tiles = 0;
  if (split < a.n_tiles) my_tiles = (a.n_tiles - split + cta_count - 1) / cta_count;
  const int64_t my_groups = 2 * my_tiles;
  const uint32_t g_bytes = a_bytes + b_bytes;            // one group slot (multiples of 1 KB: channels come in 8s)
  int n_gs = kWgRingBytes / (int)g_bytes;
  if (n_gs > kWgMaxGroups) n_gs = kWgMaxGroups;

  if (tid == 0) {
    for (int s = 0; s < kWgMaxGroups; ++s) { tc::mbar_init(&ctl->full[s], 1); tc::mbar_init(&ctl->empty[s], 5); }
    tc::mbar_init(&ctl->done, 1);
    tc::mbar_fence_init();
  }
  if (warp == 1) tc::tmem_alloc(&ctl->tmem_base, 512);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = ctl->tmem_base;

  if (warp == 0) {
    const uint8_t* a_src = (J.a_dz ? a.dacts : a.acts) + J.a_slot;
    const uint8_t* b_src = (J.b_dz ? a.dacts : a.acts) + J.b_slot;
    const size_t tile_bytes = a.tile_bytes;
    int gs = 0; uint32_t ph = 0;
    for (int64_t gi = 0; gi < my_groups; ++gi) {
      const int64_t tile = split + (gi >> 1) * cta_count;
      const size_t base = (size_t)tile * tile_bytes;
      const int hf = (int)(gi & 1);
      tc::mbar_wait(&ctl->empty[gs], ph ^ 1);
      if (tc::elect_one()) {
        uint8_t* dst = smem + (size_t)gs * g_bytes;
        tc::mbar_arrive_expect_tx(&ctl->full[gs], g_bytes);
        tc::bulk_g2s(dst, a_src + base + (size_t)hf * J.a_hstride, a_bytes, &ctl->full[gs]);
        tc::bulk_g2s(dst + a_bytes, b_src + base + (size_t)hf * J.b_hstride, b_bytes, &ctl->full[gs]);
      }
      __syncwarp();
      if (++gs == n_gs) { gs = 0; ph ^= 1; }
    }
  } else if (warp == 1) {
    const uint32_t idesc = tc::make_idesc_bf16(128, b_ch, 1, 1);
    int gs = 0; uint32_t ph = 0;
    for (int64_t gi = 0; gi < my_groups; ++gi) {
      tc::mbar_wait(&ctl->full[gs], ph);
      tc::tc_fence_after();
      const uint32_t a_base = tc::smem_u32(smem + (size_t)gs * g_bytes);
      const uint32_t b_base = a_base + a_bytes;
      if (tc::elect_one()) {
        for (int mh = 0; mh < m_halves; ++mh) {
#pragma unroll
          for (int k16 = 0; k16 < 4; ++k16) {
            // MN-major half tile: SBO = 1024 (next 8 channels), LBO = 128 (next 8 points); 16 points = 256 B
            const uint64_t da = tc::make_smem_desc(a_base + mh * 16 * 1024 + k16 * 256, 128, 1024);
            const uint64_t db = tc::make_smem_desc(b_base + k16 * 256, 128, 1024);
            tc::mma_bf16_ss(tmem + mh * 256, da, db, idesc, (gi > 0 || k16 > 0) ? 1u : 0u);
          }
        }
        tc::mma_commit(&ctl->empty[gs]);
        if (gi == my_groups - 1) tc::mma_commit(&ctl->done);
      }
      __syncwarp();
      if (++gs == n_gs) { gs = 0; ph ^= 1; }
    }
  } else {
    // ---- column sums of the dZ operand (bias gradients), then the flush ----
    const int cw = warp - 2;  // 0..3
    const bool do_bias = J.bias_out != nullptr;
    const int bias_from_b = J.bias_from_b;
    const int dz_ch = bias_from_b ? b_ch : a_ch;
    const int n_chunks = dz_ch / 8;
    float s_lo[8], s_hi[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { s_lo[i] = 0.f; s_hi[i] = 0.f; }
    int gs = 0; uint32_t ph = 0;
    for (int64_t gi = 0; gi < my_groups; ++gi) {
      // always wait for the group: keeps these warps within one ring phase of the MMA issuer
      tc::mbar_wait(&ctl->full[gs], ph);
      if (do_bias) {
        const uint8_t* tile = smem + (size_t)gs * g_bytes + (bias_from_b ? a_bytes : 0u);
#pragma unroll
        for (int ci = 0; ci < 8; ++ci) {
          const int c = cw + ci * 4;
          if (c < n_chunks) {
#pragma unroll
            for (int gp = 0; gp < 8; ++gp) {
              const uint32_t w2 = *reinterpret_cast<const uint32_t*>(tile + c * 1024 + gp * 128 + lane * 4);
              s_lo[ci] += __uint_as_float(w2 << 16);
              s_hi[ci] += __uint_as_float(w2 & 0xffff0000u);
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&ctl->empty[gs]);
      if (++gs == n_gs) { gs = 0; ph ^= 1; }
    }
    if (do_bias) {
#pragma unroll
      for (int ci = 0; ci < 8; ++ci) {
        float lo = s_lo[ci], hi = s_hi[ci];
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
          lo += __shfl_xor_sync(CTX_FULL_MASK, lo, o);
          hi += __shfl_xor_sync(CTX_FULL_MASK, hi, o);
        }
        const int c = cw + ci * 4;
        if (c < n_chunks && lane < 4 && my_tiles > 0) {
          const int ch = c * 8 + lane * 2;
          float* bp = J.part + (size_t)cta_count * (J.n_hi - J.n_lo) * J.m_valid + (size_t)split * (J.bias_hi - J.bias_lo);
          if (ch >= J.bias_lo && ch < J.bias_hi) bp[ch - J.bias_lo] = lo;
          if (ch + 1 >= J.bias_lo && ch + 1 < J.bias_hi) bp[ch + 1 - J.bias_lo] = hi;
        }
      }
    }
    // ---- flush the TMEM accumulators: warp%4 selects the lane quarter ----
    if (my_tiles > 0) {
      tc::mbar_wait(&ctl->done, 0);
      tc::tc_fence_after();
      const int q = warp & 3;
      const int n_lo = J.n_lo, n_hi = J.n_hi, m_valid = J.m_valid;
      float* const outp = J.part + (size_t)split * (n_hi - n_lo) * m_valid;
      for (int mh = 0; mh < m_halves; ++mh) {
        const int m = mh * 128 + q * 32 + lane;
        for (int cb = 0; cb < (b_ch + 31) / 32; ++cb) {
          uint32_t vr[32];
          if (b_ch - cb * 32 >= 32) {
            tc::tmem_ld32(tmem + mh * 256 + cb * 32 + ((uint32_t)(q * 32) << 16), vr);
          } else {  // N = 16 heads: load 16 columns
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                : "=r"(vr[0]), "=r"(vr[1]), "=r"(vr[2]), "=r"(vr[3]), "=r"(vr[4]), "=r"(vr[5]), "=r"(vr[6]),
                  "=r"(vr[7]), "=r"(vr[8]), "=r"(vr[9]), "=r"(vr[10]), "=r"(vr[11]), "=r"(vr[12]), "=r"(vr[13]),
                  "=r"(vr[14]), "=r"(vr[15])
                : "r"(tmem + mh * 256 + cb * 32 + ((uint32_t)(q * 32) << 16))
                : "memory");
#pragma unroll
            for (int j = 16; j < 32; ++j) vr[j] = 0u;
          }
          tc::tmem_wait_ld(vr);
          if (m < m_valid) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int n = cb * 32 + j;
              if (n >= n_lo && n < n_hi) outp[(size_t)(n - n_lo) * m_valid + m] = __uint_as_float(vr[j]);
            }
          }
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc::tmem_dealloc(tmem, 512);
  }
}

// Sums the partials of every job over its CTAs, in CTA order, into the gradients (one thread per gradient element:
// the jobs write disjoint elements, so the result does not depend on the schedule).
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const __grid_constant__ WgradArgs a, int64_t n_elems) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n_elems; e += (int64_t)gridDim.x * blockDim.x) {
    int ji = 0;
    for (int j = 1; j < a.n_jobs; ++j)
      if (e >= a.job[j].red_begin) ji = j;
    const WgJob& J = a.job[ji];
    const int64_t k = e - J.red_begin;
    const int64_t nw = (int64_t)(J.n_hi - J.n_lo) * J.m_valid;
    const int nc = (int)(J.cta_count < a.n_tiles ? J.cta_count : a.n_tiles);
    float acc = 0.f;
    if (k < nw) {
      for (int s = 0; s < nc; ++s) acc += J.part[s * nw + k];
      const int n = (int)(k / J.m_valid), m = (int)(k % J.m_valid);
      float* dst = J.transposed ? (J.out + (size_t)n * J.ld_out + J.col_off + m)
                                : (J.out + (size_t)m * J.ld_out + J.col_off + n);
      *dst += acc;
    } else {
      const int nb = J.bias_hi - J.bias_lo, b = (int)(k - nw);
      const float* bp = J.part + (size_t)J.cta_count * nw;
      for (int s = 0; s < nc; ++s) acc += bp[s * nb + b];
      J.bias_out[b] += acc;
    }
  }
}

// Scratch of the per-CTA partials: at most kNumSMs CTAs, each with at most a 256 x 256 block and 256 bias sums.
constexpr int64_t kWgPartFloats = (int64_t)kNumSMs * (256 * 256 + 256);

// ---------------------------------------------------------------------------------------------------------
// View-direction head without a feature-layer record.  feature = W_f h + b_f is linear (no activation,
// reference comment block src/run_nerf_helpers.py:119-121), v = relu(W_vh feature + W_vd x_d + b_v).  With
//     G[h-channel m][n] = sum_points [dZ_v | g_out][point, n] * h[point, m]      (ONE wgrad job, N = 144)
//     s[n]              = sum_points [dZ_v | g_out][point, n]                     (its column sums)
// the gradients of feature_linear, of the feature columns of views_linears.0 and of alpha_linear follow exactly:
//     dW_f  = W_vh^T G_v          db_f = W_vh^T s_v
//     dW_vh = G_v W_f^T + s_v b_f^T        db_v = s_v
//     dw_alpha = G[:, 128+3]      db_alpha = s[128+3]
// (W_vh, W_f, b_f as the kernels see them: rounded to bf16).  So neither the feature activations nor dZ_feature are
// ever written to HBM, and the two 1 KB-per-point jobs that read them are replaced by one 800 B-per-point job.
// scratch: Gt [144][256] (n-major) followed by s [144], fp32, zeroed by the launcher; the wgrad partials follow.
constexpr int kPostGtFloats = 144 * 256, kPostScratchFloats = 144 * 256 + 144;
__device__ __forceinline__ float bf16r(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// One 256-thread block per 32 x 32 output tile (shared-memory tiles, K swept in steps of 32):
//   blocks [0, 64)   : dW_f[f][m]  (256 x 256, K = v over 128)     A = W_vh^T (read [v][f]), B = Gt [v][m]
//   blocks [64, 96)  : dW_vh[v][f] (128 x 256, K = m over 256)     A = Gt [v][m],            B = W_f^T (read [f][m])
//   block 96         : alpha head + the three bias vectors
__global__ void __launch_bounds__(256) wgrad_post_kernel(
    const float* __restrict__ scratch, const float* __restrict__ W_f, const float* __restrict__ b_f,
    const float* __restrict__ W_v, int ld_v, float* __restrict__ gW_f, float* __restrict__ gb_f,
    float* __restrict__ gW_v, float* __restrict__ gb_v, float* __restrict__ gw_alpha, float* __restrict__ gb_alpha) {
  const float* Gt = scratch;
  const float* sv = scratch + kPostGtFloats;
  __shared__ float sA[32][33], sB[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8 threads, 4 outputs each (rows ty, ty+8, ...)
  const int blk = blockIdx.x;
  if (blk < 64) {
    const int f0 = (blk >> 3) * 32, m0 = (blk & 7) * 32;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int v0 = 0; v0 < 128; v0 += 32) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int v = v0 + ty + 8 * r;
        sA[ty + 8 * r][tx] = bf16r(__ldg(W_v + v * ld_v + f0 + tx));   // [v][f]
        sB[ty + 8 * r][tx] = Gt[v * 256 + m0 + tx];                    // [v][m]
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const float b = sB[k][tx];
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[r] = fmaf(sA[k][ty + 8 * r], b, acc[r]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) gW_f[(f0 + ty + 8 * r) * 256 + m0 + tx] += acc[r];
    return;
  }
  if (blk < 96) {
    const int t = blk - 64;
    const int v0 = (t >> 3) * 32, f0 = (t & 7) * 32;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int m0 = 0; m0 < 256; m0 += 32) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        sA[ty + 8 * r][tx] = Gt[(v0 + ty + 8 * r) * 256 + m0 + tx];               // [v][m]
        sB[ty + 8 * r][tx] = bf16r(__ldg(W_f + (f0 + ty + 8 * r) * 256 + m0 + tx));   // [f][m]
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const float b = sB[tx][k];
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[r] = fmaf(sA[ty + 8 * r][k], b, acc[r]);
      }
      __syncthreads();
    }
    const float bf = bf16r(b_f[f0 + tx]);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int v = v0 + ty + 8 * r;
      gW_v[v * ld_v + f0 + tx] += acc[r] + sv[v] * bf;
    }
    return;
  }
  // heads and biases
  const int i = threadIdx.x;
  gw_alpha[i] += Gt[(128 + 3) * 256 + i];
  if (i == 0) gb_alpha[0] += sv[128 + 3];
  if (i < 128) gb_v[i] += sv[i];
  {
    float b = 0.f;                                            // db_f[f] = sum_v W_vh[v][f] s_v
    for (int v = 0; v < 128; ++v) b = fmaf(bf16r(__ldg(W_v + v * ld_v + i)), sv[v], b);
    gb_f[i] += b;
  }
}

}  // namespace ctx

// grads: HOST array of DEVICE pointers in the order of ctx_mlp_pack's `params`
// (gradients are ACCUMULATED into them: zero them first for a fresh gradient).
// params: the fp32 parameters themselves, same order (the view-direction head rebuilds the gradients of
// feature_linear / views_linears.0[:, :256] from G and the weights, see wgrad_post_kernel; only used with a
// view-direction net, may be null otherwise); scratch: device buffer of ctx_mlp_wgrad_scratch_floats() floats.
// max_sms > 0: use at most that many CTAs (rounded down to even) and launch them as 2-CTA clusters, so that they
// pack into whole SM pairs and a concurrent cluster kernel (dgrad of the other network) finds free pairs.
extern "C" int ctx_mlp_wgrad_scratch_floats(void) { return (int)(ctx::kPostScratchFloats + ctx::kWgPartFloats); }

extern "C" int ctx_mlp_wgrad_ex(const void* net_host, const void* acts, const void* dacts, int64_t P,
                                float* const* grads, int n_grads, const float* const* params, float* scratch,
                                int max_sms, void* stream) {
  if (P < 0) return CTX_ERR_BAD_ARG;
  if (P == 0) return 0;
  if (!net_host || !acts || !dacts || !grads || !scratch) return CTX_ERR_BAD_ARG;
  const CtxMlpNet& net = *reinterpret_cast<const CtxMlpNet*>(net_host);
  const bool views = net.in_views > 0;
  const int D = views ? net.n_layers - 2 : net.n_layers;
  if (n_grads != 2 * D + (views ? 8 : 2)) return CTX_ERR_BAD_ARG;
  if (views && !params) return CTX_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  static ctx::DeviceOnce attr_once;
  if (attr_once.needed()) {
    cudaError_t e = cudaFuncSetAttribute(ctx::mlp_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)ctx::kWgSmemBytes);
    if (e != cudaSuccess) return (int)e;
  }
  if (views) {
    cudaError_t e = cudaMemsetAsync(scratch, 0, sizeof(float) * ctx::kPostScratchFloats, st);
    if (e != cudaSuccess) return (int)e;
  }
  // ---------------- wgrad ----------------
  {
    ctx::WgradArgs w;
    memset(&w, 0, sizeof(w));
    w.acts = (const uint8_t*)acts; w.dacts = (const uint8_t*)dacts; w.tile_bytes = net.act_tile_bytes;
    const int64_t n_tiles = ctx::ceil_div(P, 128);
    w.n_tiles = n_tiles;
    int nj = 0;
    float cost[ctx::kWgMaxJobs];
    // operand = (slot byte offset, slot channel width, first channel, channels)
    struct Opnd { int slot, rec_ch, ch0, ch, dz; };
    auto add = [&](Opnd A, Opnd B, float* out, int ld, int col_off, int transposed, int m_valid, int n_lo, int n_hi,
                   float* bias, int bias_from_b, int blo, int bhi) {
      ctx::WgJob& J = w.job[nj];
      J.a_slot = A.slot + (A.ch0 >> 3) * 1024; J.a_ch = A.ch; J.a_dz = A.dz; J.a_hstride = A.rec_ch * 128;
      J.b_slot = B.slot + (B.ch0 >> 3) * 1024; J.b_ch = B.ch; J.b_dz = B.dz; J.b_hstride = B.rec_ch * 128;
      J.out = out; J.ld_out = ld; J.col_off = col_off; J.transposed = transposed; J.m_valid = m_valid;
      J.n_lo = n_lo; J.n_hi = n_hi; J.bias_out = bias; J.bias_from_b = bias_from_b; J.bias_lo = blo; J.bias_hi = bhi;
      cost[nj] = (float)(A.ch + B.ch);   // HBM bytes per point decide the split, the kernel is bandwidth-bound
      ++nj;
    };
    const Opnd XP = {net.xp_slot, CTX_MLP_XP_PAD, 0, CTX_MLP_XP_PAD, 0};
    const Opnd XD = {net.xd_slot, CTX_MLP_XD_PAD, 0, CTX_MLP_XD_PAD, 0};
    const Opnd GOUT = {net.gout_slot, net.gout_rec_ch, net.gout_ch0, 16, 1};
    for (int l = 0; l < net.n_layers; ++l) {
      const CtxMlpLayer& L = net.L[l];
      if (views && l == D) continue;   // feature_linear: rebuilt from G (below)
      const bool is_views_layer = views && l == D + 1;
      int pi;
      if (l < D) pi = 2 * l; else pi = 2 * D + 4;
      float* gW = grads[pi];
      float* gb = grads[pi + 1];
      int ld = 0;
      if (L.n_x_pre) ld += net.in_pts;
      const int h_col = ld;
      if (L.n_h) ld += 256;
      const int xd_col = ld;
      if (L.n_x_post) ld += net.in_views;
      const Opnd DZ = {L.act_slot, L.rec_ch, 0, L.N, 1};
      bool bias_done = false;
      if (L.n_h && !is_views_layer) {  // h segment: transposed job, A = input activations (M = in), B = dZ (N = out)
        add({L.in_slot, 256, 0, 256, 0}, DZ, gW, ld, h_col, 1, 256, 0, L.N, gb, 1, 0, L.N);
        bias_done = true;
      }
      if (L.n_x_pre) {  // point-encoding segment: A = dZ (M = out), B = x_p tile (N = 64, 63 real)
        add(DZ, XP, gW, ld, 0, 0, L.N, 0, net.in_pts, bias_done ? nullptr : gb, 0, 0, L.N);
        bias_done = true;
      }
      if (L.n_x_post) {  // view-encoding segment (its bias comes out of the G job's column sums)
        add(DZ, XD, gW, ld, xd_col, 0, L.N, 0, net.in_views, nullptr, 0, 0, 0);
      }
    }
    if (views) {
      const CtxMlpLayer& H = net.L[D - 1];           // h_{D-1}: input of feature_linear and alpha_linear
      const CtxMlpLayer& V = net.L[net.n_layers - 1];
      // G job: A = h_{D-1} (M = 256), B = [dZ_views | g_out] (N = 144) -> Gt [144][256] and the column sums s [144]
      add({H.act_slot, 256, 0, 256, 0}, {V.act_slot, V.rec_ch, 0, V.rec_ch, 1}, scratch, 256, 0, 1, 256, 0, V.rec_ch,
          scratch + ctx::kPostGtFloats, 1, 0, V.rec_ch);
      // rgb_linear: A = v (M = 128), B = g_out (N = 16, channels 0..2 are g_rgb)
      add({V.act_slot, V.rec_ch, 0, 128, 0}, GOUT, grads[2 * D + 6], 128, 0, 1, 128, 0, 3, grads[2 * D + 7], 1, 0, 3);
    } else {
      const CtxMlpLayer& H = net.L[D - 1];
      add({H.act_slot, 256, 0, 256, 0}, GOUT, grads[2 * D], 256, 0, 1, 256, 0, net.out_ch, grads[2 * D + 1], 1,
          0, net.out_ch);
    }
    // distribute the CTAs over the jobs proportionally to their HBM traffic
    float total = 0.f;
    for (int j = 0; j < nj; ++j) total += cost[j];
    int budget = ctx::num_sms(), begin = 0;
    if (budget > ctx::kNumSMs) budget = ctx::kNumSMs;
    const bool capped = max_sms > 0 && max_sms < budget;
    if (capped) budget = max_sms & ~1;
    if (budget < 2 * nj) return CTX_ERR_UNSUPPORTED;
    int given[ctx::kWgMaxJobs];
    int used = 0;
    for (int j = 0; j < nj; ++j) {
      int c = (int)(cost[j] / total * (budget - nj)) + 1;
      if ((int64_t)c > n_tiles) c = (int)n_tiles;
      if (c < 1) c = 1;
      given[j] = c; used += c;
    }
    for (int j = 0; used < budget && j < 4 * nj; ++j) {   // hand out the remainder to the big jobs
      const int k = j % nj;
      if (cost[k] >= 384.f && (int64_t)given[k] < n_tiles) { ++given[k]; ++used; }
    }
    float* part = scratch + ctx::kPostScratchFloats;
    int64_t red = 0;
    for (int j = 0; j < nj; ++j) {
      ctx::WgJob& J = w.job[j];
      J.cta_begin = begin; J.cta_count = given[j]; begin += given[j];
      if (!J.bias_out) J.bias_lo = J.bias_hi = 0;
      const int64_t per_cta = (int64_t)(J.n_hi - J.n_lo) * J.m_valid + (J.bias_hi - J.bias_lo);
      J.part = part; part += per_cta * given[j];
      J.red_begin = red; red += per_cta;
    }
    if (part > scratch + ctx::kPostScratchFloats + ctx::kWgPartFloats) return CTX_ERR_UNSUPPORTED;
    w.n_jobs = nj;
    if (capped && (begin & 1) == 0) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(begin); cfg.blockDim = dim3(ctx::kWgThreads); cfg.dynamicSmemBytes = ctx::kWgSmemBytes;
      cfg.stream = st;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      cudaError_t e = cudaLaunchKernelEx(&cfg, ctx::mlp_wgrad_kernel, w);
      if (e != cudaSuccess) return (int)e;
    } else {
      ctx::mlp_wgrad_kernel<<<begin, ctx::kWgThreads, ctx::kWgSmemBytes, st>>>(w);
    }
    ctx::wgrad_reduce_kernel<<<2 * budget, 256, 0, st>>>(w, red);
  }
  {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
  }
  if (views) {
    const int ld_v = 256 + net.in_views;
    ctx::wgrad_post_kernel<<<97, 256, 0, st>>>(scratch, params[2 * D], params[2 * D + 1],
                                                                params[2 * D + 4], ld_v, grads[2 * D], grads[2 * D + 1],
                                                                grads[2 * D + 4], grads[2 * D + 5], grads[2 * D + 2],
                                                                grads[2 * D + 3]);
  }
  CTX_RETURN_LAST();
}

extern "C" int ctx_mlp_wgrad(const void* net_host, const void* acts, const void* dacts, int64_t P,
                             float* const* grads, int n_grads, const float* const* params, float* scratch,
                             void* stream) {
  return ctx_mlp_wgrad_ex(net_host, acts, dacts, P, grads, n_grads, params, scratch, 0, stream);
}

extern "C" int ctx_mlp_dgrad_ex(const void* net_host, const void* wtpacked, const float* fparams, const float* g_out,
                                const void* acts, void* dacts, int64_t P, int max_sms, void* stream) {
  if (P < 0) return CTX_ERR_BAD_ARG;
  if (P == 0) return 0;
  if (!net_host || !wtpacked || !fparams || !g_out || !acts || !dacts) return CTX_ERR_BAD_ARG;
  return ctx_launch_dgrad(*reinterpret_cast<const CtxMlpNet*>(net_host), wtpacked, fparams, g_out, acts, dacts, P,
                          max_sms, (cudaStream_t)stream);
}

extern "C" int ctx_mlp_dgrad(const void* net_host, const void* wtpacked, const float* fparams, const float* g_out,
                             const void* acts, void* dacts, int64_t P, void* stream) {
  return ctx_mlp_dgrad_ex(net_host, wtpacked, fparams, g_out, acts, dacts, P, 0, stream);
}

extern "C" int ctx_mlp_bwd(const void* net_host, const void* wtpacked, const float* fparams,
                           const float* g_out, const void* acts, void* dacts, int64_t P, float* const* grads,
                           int n_grads, const float* const* params, float* scratch, void* stream) {
  const int rc = ctx_mlp_dgrad(net_host, wtpacked, fparams, g_out, acts, dacts, P, stream);
  if (rc != 0) return rc;
  return ctx_mlp_wgrad(net_host, acts, dacts, P, grads, n_grads, params, scratch, stream);
}
