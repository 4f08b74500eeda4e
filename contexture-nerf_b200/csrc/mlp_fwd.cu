// Fused coordinate-MLP forward on tcgen05 / TMEM (sm_100a): 2-CTA MMAs (cta_group::2) + ping-pong.
//
// A cluster of two CTAs (one SM pair) owns 512 points per iteration, arranged as
// two 256-row tile pairs A and B (each CTA holds 128 rows of A and 128 rows of B,
// i.e. two 128x256 fp32 accumulators = all 512 TMEM columns).  Every
// MMA is M=256 across the pair: each CTA feeds its own 128 activation rows and
// HALF of the weight rows (N/2), so per CTA the B-operand shared-memory reads and
// the weight staging are halved with respect to cta_group::1.  Layers alternate
// between the tile pairs,
//     MMA(l, A) | MMA(l, B) | MMA(l+1, A) | ...
//                 epi(l, A) | epi(l, B)   | ...
// so the TMEM->ReLU->bf16->shared-memory epilogue of one pair (and, when
// training, the activation-record stores) runs under the MMAs of the other one.
// Weights are streamed twice per layer (once per pair) as 8 KB half-chunks by
// 1-D bulk TMA through an 8-stage ring (1.2 MB of L2 reads per CTA per 256 points).
//
// Synchronisation: full/empty/acc_full barriers are local to each CTA (the MMA
// completion is multicast to both with tcgen05.commit...multicast::cluster).  The
// leader's `full` barrier of a ring pair counts two arrivals: its own producer's and
// the peer's "my half landed too", relayed by the peer's otherwise idle warp 1 with a
// remote mbarrier arrive -- so an issuer makes one wait per 16 KB of weights.  Each
// issuer is ONE elected thread running the whole loop (no per-chunk elect / warp
// sync); it also waits for both CTAs' epilogue warps to be done with the next A
// operand (act_ready, 16 warp arrivals, the peer's are remote).  The two issuers
// consume interleaved ring pairs and mbarrier waits only see the phase parity: the
// first pairs of a layer phase check `empty` of the pair's previous use (possibly the
// other issuer's) before trusting `full`.  tcgen05.wait::ld is tied to the loaded
// registers so that their consumers cannot be scheduled above it.
//
// Reference semantics: NeRF2D.forward, /root/reference/src/run_nerf_helpers.py:106-135
// (+ commented view branch :117-127); Embedder.embed :44-45.
#include "mlp_common.cuh"

namespace ctx {

// Measured and not kept (round 2, profiles/README.md): sixteen epilogue warps on 16-column blocks (four per TMEM lane
// quarter, 104 registers) -- training forward 0.95 -> 1.01 ms; eight warps on 16-column blocks -- 0.950 -> 0.966 ms:
// the epilogue is not latency-bound per warp.  A setmaxnreg split must hand out exactly what the CTA was launched with
// (4 x 56 + 8 x 224 = 12 x 168 here): setmaxnreg.inc only draws on registers the CTA itself released, and a split
// that asks for more (4 x 56 + 16 x 112 > 20 x 96) hangs the kernel.  Shipping each finished activation tile to its
// record with one TMA tensor store from a store warp, instead of the epilogue's register stores: 0.95 -> 1.14 ms.
constexpr int kStages2 = 8;          // 8 KB half-chunk stages, handled in PAIRS (one full/empty barrier per pair)
constexpr int kPairs2 = kStages2 / 2;
constexpr int kHeadFloats = 648;    // view-direction head block staged in shared memory (w_alpha, W_rgb, biases)
constexpr int kStage2Bytes = kStageBytes / 2;   // 8 KB half-chunk

struct __align__(8) Mlp2SmemCtl {
  uint64_t full[kPairs2], empty[kPairs2];
  uint64_t acc_full[kTiles], act_ready[kTiles];
  uint32_t tmem_base;
};
constexpr size_t kMlp2SmemBytes = (size_t)kTiles * (kHBytes + kXBytes) + (size_t)kStages2 * kStage2Bytes +
                                  kHeadFloats * 4 + 256;

template <int PAD, int MAXL, int D = 3>
__device__ __forceinline__ void encode_row2(uint8_t* tile, int row, const float* xyz, int L, bool valid,
                                            uint8_t* gtile) {
  float v[PAD];
#pragma unroll
  for (int i = 0; i < PAD; ++i) v[i] = 0.f;
  if (valid) {
#pragma unroll
    for (int j = 0; j < D; ++j) v[j] = xyz[j];
#pragma unroll
    for (int k = 0; k < MAXL; ++k) {
      if (k < L) {
        const float f = (float)(1 << k);
#pragma unroll
        for (int j = 0; j < D; ++j) {
          float s, c;
          fast_sincos(xyz[j] * f, s, c);
          const int b = D + k * 2 * D;
          if (b + D + j < PAD) { v[b + j] = s; v[b + D + j] = c; }
        }
      }
    }
  }
  v[PAD - 1] = 1.0f;   // constant-1 channel: carries the bias through the GEMM
#pragma unroll
  for (int c0 = 0; c0 < PAD; c0 += 8) store_row8(tile, row, c0, v + c0, false, gtile, PAD);
}

// Diagnostics: spin on an mbarrier; when a (pinned, host-visible) buffer is supplied a waiter that has been
// stuck for ~0.2 s records {tag, block, warp, info, parity} there and traps, so a deadlock names its waiters.
__device__ __forceinline__ void hang_report(unsigned long long* buf, uint32_t tag, uint32_t info, uint32_t parity) {
  const unsigned long long i = atomicAdd(buf, 1ull);
  if (i < 60) {
    unsigned long long* e = buf + 8 + i * 4;
    e[0] = tag; e[1] = ((unsigned long long)blockIdx.x << 32) | (threadIdx.x >> 5); e[2] = info; e[3] = parity;
  }
  __threadfence_system();
  const long long t0 = clock64();
  while (clock64() - t0 < 200000000ll) {
  }
  __trap();
}
template <bool kDiag>
__device__ __forceinline__ void mbar_wait_dbg(uint32_t addr, uint32_t parity, unsigned long long* buf, uint32_t tag,
                                              uint32_t info) {
  if constexpr (!kDiag) {   // production kernels: the plain spin
    tc::mbar_wait_addr(addr, parity);
    return;
  }
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
  if (ok) return;
  const long long t0 = clock64();
  for (;;) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    if (ok) return;
    if (buf && clock64() - t0 > 400000000ll) hang_report(buf, tag, info, parity);
  }
}

template <bool kProf, bool kRec>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kMlpThreads, 1)
mlp_fwd_kernel(const __grid_constant__ MlpFwdArgs a) {
#define PCLK() (kProf ? clock64() : 0ll)
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* h_buf = smem;
  uint8_t* x_buf = smem + kTiles * kHBytes;
  uint8_t* w_buf = x_buf + kTiles * kXBytes;
  float* s_head = reinterpret_cast<float*>(w_buf + kStages2 * kStage2Bytes);   // head weights, loaded once
  Mlp2SmemCtl* ctl = reinterpret_cast<Mlp2SmemCtl*>(s_head + kHeadFloats);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t r = tc::cluster_ctarank();
  const CtxMlpNet& net = a.net;
  const int64_t n_citers = ceil_div(a.P, (int64_t)kTileM * 4);
  const int64_t cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;
  const uint8_t* wstream = a.wpacked;   // half-split chunk layout (mlp_pack.cu)

  if (tid == 0) {
    for (int s = 0; s < kPairs2; ++s) {
      // leader: its own producer's arrive + the peer's relay ("my half landed too")
      tc::mbar_init(&ctl->full[s], r == 0 ? 2 : 1); tc::mbar_init(&ctl->empty[s], 1);
    }
    for (int t = 0; t < kTiles; ++t) {
      tc::mbar_init(&ctl->acc_full[t], 1); tc::mbar_init(&ctl->act_ready[t], 16);
    }
    tc::mbar_fence_init();
  }
  if (warp == 1) tc::tmem_alloc2(&ctl->tmem_base, 512);
  {
    if (net.in_views > 0)
      for (int i = tid; i < kHeadFloats; i += kMlpThreads) s_head[i] = a.fparams[net.head_off + i];
  }
  tc::tc_fence_before();
  tc::cluster_sync_all();
  tc::tc_fence_after();
  const uint32_t tmem = ctl->tmem_base;
  // registers: from the control warpgroup to the two epilogue warpgroups (every warp of a warpgroup executes its call)
  // (the calls sit INSIDE the role branches: ptxas budgets each region by the setmaxnreg that dominates it)
  if (warp < 4) {
  reg_dealloc<kCtlRegs>();
  if (warp == 0) {
    // ============ weight-stream producer: this CTA's half of every chunk, twice per layer ============
    // chunks are staged in pairs: one expect_tx / full barrier covers two consecutive 8 KB stages
    {
      uint32_t g = 0;
      for (int64_t it = cid; it < n_citers; it += ncl) {
        for (int l = 0; l < net.n_layers; ++l) {
          // (layer fields are copied to registers: the asm memory clobbers would otherwise force a
          //  constant-bank reload of every field on every chunk)
          const int nchunks = net.L[l].n_x_pre + net.L[l].n_h + net.L[l].n_x_post;
          const int ntot = nchunks + net.L[l].bias_mma;
          const int npad = (ntot + 1) & ~1;   // phases are padded to whole chunk PAIRS (dummy chunk: no copy)
          const uint32_t half = (uint32_t)net.L[l].N * CTX_MLP_KC;   // (N/2 rows) x 32 K x 2 B
          const uint8_t* lsrc = wstream + net.L[l].w_off;
          for (int ph = 0; ph < 2; ++ph) {
            for (int c = 0; c < npad; ++c, ++g) {
              const int s = g % kStages2, pr = s >> 1;
              // regular chunk: 32 K ; trailing bias chunk (c == nchunks): 16 K
              const uint32_t bytes = c < nchunks ? half : half / 2;
              if (!(g & 1)) mbar_wait_dbg<kProf>(tc::smem_u32(&ctl->empty[pr]), ((g / kStages2) & 1) ^ 1, a.hang, 1, (uint32_t)(l * 1000 + g % 1000));
              if (tc::elect_one()) {
                if (c < ntot) {
                  tc::mbar_expect_tx(&ctl->full[pr], bytes);
                  tc::bulk_g2s(w_buf + s * kStage2Bytes, lsrc + (size_t)c * 2 * half + r * bytes, bytes, &ctl->full[pr]);
                }
                if (g & 1) tc::mbar_arrive(&ctl->full[pr]);
              }
              __syncwarp();
            }
          }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    {
      if (r != 0) {
        if (warp == 1) {
        // ============ peer CTA: relay "my half landed" to the leader ============
        uint32_t g = 0;
        for (int64_t it = cid; it < n_citers; it += ncl)
          for (int l = 0; l < net.n_layers; ++l) {
            const int nchunks = (net.L[l].n_x_pre + net.L[l].n_h + net.L[l].n_x_post + net.L[l].bias_mma + 1) & ~1;
            for (int c = 0; c < 2 * nchunks; ++c, ++g) {
              if (g & 1) {   // one relay per chunk pair
                const int pr = (g % kStages2) >> 1;
                mbar_wait_dbg<kProf>(tc::smem_u32(&ctl->full[pr]), (g / kStages2) & 1, a.hang, 2, (uint32_t)(l * 1000 + g % 1000));
                if (tc::elect_one()) tc::mbar_arrive_remote(&ctl->full[pr], 0);
                __syncwarp();
              }
            }
          }
        }
      } else {
        // ============ leader CTA: two MMA issuers, warp 1 -> tile pair A, warp 2 -> tile pair B ============
        // Issuing is single-thread work (~400 cycles of dependent instructions per chunk: barrier polls,
        // descriptor builds, vector->uniform register moves); one thread cannot keep a 128-cycle-per-MMA
        // pipe fed, two threads working on alternate phases can.  Phases are padded to whole chunk pairs so
        // each issuer owns (waits on, commits) complete ring pairs.
        const int ph = warp == 1 ? 0 : 1;
        long long t_act = 0, t_full = 0, t_peer = 0, t_issue = 0;
        const long long t_begin = PCLK();
        if (tc::elect_one()) {
          // One thread runs the whole issue loop (no per-chunk elect / warp sync).  Descriptor hi words are
          // constants; the lo words (address>>4 | LBO>>4<<16) advance by integer adds.  A ring pair = 2 chunks
          // = up to 4 MMAs per barrier wait, one commit per pair.
          constexpr uint32_t kDescHi = (128u >> 4) | (1u << 14);            // SBO = 128 B, descriptor version 1
          constexpr uint32_t kALbo = (uint32_t)(kK8Stride >> 4) << 16;
          constexpr uint32_t kAStep = 4 * kK8Stride >> 4;                   // one 32-wide K chunk of an A tile
          const uint32_t x_lo = kALbo | (tc::smem_u32(x_buf + ph * kXBytes) >> 4);
          const uint32_t h_lo = kALbo | (tc::smem_u32(h_buf + ph * kHBytes) >> 4);
          const uint32_t w_lo = tc::smem_u32(w_buf) >> 4;
          const uint32_t full0 = tc::smem_u32(&ctl->full[0]), empty0 = tc::smem_u32(&ctl->empty[0]);
          const uint32_t accf = tc::smem_u32(&ctl->acc_full[ph]), actr = tc::smem_u32(&ctl->act_ready[ph]);
          const uint32_t acc = tmem + ph * CTX_MLP_W;
          uint32_t gl = 0, act_phase = 0;
          for (int64_t it = cid; it < n_citers; it += ncl) {
            for (int l = 0; l < net.n_layers; ++l) {
              const int n1 = net.L[l].n_x_pre, n2 = n1 + net.L[l].n_h, n3 = n2 + net.L[l].n_x_post;
              const int ntot = n3 + net.L[l].bias_mma, npad = (ntot + 1) & ~1;
              const int LN = net.L[l].N;
              const uint32_t bias_lo = x_lo + ((uint32_t)net.L[l].bias_a_off >> 4);
              const uint32_t idesc = tc::make_idesc_bf16(256, LN, 0, 0);
              const uint32_t b_k16 = (uint32_t)LN;                 // 2 * LBO >> 4 : the second 16-wide K half
              const uint32_t b_lo0 = w_lo | ((uint32_t)(LN / 2) << 16);   // LBO = (N/2) * 16 B
              uint32_t g = gl + ph * npad;   // this issuer's first chunk of the layer
              gl += 2 * npad;
              const long long w0 = PCLK();
              mbar_wait_dbg<kProf>(actr, act_phase, a.hang, 3 + ph * 10, (uint32_t)(l + 100 * (int)((it - cid) / ncl)));
              t_act += PCLK() - w0;
              act_phase ^= 1;
              tc::tc_fence_after();
              for (int c = 0; c < npad; c += 2, g += 2) {
                const uint32_t s = g & (kStages2 - 1);
                // mbarrier waits only know the phase PARITY.  The previous use of this ring pair may belong to the
                // other issuer (the first 4 pairs of a layer phase): until that use has been consumed the full
                // barrier still sits in the older phase and a wait for this one would pass spuriously, so make sure
                // of it first (own pairs need no check: this thread saw their phase complete before issuing).
                const long long f0 = PCLK();
                if (c < kStages2 && g >= kStages2)
                  mbar_wait_dbg<kProf>(empty0 + (s >> 1) * 8, ((g - kStages2) / kStages2) & 1, a.hang, 6 + ph * 10,
                                (uint32_t)(l * 1000 + g % 1000));
                mbar_wait_dbg<kProf>(full0 + (s >> 1) * 8, (g / kStages2) & 1, a.hang, 4 + ph * 10, (uint32_t)(l * 1000 + g % 1000));   // both halves landed (peer relays)
                t_full += PCLK() - f0;
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                  const int cc = c + j;
                  const uint32_t a_lo = cc < n1   ? x_lo + cc * kAStep
                                        : cc < n2 ? h_lo + (cc - n1) * kAStep
                                        : cc < n3 ? x_lo + (cc - n2) * kAStep
                                                  : bias_lo;   // 16 channels ending in the constant 1
                  const uint32_t b_lo = b_lo0 + (s + j) * (kStage2Bytes >> 4);
                  if (cc < ntot) tc::mma2_bf16_ss_w(acc, a_lo, kDescHi, b_lo, kDescHi, idesc, cc > 0 ? 1u : 0u);
                  if (cc < n3)
                    tc::mma2_bf16_ss_w(acc, a_lo + (2 * kK8Stride >> 4), kDescHi, b_lo + b_k16, kDescHi, idesc, 1u);
                }
                if (c + 2 >= ntot) tc::mma2_commit_addr(accf);
                tc::mma2_commit_addr(empty0 + (s >> 1) * 8);
              }
            }
          }
        }
        __syncwarp();
        if (kProf && a.prof && lane == 0) {
          unsigned long long* pp = a.prof + blockIdx.x * 16 + (ph ? 0 : 2);
          if (ph == 0) { pp[0] = t_act; pp[1] = t_full; pp[2] = t_peer; pp[7] = t_issue; pp[3] = PCLK() - t_begin; }
          else { pp[0] = t_act; pp[1] = t_full; }
        }
      }
    }
  }
  } else {
    reg_alloc<kEpiRegs>();
    // ============ encode + epilogue warps ============
    const int q = warp & 3;                 // TMEM lane quarter
    const int hi = (warp - 4) >> 2;         // epilogue: column half ; encode: tile (0 = A, 1 = B)
    const int row = q * 32 + lane;
    // head weights: shared memory for the view-direction net, global (L2) for the 4 x 256 output_linear
    const float* hw = net.in_views > 0 ? s_head : a.fparams + net.head_off;
    uint32_t acc_phase[2] = {0, 0};
    float alpha_part[2] = {0.f, 0.f};
    uint8_t* const acts_base = a.acts;
    const int act_tile_bytes = net.act_tile_bytes, dbg = a.debug;
    const int64_t nP = a.P;
    long long t_acc = 0, t_body = 0, t_enc = 0;
    const long long t_begin = PCLK();

    auto arrive_act = [&](int ph) {
      tc::fence_proxy_async_smem();
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (r == 0) tc::mbar_arrive(&ctl->act_ready[ph]);
        else tc::mbar_arrive_remote(&ctl->act_ready[ph], 0);
      }
    };
    auto encode_tile = [&](int64_t it, int te) {   // encode rows of tile `te` for cluster iteration `it`
      const int64_t tile_idx = it * 4 + te * 2 + r;
      const int64_t p = tile_idx * kTileM + row;
      const bool valid = p < a.P;
      uint8_t* rec = a.acts ? a.acts + (size_t)tile_idx * net.act_tile_bytes : nullptr;
      uint8_t* my_x = x_buf + te * kXBytes;
      if (a.mode == 1) {
        float xyz[3] = {0.f, 0.f, 0.f};
        if (valid) {
          const int64_t ry = p / a.S;
          const float zv = a.z[p];
#pragma unroll
          for (int j = 0; j < 3; ++j) xyz[j] = a.rays_o[ry * 3 + j] + a.rays_d[ry * 3 + j] * zv;
        }
        encode_row2<CTX_MLP_XP_PAD, 10>(my_x, row, xyz, a.L_pts, valid, rec ? rec + net.xp_slot : nullptr);
      } else if (a.mode == 2) {
        // UV grid of the texture atlas (reference get_texture_map, src/models/textured_mesh.py:266-272):
        // point p = y*res + x  ->  (u, v) = (linspace(0,1,res)[x], linspace(0,1,res)[y]), encoded in place
        float uv[3] = {0.f, 0.f, 0.f};
        if (valid) {
          const int res = a.S;
          const int py = (int)(p / res), px = (int)(p - (int64_t)py * res);
          uv[0] = linspace_at(0.0f, 1.0f, res, px);
          uv[1] = linspace_at(0.0f, 1.0f, res, py);
        }
        encode_row2<CTX_MLP_XP_PAD, 10, 2>(my_x, row, uv, a.L_pts, valid, rec ? rec + net.xp_slot : nullptr);
      } else if (a.mode == 3) {
        // raw coordinates, e.g. the rasterised UVs of the texels a mesh actually uses
        // (reference get_texture_map_only_valid_areas, src/models/textured_mesh.py:303-347), optionally gathered
        float pt[3] = {0.f, 0.f, 0.f};
        if (valid) {
          const int64_t src = a.gather ? a.gather[p] : p;
          pt[0] = __ldg(a.x + src * a.x_ld);
          pt[1] = __ldg(a.x + src * a.x_ld + 1);
          if (a.x_ld > 2) pt[2] = __ldg(a.x + src * a.x_ld + 2);
        }
        if (a.x_ld == 2) encode_row2<CTX_MLP_XP_PAD, 10, 2>(my_x, row, pt, a.L_pts, valid, rec ? rec + net.xp_slot : nullptr);
        else encode_row2<CTX_MLP_XP_PAD, 10, 3>(my_x, row, pt, a.L_pts, valid, rec ? rec + net.xp_slot : nullptr);
      } else {
        float v[CTX_MLP_XP_PAD];
#pragma unroll
        for (int i = 0; i < CTX_MLP_XP_PAD; ++i) v[i] = (valid && i < net.in_pts) ? __ldg(a.x + p * a.x_ld + i) : 0.f;
        v[CTX_MLP_XP_PAD - 1] = 1.0f;
#pragma unroll
        for (int c0 = 0; c0 < CTX_MLP_XP_PAD; c0 += 8)
          store_row8(my_x, row, c0, v + c0, false, rec ? rec + net.xp_slot : nullptr, CTX_MLP_XP_PAD);
      }
    };

    // prologue: both tiles of the first iteration
    if (cid < n_citers) encode_tile(cid, hi);
    arrive_act(0);
    arrive_act(1);

    for (int64_t it = cid; it < n_citers; it += ncl) {
      for (int l = 0; l < net.n_layers; ++l) {
        const int Lepi = net.L[l].epi, LN = net.L[l].N, Lrelu = net.L[l].relu;
        const int Lmask = net.L[l].mask_slot, Lact = net.L[l].act_slot, Lrec = net.L[l].rec_ch;
        const bool is_final = (Lepi == CTX_EPI_FINAL_VIEWS || Lepi == CTX_EPI_FINAL_OUT);
        const int ncb = LN / 64;            // 32-column blocks handled by this warp (its half of N)
#pragma unroll
        for (int ph = 0; ph < 2; ++ph) {
          const int64_t tile_idx = it * 4 + ph * 2 + r;
          const int64_t p = tile_idx * kTileM + row;
          const bool valid = p < nP;
          uint8_t* rec = acts_base ? acts_base + (size_t)tile_idx * act_tile_bytes : nullptr;
          uint8_t* my_h = h_buf + ph * kHBytes;
          uint8_t* my_x = x_buf + ph * kXBytes;
          const uint32_t my_acc = tmem + ph * CTX_MLP_W + ((uint32_t)(q * 32) << 16);
          const long long e0 = PCLK();
          mbar_wait_dbg<kProf>(tc::smem_u32(&ctl->acc_full[ph]), acc_phase[ph], a.hang, 5 + ph * 10, (uint32_t)(l + 100 * (int)((it - cid) / ncl)));
          const long long e1 = PCLK();
          t_acc += e1 - e0;
          acc_phase[ph] ^= 1;
          tc::tc_fence_after();
          float head[4] = {0.f, 0.f, 0.f, 0.f};
          // The bias is already inside the accumulator (constant-1 channel x bias row of the weight stream),
          // so a hidden-layer epilogue is: TMEM load -> (training: sign mask) -> relu+bf16 pack -> store.
          // One straight-line instantiation per (epilogue kind, relu): the per-block path of a plain hidden
          // layer is TMEM load -> 16 cvt.relu.bf16x2 -> 4 STS.128 (+ mask word and 4 STG.128 when recording).
          auto run = [&](auto epi_c, auto relu_c) {
            constexpr int EPI = decltype(epi_c)::value;
            constexpr bool RELU = decltype(relu_c)::value;
            constexpr bool FINAL = (EPI == CTX_EPI_FINAL_VIEWS || EPI == CTX_EPI_FINAL_OUT);
            uint8_t* const grec = (kRec && Lact >= 0) ? rec + Lact : nullptr;   // (feature layer: no record)
            auto process = [&](const uint32_t (&vr)[32], int cb) {
              if constexpr (kRec && RELU) {
                // bit (31-j) = sign of pre-activation j (the ReLU mask the dgrad kernel reads); four independent
                // shift chains instead of one 32-deep dependent one
                uint32_t n0 = 0, n1 = 0, n2 = 0, n3 = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  n0 = __funnelshift_l(vr[j], n0, 1);
                  n1 = __funnelshift_l(vr[8 + j], n1, 1);
                  n2 = __funnelshift_l(vr[16 + j], n2, 1);
                  n3 = __funnelshift_l(vr[24 + j], n3, 1);
                }
                const uint32_t neg = (n0 << 24) | (n1 << 16) | (n2 << 8) | n3;
                                __stcs(reinterpret_cast<uint32_t*>(rec + Lmask) + cb * kTileM + row, neg);   // [column block][row]: coalesced
              }
              float v[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(vr[j]);
              if constexpr (EPI == CTX_EPI_HIDDEN_ALPHA) {
                float acc = alpha_part[ph];
#pragma unroll
                for (int j = 0; j < 32; ++j) acc = fmaf(bf16_round(fmaxf(v[j], 0.f)), hw[cb * 32 + j], acc);
                alpha_part[ph] = acc;
              } else if constexpr (EPI == CTX_EPI_FINAL_VIEWS) {
                const float* wr = hw + 260;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  const float hv = bf16_round(fmaxf(v[j], 0.f));
                  head[0] = fmaf(hv, wr[cb * 32 + j], head[0]);
                  head[1] = fmaf(hv, wr[128 + cb * 32 + j], head[1]);
                  head[2] = fmaf(hv, wr[256 + cb * 32 + j], head[2]);
                }
              } else if constexpr (EPI == CTX_EPI_FINAL_OUT) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  const float hv = bf16_round(fmaxf(v[j], 0.f));
#pragma unroll
                  for (int o = 0; o < 4; ++o) head[o] = fmaf(hv, hw[o * 256 + cb * 32 + j], head[o]);
                }
              }
              if constexpr (!FINAL || kRec) {
#pragma unroll
                for (int j = 0; j < 32; j += 8)
                  store_row8(FINAL ? nullptr : my_h, row, cb * 32 + j, v + j, RELU, grec, Lrec);
              }
            };
            const int cb0 = hi * ncb;
            // (loads are NOT run ahead of the processing: measured slower in this kernel, before and after the
            //  epilogue warps got 224 registers; the dgrad epilogue does profit from it)
            uint32_t va[32];
            for (int cbi = 0; cbi < ncb; ++cbi) {
              tc::tmem_ld32(my_acc + (cb0 + cbi) * 32, va);
              tc::tmem_wait_ld(va);
              process(va, cb0 + cbi);
            }
          };
          if (!(dbg & 1)) {
            using std::integral_constant;
            switch (Lepi) {
              case CTX_EPI_HIDDEN:
                if (Lrelu) run(integral_constant<int, CTX_EPI_HIDDEN>{}, integral_constant<bool, true>{});
                else run(integral_constant<int, CTX_EPI_HIDDEN>{}, integral_constant<bool, false>{});
                break;
              case CTX_EPI_HIDDEN_ALPHA:
                run(integral_constant<int, CTX_EPI_HIDDEN_ALPHA>{}, integral_constant<bool, true>{});
                break;
              case CTX_EPI_FINAL_VIEWS:
                run(integral_constant<int, CTX_EPI_FINAL_VIEWS>{}, integral_constant<bool, true>{});
                break;
              default:
                run(integral_constant<int, CTX_EPI_FINAL_OUT>{}, integral_constant<bool, true>{});
                break;
            }
          }
          if (Lepi == CTX_EPI_HIDDEN_ALPHA && hi == 0) {
            // the point encoding of this tile is dead: its x buffer now takes the view-direction encoding
            if (a.mode == 1) {
              float dirs[3] = {0.f, 0.f, 0.f};
              if (valid) {
                const int64_t ry = p / a.S;
#pragma unroll
                for (int j = 0; j < 3; ++j) dirs[j] = a.viewdirs[ry * 3 + j];
              }
              encode_row2<CTX_MLP_XD_PAD, 4>(my_x, row, dirs, a.L_dirs, valid, rec ? rec + net.xd_slot : nullptr);
            } else {
              float vv[CTX_MLP_XD_PAD];
#pragma unroll
              for (int i = 0; i < CTX_MLP_XD_PAD; ++i)
                vv[i] = (valid && i < net.in_views) ? __ldg(a.x + p * a.x_ld + net.in_pts + i) : 0.f;
              vv[CTX_MLP_XD_PAD - 1] = 1.0f;
#pragma unroll
              for (int c0 = 0; c0 < CTX_MLP_XD_PAD; c0 += 8)
                store_row8(my_x, row, c0, vv + c0, false, rec ? rec + net.xd_slot : nullptr, CTX_MLP_XD_PAD);
            }
          }
          if (is_final) {
            // the two column halves add their partial head sums into the zero-initialised output
            if (valid) {
              if (Lepi == CTX_EPI_FINAL_VIEWS) {
                const float* br = hw + 260 + 384;
                float* o4 = a.out + p * 4;
                atomicAdd(o4 + 0, head[0] + (hi == 0 ? br[0] : 0.f));
                atomicAdd(o4 + 1, head[1] + (hi == 0 ? br[1] : 0.f));
                atomicAdd(o4 + 2, head[2] + (hi == 0 ? br[2] : 0.f));
                atomicAdd(o4 + 3, alpha_part[ph] + (hi == 0 ? hw[256] : 0.f));
              } else {
                const float* bo = hw + 1024;
#pragma unroll
                for (int o = 0; o < 4; ++o)
                  if (o < net.out_ch) atomicAdd(a.out + p * net.out_ch + o, head[o] + (hi == 0 ? bo[o] : 0.f));
              }
            }
            alpha_part[ph] = 0.f;
            // next iteration's point encoding of this tile can start as soon as its last MMAs are done
            const int64_t nit = it + ncl;
            const long long e2 = PCLK();
            if (nit < n_citers && hi == ph) encode_tile(nit, ph);
            t_enc += PCLK() - e2;
            if (nit < n_citers) arrive_act(ph);
          } else {
            arrive_act(ph);
          }
          t_body += PCLK() - e1;
        }
      }
    }
    if (kProf && a.prof && lane == 0 && (warp == 2 || warp == 9)) {
      unsigned long long* pp = a.prof + blockIdx.x * 16 + (warp == 2 ? 6 : 10);
      pp[0] = t_acc; pp[1] = t_body; pp[2] = PCLK() - t_begin;
      if (warp == 2) a.prof[blockIdx.x * 16 + 13] = t_enc;
    }
  }

  tc::tc_fence_before();
  tc::cluster_sync_all();
  if (warp == 1) {
    __syncwarp();
    tc::tmem_dealloc2(tmem, 512);
  }
#undef PCLK
}

}  // namespace ctx

// Diagnostics live in libctxnerf_diag.so only (built with -DCTXNERF_DIAG, include/ctxnerf_diag.h): if set (device
// pointer, 16 x uint64 per CTA), the profiling instantiation of the kernel records where its roles wait.  The product
// library carries neither the hooks nor the profiling kernels.
#ifdef CTXNERF_DIAG
static void* ctx_mlp_prof_buffer = nullptr;
static int ctx_mlp_debug_flags = 0;
static void* ctx_mlp_hang_buffer = nullptr;
extern "C" int ctx_mlp_set_hang_buffer(void* p) { ctx_mlp_hang_buffer = p; return 0; }
extern "C" int ctx_mlp_set_debug(int f) { ctx_mlp_debug_flags = f; return 0; }
extern "C" int ctx_mlp_set_prof_buffer(void* p) { ctx_mlp_prof_buffer = p; return 0; }
#else
static void* const ctx_mlp_prof_buffer = nullptr;
static const int ctx_mlp_debug_flags = 0;
static void* const ctx_mlp_hang_buffer = nullptr;
#endif

extern "C" int ctx_mlp_fwd_ex(const void* net_host, const void* wpacked, const float* fparams, int mode,
                               const float* x, int x_ld, const float* rays_o, const float* rays_d,
                               const float* viewdirs, const float* z, int S, int L_pts, int L_dirs, int64_t P,
                               float* out, void* acts, const int64_t* gather, int max_sms, void* stream) {
  if (P < 0) return CTX_ERR_BAD_ARG;
  if (P == 0) return 0;                       // empty batch: nothing to launch (its pointers may be null)
  if (!net_host || !wpacked || !fparams || !out) return CTX_ERR_BAD_ARG;
  ctx::MlpFwdArgs a;
  a.net = *reinterpret_cast<const CtxMlpNet*>(net_host);
  if (mode == 0) {
    if (!x || x_ld < a.net.in_pts + a.net.in_views) return CTX_ERR_BAD_ARG;
  } else if (mode == 1) {
    if (!rays_o || !rays_d || !z || S < 1 || (a.net.in_views > 0 && !viewdirs)) return CTX_ERR_BAD_ARG;
    if (a.net.in_pts != 3 * (1 + 2 * L_pts) || L_pts > 10) return CTX_ERR_UNSUPPORTED;
    if (a.net.in_views > 0 && (a.net.in_views != 3 * (1 + 2 * L_dirs) || L_dirs > 4)) return CTX_ERR_UNSUPPORTED;
  } else if (mode == 2) {
    if (S < 2 || (int64_t)S * S != P || a.net.in_views != 0) return CTX_ERR_BAD_ARG;
    if (a.net.in_pts != 2 * (1 + 2 * L_pts) || L_pts > 10) return CTX_ERR_UNSUPPORTED;
  } else if (mode == 3) {
    if (!x || (x_ld != 2 && x_ld != 3) || a.net.in_views != 0) return CTX_ERR_BAD_ARG;
    if (a.net.in_pts != x_ld * (1 + 2 * L_pts) || L_pts > 10) return CTX_ERR_UNSUPPORTED;
  } else {
    return CTX_ERR_BAD_ARG;
  }
  a.gather = (const long long*)gather;
  a.wpacked = (const uint8_t*)wpacked; a.fparams = fparams; a.mode = mode; a.x = x; a.x_ld = x_ld;
  a.rays_o = rays_o; a.rays_d = rays_d; a.viewdirs = viewdirs; a.z = z; a.S = S; a.L_pts = L_pts;
  a.L_dirs = L_dirs; a.P = P; a.out = out; a.acts = (uint8_t*)acts;
  a.prof = (unsigned long long*)ctx_mlp_prof_buffer; a.debug = ctx_mlp_debug_flags;
  a.hang = (unsigned long long*)ctx_mlp_hang_buffer;
  cudaStream_t st = (cudaStream_t)stream;
  using KernelFn = void (*)(ctx::MlpFwdArgs);
#ifdef CTXNERF_DIAG
  static const KernelFn kernels[4] = {ctx::mlp_fwd_kernel<false, false>, ctx::mlp_fwd_kernel<false, true>,
                                      ctx::mlp_fwd_kernel<true, false>, ctx::mlp_fwd_kernel<true, true>};
#else
  static const KernelFn kernels[2] = {ctx::mlp_fwd_kernel<false, false>, ctx::mlp_fwd_kernel<false, true>};
#endif
  static ctx::DeviceOnce attr_once;
  if (attr_once.needed()) {
    for (KernelFn k : kernels) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx::kMlp2SmemBytes);
      if (e != cudaSuccess) return (int)e;
    }
  }
  cudaError_t e = cudaMemsetAsync(out, 0, (size_t)P * a.net.out_ch * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  const int64_t citers = ctx::ceil_div(P, (int64_t)ctx::kTileM * 4);
  int cap = ctx::num_sms() / 2;   // one cluster per SM pair; a smaller SM budget leaves room for a concurrent kernel
  if (max_sms > 0 && max_sms / 2 < cap) cap = max_sms / 2;
  if (cap < 1) cap = 1;
  const int ncl = (int)(citers < cap ? citers : cap);
  kernels[(a.prof ? 2 : 0) + (a.acts ? 1 : 0)]<<<2 * ncl, ctx::kMlpThreads, ctx::kMlp2SmemBytes, st>>>(a);
  CTX_RETURN_LAST();
}

extern "C" int ctx_mlp_fwd(const void* net_host, const void* wpacked, const float* fparams, int mode,
                            const float* x, int x_ld, const float* rays_o, const float* rays_d,
                            const float* viewdirs, const float* z, int S, int L_pts, int L_dirs, int64_t P,
                            float* out, void* acts, void* stream) {
  return ctx_mlp_fwd_ex(net_host, wpacked, fparams, mode, x, x_ld, rays_o, rays_d, viewdirs, z, S, L_pts, L_dirs, P,
                        out, acts, nullptr, 0, stream);
}
