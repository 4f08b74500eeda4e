// dgrad of the coordinate MLP on tcgen05 / TMEM: 2-CTA MMAs (cta_group::2) + ping-pong.
//
// Same machinery as mlp_fwd.cu run backwards: a cluster of two CTAs owns 512
// points per iteration as two 256-row tile pairs; for every step (layer l, last
// to first) dH = dZ_l * W_l is one chain of M=256 MMAs over the half-split
// transposed weight stream, and the epilogue of one tile pair (ReLU sign mask
// from the forward's bit record, alpha-head term, bf16 pack, store to shared
// memory as the next A operand and to the dZ record for wgrad) runs under the
// MMAs of the other pair.  The heads (rgb / alpha / output_linear) are
// differentiated on the CUDA cores when a tile is (re)initialised.
//
// Reference semantics: autograd through NeRF2D.forward,
// /root/reference/src/run_nerf_helpers.py:106-135.
#include "mlp_common.cuh"
#include <stdlib.h>
#include <string.h>

#ifdef CTXNERF_DIAG     // diagnostics build (include/ctxnerf_diag.h): per-role cycle counters, 16 x uint64 per CTA
static unsigned long long* g_dg_prof = nullptr;
extern "C" int ctx_dgrad_set_prof(void* p) { g_dg_prof = (unsigned long long*)p; return 0; }
#define DGCLK() clock64()
#else
#define DGCLK() 0ll
#endif

namespace ctx {

constexpr int kDgStages = 8;
constexpr int kDgPairs = kDgStages / 2;
constexpr int kDgStageBytes = 8192;          // 128 in-feature rows x 32 K x 2 B
constexpr int kDgHeadFloats = 1028;

struct DgradArgs {
  CtxMlpNet net;
  const uint8_t* wtstream;   // half-split transposed stream
  const float* fparams;
  const float* g_out;        // [P, out_ch]
  const uint8_t* acts;       // forward records (ReLU masks)
  uint8_t* dacts;            // dZ records
  int64_t P;
  int n_steps;
  int step_src[CTX_MLP_MAX_LAYERS];
  int step_dst[CTX_MLP_MAX_LAYERS];
  unsigned long long* prof;  // diagnostics build only
  int use_tma;               // dZ tiles of the inner steps leave through one tensor-map TMA store per tile-layer
  CUtensorMap tmap;          // over the dZ record buffer (mlp_common.cuh: make_record_tensor_map)
};

struct __align__(8) DgSmemCtl {
  uint64_t full[kDgPairs], empty[kDgPairs];
  uint64_t acc_full[kTiles], act_ready[kTiles];
  uint64_t rec_ready[kTiles], rec_free[kTiles];   // epilogue -> store warp: tile written ; store warp -> epilogue: read
  uint32_t tmem_base;
};
// two 64 KB dZ tiles + weight ring + head weights (fp32) + barriers
constexpr size_t kDgSmemBytes = (size_t)kTiles * kHBytes + (size_t)kDgStages * kDgStageBytes + kDgHeadFloats * 4 + 256;

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kMlpThreads, 1)
mlp_dgrad_kernel(const __grid_constant__ DgradArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* h_buf = smem;
  uint8_t* w_buf = smem + kTiles * kHBytes;
  float* s_head = reinterpret_cast<float*>(w_buf + kDgStages * kDgStageBytes);
  DgSmemCtl* ctl = reinterpret_cast<DgSmemCtl*>(s_head + kDgHeadFloats);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t r = tc::cluster_ctarank();
  const CtxMlpNet& net = a.net;
  const int64_t n_citers = ceil_div(a.P, (int64_t)kTileM * 4);
  const int64_t cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;
  const int n_steps = a.n_steps;

  if (tid == 0) {
    for (int s = 0; s < kDgPairs; ++s) {
      // full: the leader also counts the peer's relay; empty: BOTH issuers release a ring pair (the two tile pairs
      // read the same weights: one stream per step serves both)
      tc::mbar_init(&ctl->full[s], r == 0 ? 2 : 1); tc::mbar_init(&ctl->empty[s], 2);
    }
    for (int t = 0; t < kTiles; ++t) {
      tc::mbar_init(&ctl->acc_full[t], 1); tc::mbar_init(&ctl->act_ready[t], 16);
      tc::mbar_init(&ctl->rec_ready[t], 8); tc::mbar_init(&ctl->rec_free[t], 1);
    }
    tc::mbar_fence_init();
  }
  if (warp == 1) tc::tmem_alloc2(&ctl->tmem_base, 512);
  {
    const int nhead = net.in_views > 0 ? 648 : 1028;
    for (int i = tid; i < nhead; i += kMlpThreads) s_head[i] = a.fparams[net.head_off + i];
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
    // ============ transposed-weight producer: this CTA's half of every chunk, ONCE per step ============
    // Both tile pairs consume the same ring pair (issuer A and issuer B each wait on `full` and each commit to
    // `empty`), so the ring holds a whole step's weights and the next step's chunks are requested while the second
    // tile pair is still running this step's MMAs: the L2 latency of the weight stream hides behind them instead
    // of opening a bubble at every phase change, and the stream's L2 traffic is halved.
    uint32_t g = 0;
    for (int64_t it = cid; it < n_citers; it += ncl) {
      for (int si = 0; si < n_steps; ++si) {
        const int src = a.step_src[si];
        const int nchunks = net.L[src].N / CTX_MLP_KC;
        const uint8_t* lsrc = a.wtstream + net.L[src].wt_off + r * kDgStageBytes;
        for (int c = 0; c < nchunks; ++c, ++g) {
          const int s = g % kDgStages, pr = s >> 1;
          if (!(g & 1)) tc::mbar_wait(&ctl->empty[pr], ((g / kDgStages) & 1) ^ 1);
          if (tc::elect_one()) {
            tc::mbar_expect_tx(&ctl->full[pr], kDgStageBytes);
            tc::bulk_g2s(w_buf + s * kDgStageBytes, lsrc + (size_t)c * 2 * kDgStageBytes, kDgStageBytes, &ctl->full[pr]);
            if (g & 1) tc::mbar_arrive(&ctl->full[pr]);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    if (r != 0) {
      if (warp == 1) {
      // ============ peer CTA: relay "my half landed" to the leader, once per chunk pair ============
      uint32_t g = 0;
      for (int64_t it = cid; it < n_citers; it += ncl)
        for (int si = 0; si < n_steps; ++si) {
          const int nchunks = net.L[a.step_src[si]].N / CTX_MLP_KC;
          for (int c = 0; c < nchunks; ++c, ++g) {
            if (g & 1) {
              const int pr = (g % kDgStages) >> 1;
              tc::mbar_wait(&ctl->full[pr], (g / kDgStages) & 1);
              if (tc::elect_one()) tc::mbar_arrive_remote(&ctl->full[pr], 0);
              __syncwarp();
            }
          }
        }
      }
    } else {
      // ============ leader CTA: two MMA issuers, warp 1 -> tile pair A, warp 2 -> tile pair B ============
      // (one thread cannot issue fast enough to keep the tensor pipe fed; see mlp_fwd.cu)
      const int ph = warp == 1 ? 0 : 1;
      if (tc::elect_one()) {
        // single issuing thread, descriptor lo words advanced by adds, one barrier wait + one commit per ring
        // pair (4 MMAs) -- see mlp_fwd.cu
        constexpr uint32_t kDescHi = (128u >> 4) | (1u << 14);
        constexpr uint32_t kALbo = (uint32_t)(kK8Stride >> 4) << 16, kBLbo = (2048u >> 4) << 16;
        constexpr uint32_t kAStep = 4 * kK8Stride >> 4;
        const uint32_t idesc = tc::make_idesc_bf16(256, 256, 0, 0);
        const uint32_t h_lo = kALbo | (tc::smem_u32(h_buf + ph * kHBytes) >> 4);
        const uint32_t w_lo = kBLbo | (tc::smem_u32(w_buf) >> 4);
        const uint32_t full0 = tc::smem_u32(&ctl->full[0]), empty0 = tc::smem_u32(&ctl->empty[0]);
        const uint32_t accf = tc::smem_u32(&ctl->acc_full[ph]), actr = tc::smem_u32(&ctl->act_ready[ph]);
        const uint32_t acc = tmem + ph * CTX_MLP_W;
        uint32_t gl = 0, act_phase = 0;
        long long t_act = 0, t_full = 0; const long long t_beg = DGCLK();
        for (int64_t it = cid; it < n_citers; it += ncl) {
          for (int si = 0; si < n_steps; ++si) {
            const int nchunks = net.L[a.step_src[si]].N / CTX_MLP_KC;   // 4 or 8: phases are whole chunk pairs
            uint32_t g = gl;             // both issuers walk the same chunk sequence (shared ring)
            gl += nchunks;
            const long long w0 = DGCLK();
            tc::mbar_wait_addr(actr, act_phase);
            t_act += DGCLK() - w0;
            act_phase ^= 1;
            tc::tc_fence_after();
            for (int c = 0; c < nchunks; c += 2, g += 2) {
              const uint32_t s = g & (kDgStages - 1);
              // every issuer sees every use of every ring pair, in order: a parity wait cannot alias an older phase
              const long long f0 = DGCLK();
              tc::mbar_wait_addr(full0 + (s >> 1) * 8, (g / kDgStages) & 1);   // both halves landed
              t_full += DGCLK() - f0;
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const uint32_t a_lo = h_lo + (c + j) * kAStep;
                const uint32_t b_lo = w_lo + (s + j) * (kDgStageBytes >> 4);
                tc::mma2_bf16_ss_w(acc, a_lo, kDescHi, b_lo, kDescHi, idesc, (c + j) > 0 ? 1u : 0u);
                tc::mma2_bf16_ss_w(acc, a_lo + (2 * kK8Stride >> 4), kDescHi, b_lo + (2 * 2048 >> 4), kDescHi, idesc,
                                   1u);
              }
              if (c + 2 >= nchunks) tc::mma2_commit_addr(accf);
              tc::mma2_commit_addr(empty0 + (s >> 1) * 8);
            }
          }
        }
#ifdef CTXNERF_DIAG
        if (a.prof) { unsigned long long* pp = a.prof + blockIdx.x * 16 + ph * 3; pp[0] = t_act; pp[1] = t_full; pp[2] = DGCLK() - t_beg; }
#endif
      }
      __syncwarp();
    }
  } else if (warp == 3 && a.use_tma) {
    // ============ record-store warp: one TMA tensor store per finished dZ tile of the inner steps ============
    // The epilogue leaves the tile in shared memory anyway (it is the next step's A operand); this warp ships the
    // same bytes to the dZ record with ONE instruction, so the epilogue warps issue no global stores for it.
    uint32_t n_st = 0;                      // stores issued per tile buffer (both buffers advance together)
    long long t_rdy = 0, t_rd = 0;
    for (int64_t it = cid; it < n_citers; it += ncl) {
      for (int si = 0; si + 1 < n_steps; ++si) {
        const int Dact = net.L[a.step_dst[si]].act_slot;
        if (Dact < 0) continue;
#pragma unroll
        for (int ph = 0; ph < 2; ++ph) {
          const long long s0 = DGCLK();
          tc::mbar_wait(&ctl->rec_ready[ph], n_st & 1);
          const long long s1 = DGCLK();
          if (tc::elect_one()) {
            tc::tma_store_4d(&a.tmap, h_buf + ph * kHBytes, 0, 0, Dact >> 10, (int)(it * 4 + ph * 2 + r));
            tc::bulk_commit();
            tc::bulk_wait_read<0>();          // the tile may be overwritten once the copy has read it
            tc::mbar_arrive(&ctl->rec_free[ph]);
          }
          __syncwarp();
          t_rdy += s1 - s0; t_rd += DGCLK() - s1;
        }
        ++n_st;
      }
    }
    if (tc::elect_one()) tc::bulk_wait<0>();
    __syncwarp();
#ifdef CTXNERF_DIAG
    if (a.prof && lane == 0) { a.prof[blockIdx.x * 16 + 6] = t_rdy; a.prof[blockIdx.x * 16 + 7] = t_rd; }
#endif
  }
  } else {
    reg_alloc<kEpiRegs>();
    // ============ head-init + epilogue warps ============
    const int q = warp & 3;                 // TMEM lane quarter
    const int hi = (warp - 4) >> 2;         // epilogue: column half ; head init: tile (0 = A, 1 = B)
    const int row = q * 32 + lane;
    const float* hw = s_head;
    const bool has_views = net.in_views > 0;
    const int out_ch = net.out_ch, act_tile_bytes = net.act_tile_bytes, gout_slot = net.gout_slot;
    const int last = net.n_layers - 1;
    const int lastN = net.L[last].N, last_mask = net.L[last].mask_slot, last_act = net.L[last].act_slot;
    const int last_rec = net.L[last].rec_ch, gout_ch0 = net.gout_ch0, gout_rec = net.gout_rec_ch;
    const int64_t nP = a.P;
    const bool use_tma = a.use_tma != 0;
    uint32_t acc_phase[2] = {0, 0};
    uint32_t n_st0 = 0, n_st1 = 0;          // TMA stores issued so far from each tile buffer
    long long t_acc = 0, t_free = 0, t_body = 0, t_head = 0; const long long t_beg = DGCLK();

    auto arrive_act = [&](int ph, bool rec = false) {
      tc::fence_proxy_async_smem();
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rec) tc::mbar_arrive(&ctl->rec_ready[ph]);
        if (r == 0) tc::mbar_arrive(&ctl->act_ready[ph]);
        else tc::mbar_arrive_remote(&ctl->act_ready[ph], 0);
      }
    };
    // before (re)writing a tile buffer: the last TMA store issued from it must have finished reading it
    auto wait_tile_free = [&](int ph) {
      const uint32_t n = ph ? n_st1 : n_st0;
      if (n > 0) tc::mbar_wait(&ctl->rec_free[ph], (n - 1) & 1);
    };
    // dZ of the last GEMM layer from g_out (through the rgb / output head and that layer's ReLU mask)
    auto head_init = [&](int64_t it, int te) {
      const int64_t tile_idx = it * 4 + te * 2 + r;
      const int64_t p = tile_idx * kTileM + row;
      const bool valid = p < nP;
      const uint8_t* rec = a.acts + (size_t)tile_idx * act_tile_bytes;
      uint8_t* drec = a.dacts + (size_t)tile_idx * act_tile_bytes;
      uint8_t* my_h = h_buf + te * kHBytes;
      wait_tile_free(te);
      float g[4] = {0.f, 0.f, 0.f, 0.f};
      if (valid) {
        if (out_ch == 4) {
          const float4 g4 = *reinterpret_cast<const float4*>(a.g_out + p * 4);
          g[0] = g4.x; g[1] = g4.y; g[2] = g4.z; g[3] = g4.w;
        } else {
#pragma unroll
          for (int o = 0; o < 3; ++o) if (o < out_ch) g[o] = a.g_out[p * out_ch + o];
        }
      }
      if (hi == 0) {
        float gv[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) gv[i] = i < 4 ? g[i] : 0.f;
        store_row8(nullptr, row, gout_ch0, gv, false, drec + gout_slot, gout_rec);
        store_row8(nullptr, row, gout_ch0 + 8, gv + 8, false, drec + gout_slot, gout_rec);
      }
      // every epilogue warp builds ITS column half of the tile (hi = half), so the head costs half as much on the
      // critical path of the tile; the ReLU mask words are fetched up front (each is a ~1 us global load)
      const int nwh = lastN / 64;                    // 32-column blocks per half: 2 (views layer) or 4
      const uint32_t* mrow = reinterpret_cast<const uint32_t*>(rec + last_mask) + row;   // [column block][row]
      uint32_t negs[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) negs[i] = i < nwh ? __ldcs(mrow + (hi * nwh + i) * kTileM) : 0u;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (i < nwh) {
          const int cb = hi * nwh + i;
          const uint32_t neg = negs[i];
          float v[32];
          if (has_views) {
            const float* wr = hw + 260;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int c = cb * 32 + j;
              v[j] = g[0] * wr[c] + g[1] * wr[128 + c] + g[2] * wr[256 + c];
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int c = cb * 32 + j;
              v[j] = g[0] * hw[c] + g[1] * hw[256 + c] + g[2] * hw[512 + c] + g[3] * hw[768 + c];
            }
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = ((neg >> (31 - j)) & 1u) ? 0.f : v[j];
#pragma unroll
          for (int j = 0; j < 32; j += 8) store_row8(my_h, row, cb * 32 + j, v + j, false, drec + last_act, last_rec);
        }
      }
    };

    if (cid < n_citers) { head_init(cid, 0); head_init(cid, 1); }
    arrive_act(0);
    arrive_act(1);

    for (int64_t it = cid; it < n_citers; it += ncl) {
      for (int si = 0; si < n_steps; ++si) {
        const int dst = a.step_dst[si];
        const int Drelu = net.L[dst].relu, Dmask = net.L[dst].mask_slot, Dact = net.L[dst].act_slot;
        const bool add_alpha = net.L[dst].epi == CTX_EPI_HIDDEN_ALPHA;
        const bool has_next = si + 1 < n_steps;
#pragma unroll 1
        for (int ph = 0; ph < 2; ++ph) {
          const int64_t tile_idx = it * 4 + ph * 2 + r;
          const int64_t p = tile_idx * kTileM + row;
          const uint8_t* rec = a.acts + (size_t)tile_idx * act_tile_bytes;
          uint8_t* drec = a.dacts + (size_t)tile_idx * act_tile_bytes;
          uint8_t* my_h = h_buf + ph * kHBytes;
          const uint32_t my_acc = tmem + ph * CTX_MLP_W + ((uint32_t)(q * 32) << 16) + hi * 128;
          // this warp's 128 columns: 4 mask words, fetched while the MMAs run
          uint4 mw = make_uint4(0u, 0u, 0u, 0u);
          if (Drelu) {
            const uint32_t* mp = reinterpret_cast<const uint32_t*>(rec + Dmask) + hi * 4 * kTileM + row;
            mw = make_uint4(__ldcs(mp), __ldcs(mp + kTileM), __ldcs(mp + 2 * kTileM), __ldcs(mp + 3 * kTileM));
          }
          float d_alpha = 0.f;
          if (add_alpha && p < nP) d_alpha = __ldg(a.g_out + p * 4 + 3);
          const uint32_t par = ph ? acc_phase[1] : acc_phase[0];
          const long long e0 = DGCLK();
          tc::mbar_wait(&ctl->acc_full[ph], par);
          const long long e1 = DGCLK();
          t_acc += e1 - e0;
          if (ph) acc_phase[1] ^= 1; else acc_phase[0] ^= 1;
          tc::tc_fence_after();
          // straight-line instantiations (alpha-head term / last step)
          const bool tma_rec = use_tma && has_next && Dact >= 0;   // this tile-layer leaves through the store warp
          uint8_t* const grec = (tma_rec || Dact < 0) ? nullptr : drec + Dact;
          if (has_next) wait_tile_free(ph);
          const long long e2 = DGCLK();
          t_free += e2 - e1;
          auto run = [&](auto alpha_c, auto next_c) {
            constexpr bool ALPHA = decltype(alpha_c)::value, NEXT = decltype(next_c)::value;
            auto process = [&](const uint32_t (&vr)[32], int cbi) {
              const uint32_t neg = cbi == 0 ? mw.x : cbi == 1 ? mw.y : cbi == 2 ? mw.z : mw.w;
              const int cb = hi * 4 + cbi;
              float v[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                float x = __uint_as_float(vr[j]);
                if constexpr (ALPHA) x = fmaf(d_alpha, hw[cb * 32 + j], x);
                v[j] = ((neg >> (31 - j)) & 1u) ? 0.f : x;
              }
#pragma unroll
              for (int j = 0; j < 32; j += 8)
                store_row8(NEXT ? my_h : nullptr, row, cb * 32 + j, v + j, false, grec, 256);
            };
            // the load of block c+1 is in flight while block c is processed (two register buffers; affordable since
            // the epilogue warps own 224 registers)
            uint32_t va[32], vb[32];
            tc::tmem_ld32(my_acc, va);
            tc::tmem_wait_ld(va);
            tc::tmem_ld32(my_acc + 32, vb);
            process(va, 0);
            tc::tmem_wait_ld(vb);
            tc::tmem_ld32(my_acc + 64, va);
            process(vb, 1);
            tc::tmem_wait_ld(va);
            tc::tmem_ld32(my_acc + 96, vb);
            process(va, 2);
            tc::tmem_wait_ld(vb);
            process(vb, 3);
          };
          {
            using std::integral_constant;
            if (add_alpha) {
              if (has_next) run(integral_constant<bool, true>{}, integral_constant<bool, true>{});
              else run(integral_constant<bool, true>{}, integral_constant<bool, false>{});
            } else {
              if (has_next) run(integral_constant<bool, false>{}, integral_constant<bool, true>{});
              else run(integral_constant<bool, false>{}, integral_constant<bool, false>{});
            }
          }
          const long long e3 = DGCLK();
          t_body += e3 - e2;
          if (has_next) {
            arrive_act(ph, tma_rec);
            if (tma_rec) { if (ph) ++n_st1; else ++n_st0; }
          } else {
            // the tile is finished: start the next iteration's head for it as soon as possible
            const int64_t nit = it + ncl;
            if (nit < n_citers) head_init(nit, ph);
            if (nit < n_citers) arrive_act(ph);
            t_head += DGCLK() - e3;
          }
        }
      }
    }
#ifdef CTXNERF_DIAG
    if (a.prof && lane == 0 && (warp == 4 || warp == 11)) {
      unsigned long long* pp = a.prof + blockIdx.x * 16 + (warp == 4 ? 8 : 12);
      pp[0] = t_acc; pp[1] = t_free; pp[2] = t_body; pp[3] = warp == 4 ? (unsigned long long)(DGCLK() - t_beg) : (unsigned long long)t_head;
    }
#endif
  }

  tc::tc_fence_before();
  tc::cluster_sync_all();
  if (warp == 1) {
    __syncwarp();
    tc::tmem_dealloc2(tmem, 512);
  }
}

}  // namespace ctx

// host launcher used by ctx_mlp_bwd (mlp_wgrad.cu)
int ctx_launch_dgrad(const CtxMlpNet& net, const void* wtpacked, const float* fparams, const float* g_out,
                      const void* acts, void* dacts, int64_t P, int max_sms, cudaStream_t st) {
  ctx::DgradArgs a;
  a.net = net;
  a.wtstream = (const uint8_t*)wtpacked;
  a.fparams = fparams; a.g_out = g_out; a.acts = (const uint8_t*)acts; a.dacts = (uint8_t*)dacts; a.P = P;
  int n = 0;
  for (int l = net.n_layers - 1; l >= 1; --l) { a.step_src[n] = l; a.step_dst[n] = l - 1; ++n; }
  a.n_steps = n;
  {
    // dZ tiles of the inner steps go out by TMA tensor stores (CTXNERF_DGRAD_TMA=0: register stores, the fallback
    // when the driver cannot encode the map)
    static const bool want = [] { const char* e = getenv("CTXNERF_DGRAD_TMA"); return !(e && e[0] == '0'); }();
    const int64_t n_tiles = 4 * ctx::ceil_div(P, (int64_t)ctx::kTileM * 4);
#ifdef CTXNERF_DIAG
    a.prof = g_dg_prof;
#else
    a.prof = nullptr;
#endif
    a.use_tma = want && ctx::make_record_tensor_map(&a.tmap, dacts, net.act_tile_bytes, n_tiles) == 0;
    if (!a.use_tma) memset(&a.tmap, 0, sizeof(a.tmap));
  }
  static ctx::DeviceOnce attr_once;
  if (attr_once.needed()) {
    cudaError_t e = cudaFuncSetAttribute(ctx::mlp_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)ctx::kDgSmemBytes);
    if (e != cudaSuccess) return (int)e;
  }
  const int64_t citers = ctx::ceil_div(P, (int64_t)ctx::kTileM * 4);
  int cap = ctx::num_sms() / 2;   // one cluster per SM pair; a smaller SM budget leaves room for a concurrent kernel
  if (max_sms > 0 && max_sms / 2 < cap) cap = max_sms / 2;
  if (cap < 1) cap = 1;
  const int ncl = (int)(citers < cap ? citers : cap);
  ctx::mlp_dgrad_kernel<<<2 * ncl, ctx::kMlpThreads, ctx::kDgSmemBytes, st>>>(a);
  return (int)cudaGetLastError();
}
