// Shared device-side pieces of the tcgen05 MLP kernels (forward, dgrad, wgrad):
// tile geometry, shared-memory control block, bf16 packing and the A-operand
// row store in the canonical no-swizzle K-major layout (tc_common.cuh).
#pragma once
#include "ctx_common.cuh"
#include "tc_common.cuh"
#include "mlp_desc.h"

#include <cuda.h>     // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint, no -lcuda)

namespace ctx {

// Tensor map over a record buffer for the dgrad epilogue's tile stores: a [128 points x 256 channels] bf16 tile sits in
// shared memory as [k8 = 32][half = 2][64 rows x 16 B] (the K-major A-operand image) and in the record as two
// 64-point halves of [k8][64 rows x 16 B]; with 8-byte elements that is the 4-D box {128, 2, 32, 1} of the tensor
//   dim0: 128 x u64 (1 KB, contiguous) | dim1: half, stride 32 KB | dim2: 1 KB units of a tile's record, stride 1 KB
//   | dim3: tile, stride tile_bytes
// so ONE cp.async.bulk.tensor moves a whole tile-layer (64 KB) into both halves of a 256-channel slot
// (coordinates {0, 0, slot_offset / 1024, tile}).  Returns 0 on success.
int make_record_tensor_map(CUtensorMap* out, void* base, int tile_bytes, int64_t n_tiles);


constexpr int kTileM = 128;
constexpr int kTiles = 2;
constexpr int kStageBytes = CTX_MLP_W * CTX_MLP_KC * 2;   // 16 KB
constexpr int kHBytes = kTileM * CTX_MLP_W * 2;            // 64 KB
constexpr int kXBytes = kTileM * CTX_MLP_XP_PAD * 2;       // 16 KB
constexpr int kK8Stride = kTileM * 16;                     // 2048 B between 8-wide K chunks of an A tile
// Three warpgroups: warpgroup 0 = control (warp 0 weight producer, warp 1 MMA issuer of tile pair A / peer relay,
// warp 2 MMA issuer of tile pair B, warp 3 idle), warpgroups 1-2 = the eight epilogue warps.  The roles are
// warpgroup-aligned so that setmaxnreg can move registers from the control warps (a handful of live values) to the
// epilogue warps, whose 32-column blocks + record addresses otherwise spill at the 168 registers a 12-warp CTA gets.
constexpr int kMlpThreads = 384;
constexpr int kCtlRegs = 56, kEpiRegs = 224;     // per scheduler: (56 + 2 x 224) x 32 = 16 128 <= 16 384 registers

template <int N> __device__ __forceinline__ void reg_dealloc() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N> __device__ __forceinline__ void reg_alloc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
constexpr int kEpiThreadsPerTile = 128;

struct MlpFwdArgs {
  CtxMlpNet net;
  const uint8_t* wpacked;
  const float* fparams;
  // input
  int mode;                 // 0: pre-encoded x [P, x_ld] fp32, 1: rays + z (encode in-kernel), 2: UV grid generated
                            // in-kernel, 3: raw points x [*, x_ld = 2|3] (optionally gathered), encoded in-kernel
  const long long* gather;  // mode 3, nullable: point p reads row gather[p] of x
  const float* x; int x_ld;
  const float* rays_o; const float* rays_d; const float* viewdirs; const float* z;
  int S; int L_pts; int L_dirs;
  int64_t P;
  float* out;               // [P, out_ch]
  uint8_t* acts;            // nullable: per-tile activation records (training)
  unsigned long long* prof; // nullable: per-CTA cycle counters (diagnostics), 16 per CTA
  unsigned long long* hang; // nullable: host-visible buffer for the deadlock reporter (diagnostics)
  int debug;                // diagnostics: 1 = epilogue skips TMEM loads/stores, 2 = issuer skips the MMAs
};


__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// sin/cos of a (possibly large) fp32 angle, good to ~2e-4 abs: enough for a bf16 operand
__device__ __forceinline__ void fast_sincos(float a, float& s, float& c) {
  float t = a * 0.15915494309189535f;
  t -= rintf(t);
  const float r = t * 6.283185307179586f;
  s = __sinf(r);
  c = __cosf(r);
}

// write 8 consecutive channels [ch0, ch0+8) of row `row` of a K-major A tile; `gtile` (nullable) is the
// record of the same tile in HBM (activation / dZ record, `gC` channels wide): the 16-byte row chunk is
// mirrored there straight from registers (a warp covers 512 contiguous bytes), so saving activations needs
// no extra pass over shared memory.  Record layout: two 64-point halves, each [gC/8][64 points][8 channels]
// -- a half is one contiguous bulk-TMA unit of the wgrad kernel (MN-major operand, K = points).
__device__ __forceinline__ void store_row8(uint8_t* tile, int row, int ch0, const float* v, bool relu,
                                           uint8_t* gtile = nullptr, int gC = 0) {
  uint4 q;
  if (relu) {
    q.x = pack_bf16x2_relu(v[0], v[1]); q.y = pack_bf16x2_relu(v[2], v[3]);
    q.z = pack_bf16x2_relu(v[4], v[5]); q.w = pack_bf16x2_relu(v[6], v[7]);
  } else {
    q.x = pack_bf16x2(v[0], v[1]); q.y = pack_bf16x2(v[2], v[3]);
    q.z = pack_bf16x2(v[4], v[5]); q.w = pack_bf16x2(v[6], v[7]);
  }
  if (tile) *reinterpret_cast<uint4*>(tile + (ch0 >> 3) * kK8Stride + (row >> 3) * 128 + (row & 7) * 16) = q;
  if (gtile)   // streaming store: the record is next read by another kernel, keep it out of the (small) L1
    __stcs(reinterpret_cast<uint4*>(gtile + (row >> 6) * (gC * 128) + (ch0 >> 3) * 1024 + ((row & 63) >> 3) * 128 +
                                    (row & 7) * 16), q);
}

}  // namespace ctx
