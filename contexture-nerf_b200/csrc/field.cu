// Queries of a trained field away from camera rays: the density lattice and the vertex colours of mesh extraction
// (the original NeRF release's extract_mesh.ipynb: the fine network's relu(sigma) on a regular lattice with zero view
// directions, and a colour per vertex).
//
// Both feed the existing fused forward (ctx_mlp_fwd_ex mode 1, encoding in shared memory) with rays built so that the
// kernel's o + d * z is the query point exactly, FMA contraction or not:
//   * lattice column (i, j) is the ray o = (x_i, y_j, 0), d = (0, 0, 1) with the depth row z_k and view direction 0;
//   * a vertex is the ray o = vertex, d = 0, z = 0 (S = 1) seen along -normal.
// The work goes through a caller-owned workspace in slabs (x-planes of the lattice, chunks of vertices).  The MLP
// computes every point on its own, so the result does not depend on the slab size.  The view-direction head of the
// lattice query is computed and discarded.
#include "ctx_common.cuh"
#include "ctxnerf.h"
#include "mlp_desc.h"

namespace ctx {

constexpr int kFieldThreads = 256;

__host__ inline int64_t field_align(int64_t b) { return (b + 255) / 256 * 256; }

// lattice coordinate o + h * i, one rounding per operation (oracle/marching_cubes.py lattice_axis)
__device__ __forceinline__ float lattice_at(float o, float h, int i) { return __fadd_rn(o, __fmul_rn(h, (float)i)); }

__global__ void __launch_bounds__(kFieldThreads)
grid_rays_kernel(int i0, int64_t n, int Y, int Z, float ox, float oy, float oz, float hx, float hy, float hz,
                 float* __restrict__ ro, float* __restrict__ rd, float* __restrict__ vd, float* __restrict__ z) {
  const int64_t q = (int64_t)blockIdx.x * kFieldThreads + threadIdx.x;
  if (q >= n) return;
  const int k = (int)(q % Z);
  const int64_t r = q / Z;
  z[q] = lattice_at(oz, hz, k);
  if (k == 0) {
    const int j = (int)(r % Y), i = i0 + (int)(r / Y);
    ro[3 * r] = lattice_at(ox, hx, i); ro[3 * r + 1] = lattice_at(oy, hy, j); ro[3 * r + 2] = 0.f;
    rd[3 * r] = 0.f; rd[3 * r + 1] = 0.f; rd[3 * r + 2] = 1.f;
    vd[3 * r] = 0.f; vd[3 * r + 1] = 0.f; vd[3 * r + 2] = 0.f;
  }
}

// sigma = relu(raw[..., 3]) (upstream: np.maximum(raw[..., -1], 0.))
__global__ void __launch_bounds__(kFieldThreads)
grid_sigma_kernel(const float* __restrict__ raw, int64_t n, float* __restrict__ sigma) {
  const int64_t q = (int64_t)blockIdx.x * kFieldThreads + threadIdx.x;
  if (q >= n) return;
  const float s = raw[4 * q + 3];
  sigma[q] = s > 0.f ? s : 0.f;
}

__global__ void __launch_bounds__(kFieldThreads)
vertex_rays_kernel(const float* __restrict__ normals, int64_t n, float* __restrict__ rd, float* __restrict__ vd,
                   float* __restrict__ z) {
  const int64_t q = (int64_t)blockIdx.x * kFieldThreads + threadIdx.x;
  if (q >= n) return;
  z[q] = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    rd[3 * q + c] = 0.f;
    vd[3 * q + c] = normals ? __fsub_rn(0.f, normals[3 * q + c]) : 0.f;
  }
}

__global__ void __launch_bounds__(kFieldThreads)
vertex_rgb_kernel(const float* __restrict__ raw, int64_t n, float* __restrict__ rgb) {
  const int64_t q = (int64_t)blockIdx.x * kFieldThreads + threadIdx.x;
  if (q >= n) return;
#pragma unroll
  for (int c = 0; c < 3; ++c) rgb[3 * q + c] = 1.0f / (1.0f + expf(-raw[4 * q + c]));
}

// the network must be a 4-channel net whose encodings the fused ray mode can form
__host__ inline bool field_net_ok(const CtxNet* net, int L_pts, int L_dirs) {
  if (!net || !net->desc || !net->wpacked || !net->fparams) return false;
  const CtxMlpNet* d = reinterpret_cast<const CtxMlpNet*>(net->desc);
  if (d->out_ch != 4 || L_pts < 0 || L_pts > 10 || d->in_pts != 3 * (1 + 2 * L_pts)) return false;
  return d->in_views == 0 || (L_dirs >= 0 && L_dirs <= 4 && d->in_views == 3 * (1 + 2 * L_dirs));
}

__host__ inline bool grid_dims_ok(int nx, int ny, int nz) {
  for (int c : {nx, ny, nz})
    if (c < 1 || c > 1024) return false;
  return (int64_t)(nx + 1) * (ny + 1) * (nz + 1) < (int64_t(1) << 31);
}

// bytes of a slab of `planes` x-planes: rays_o, rays_d, viewdirs [R,3], z [R,S], raw [R*S,4] (R = planes * Y, S = Z)
__host__ inline int64_t grid_slab_bytes(int64_t planes, int Y, int Z) {
  const int64_t R = planes * Y, P = R * Z;
  return 3 * field_align(R * 12) + field_align(P * 4) + field_align(P * 16);
}

// bytes of a chunk of n vertices: rays_d, viewdirs [n,3], z [n], raw [n,4]
__host__ inline int64_t vertex_chunk_bytes(int64_t n) {
  return 2 * field_align(n * 12) + field_align(n * 4) + field_align(n * 16);
}

}  // namespace ctx

extern "C" int64_t ctx_density_grid_workspace(int nx, int ny, int nz) {
  if (!ctx::grid_dims_ok(nx, ny, nz)) return -1;
  return ctx::grid_slab_bytes(1, ny + 1, nz + 1);
}

extern "C" int ctx_density_grid(const CtxNet* net, int L_pts, int L_dirs, int nx, int ny, int nz, float ox, float oy,
                                float oz, float hx, float hy, float hz, void* workspace, int64_t workspace_bytes,
                                float* sigma, void* stream) {
  if (!ctx::grid_dims_ok(nx, ny, nz) || !ctx::field_net_ok(net, L_pts, L_dirs) || !sigma || !workspace)
    return CTX_ERR_BAD_ARG;
  if (reinterpret_cast<uintptr_t>(workspace) % 256 != 0) return CTX_ERR_BAD_ARG;
  const int X = nx + 1, Y = ny + 1, Z = nz + 1;
  if (workspace_bytes < ctx::grid_slab_bytes(1, Y, Z)) return CTX_ERR_BAD_ARG;
  int planes = 1;                                      // the largest slab the workspace holds
  while (planes < X && ctx::grid_slab_bytes(planes + 1, Y, Z) <= workspace_bytes) ++planes;
  const int64_t Rmax = (int64_t)planes * Y, Pmax = Rmax * Z;
  uint8_t* base = (uint8_t*)workspace;
  float* ro = (float*)base;
  float* rd = (float*)(base + ctx::field_align(Rmax * 12));
  float* vd = (float*)(base + 2 * ctx::field_align(Rmax * 12));
  float* z = (float*)(base + 3 * ctx::field_align(Rmax * 12));
  float* raw = (float*)(base + 3 * ctx::field_align(Rmax * 12) + ctx::field_align(Pmax * 4));
  cudaStream_t st = (cudaStream_t)stream;
  for (int i0 = 0; i0 < X; i0 += planes) {
    const int np = X - i0 < planes ? X - i0 : planes;
    const int64_t R = (int64_t)np * Y, P = R * Z;
    const unsigned blocks = (unsigned)ctx::ceil_div(P, ctx::kFieldThreads);
    ctx::grid_rays_kernel<<<blocks, ctx::kFieldThreads, 0, st>>>(i0, P, Y, Z, ox, oy, oz, hx, hy, hz, ro, rd, vd, z);
    int rc = ctx_mlp_fwd_ex(net->desc, net->wpacked, net->fparams, 1, nullptr, 0, ro, rd, vd, z, Z, L_pts, L_dirs, P,
                            raw, nullptr, nullptr, 0, stream);
    if (rc) return rc;
    ctx::grid_sigma_kernel<<<blocks, ctx::kFieldThreads, 0, st>>>(raw, P, sigma + (int64_t)i0 * Y * Z);
  }
  CTX_RETURN_LAST();
}

extern "C" int64_t ctx_vertex_colors_workspace(int64_t n_vertices) {
  return n_vertices < 1 ? -1 : ctx::vertex_chunk_bytes(n_vertices);
}

extern "C" int ctx_vertex_colors(const CtxNet* net, int L_pts, int L_dirs, const float* vertices,
                                 const float* normals, int64_t V, void* workspace, int64_t workspace_bytes,
                                 float* rgb, void* stream) {
  if (V < 0 || !ctx::field_net_ok(net, L_pts, L_dirs)) return CTX_ERR_BAD_ARG;
  if (V == 0) return 0;
  if (!vertices || !rgb || !workspace || reinterpret_cast<uintptr_t>(workspace) % 256 != 0) return CTX_ERR_BAD_ARG;
  if (workspace_bytes < ctx::vertex_chunk_bytes(1)) return CTX_ERR_BAD_ARG;
  // the largest chunk the workspace holds: 44 bytes per vertex plus the alignment of four arrays
  int64_t chunk = (workspace_bytes - 4 * 256) / 44;
  if (chunk > V) chunk = V;
  while (chunk > 1 && ctx::vertex_chunk_bytes(chunk) > workspace_bytes) --chunk;
  if (chunk < 1) chunk = 1;
  uint8_t* base = (uint8_t*)workspace;
  float* rd = (float*)base;
  float* vd = (float*)(base + ctx::field_align(chunk * 12));
  float* z = (float*)(base + 2 * ctx::field_align(chunk * 12));
  float* raw = (float*)(base + 2 * ctx::field_align(chunk * 12) + ctx::field_align(chunk * 4));
  cudaStream_t st = (cudaStream_t)stream;
  for (int64_t v0 = 0; v0 < V; v0 += chunk) {
    const int64_t n = V - v0 < chunk ? V - v0 : chunk;
    const unsigned blocks = (unsigned)ctx::ceil_div(n, ctx::kFieldThreads);
    ctx::vertex_rays_kernel<<<blocks, ctx::kFieldThreads, 0, st>>>(normals ? normals + 3 * v0 : nullptr, n, rd, vd, z);
    int rc = ctx_mlp_fwd_ex(net->desc, net->wpacked, net->fparams, 1, nullptr, 0, vertices + 3 * v0, rd, vd, z, 1,
                            L_pts, L_dirs, n, raw, nullptr, nullptr, 0, stream);
    if (rc) return rc;
    ctx::vertex_rgb_kernel<<<blocks, ctx::kFieldThreads, 0, st>>>(raw, n, rgb + 3 * v0);
  }
  CTX_RETURN_LAST();
}
