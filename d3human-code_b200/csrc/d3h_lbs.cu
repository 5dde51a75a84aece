// Skinning of the extracted vertices (SURVEY 8f row 4; include/d3h_lbs.h).
//
// The reference (deform/smplx_exavatar_deformer.py:363-421, 472-476) blends J 4x4 joint transforms PER POINT with the
// skinning weights of the point's nearest template vertex, inverts P 4x4 matrices with torch.inverse and multiplies --
// twice per call, on every row of verts_aug, >= 80 % of which are the zeroed unreferenced slots.  With K = 1 (:39) the
// blended matrix is a function of the nearest template vertex alone, so:
//   lbs_blend_kernel      B[v] = sum_j w[v,j] A_j per TEMPLATE vertex (10 475 rows), optionally inverted (Gauss-Jordan, fp64)
//   lbs_compact_kernel    the rows of pts that are not exactly zero -> a dense list (warp-aggregated append)
//   lbs_nearest_kernel    brute-force nearest template vertex of the listed points + ONE search for the origin; the
//                         template streams through shared memory in tiles (10 475 x 12 B = 126 KB: L2-resident)
//   lbs_fill_zero_kernel  zero rows take the origin's result
//   lbs_apply_kernel      two 4x4 products per point from the per-vertex tables
//   lbs_apply_backward_kernel / lbs_blend_backward_kernel   the adjoints (gradients to the points, the joint transforms
//                         and the translation; the nearest-vertex index carries none, init_A is a constant of the run)
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/d3h_lbs.h"
#include "d3h_internal.cuh"

namespace d3h {
namespace lbs {

constexpr int kMaxJoints = 128;
constexpr int kTile = 1024;          // template vertices per shared-memory tile of the search

// ---------------------------------------------------------------------------------------------- per-vertex tables
__global__ void __launch_bounds__(128) lbs_blend_kernel(const float* __restrict__ w, const float* __restrict__ a, int64_t vt, int nj,
                                                        int invert, float* __restrict__ out) {
  __shared__ float s_a[kMaxJoints * 16];
  for (int i = threadIdx.x; i < nj * 16; i += blockDim.x) s_a[i] = a[i];
  __syncthreads();
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= vt) return;
  float m[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) m[c] = 0.f;
  for (int j = 0; j < nj; ++j) {
    const float wj = __ldg(w + v * nj + j);
    if (wj == 0.f) continue;
#pragma unroll
    for (int c = 0; c < 16; ++c) m[c] = fmaf(wj, s_a[16 * j + c], m[c]);
  }
  if (invert) {
    // Gauss-Jordan with partial pivoting on [M | I] in double
    double g[4][8];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) { g[r][c] = (double)m[4 * r + c]; g[r][4 + c] = (r == c) ? 1.0 : 0.0; }
#pragma unroll
    for (int col = 0; col < 4; ++col) {
      int piv = col;
      double best = fabs(g[col][col]);
#pragma unroll
      for (int r = 0; r < 4; ++r)
        if (r > col && fabs(g[r][col]) > best) { best = fabs(g[r][col]); piv = r; }
#pragma unroll
      for (int r = 0; r < 4; ++r)
        if (r == piv && piv != col) {
#pragma unroll
          for (int c = 0; c < 8; ++c) { const double t = g[col][c]; g[col][c] = g[r][c]; g[r][c] = t; }
        }
      const double inv = 1.0 / g[col][col];
#pragma unroll
      for (int c = 0; c < 8; ++c) g[col][c] *= inv;
#pragma unroll
      for (int r = 0; r < 4; ++r)
        if (r != col) {
          const double f = g[r][col];
#pragma unroll
          for (int c = 0; c < 8; ++c) g[r][c] -= f * g[col][c];
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) m[4 * r + c] = (float)g[r][4 + c];
  }
  float4* o = reinterpret_cast<float4*>(out + 16 * v);
  o[0] = make_float4(m[0], m[1], m[2], m[3]);
  o[1] = make_float4(m[4], m[5], m[6], m[7]);
  o[2] = make_float4(m[8], m[9], m[10], m[11]);
  o[3] = make_float4(m[12], m[13], m[14], m[15]);
}

// g_a[j][c] = sum_v w[v,j] g_b[v][c], c < 12; one CTA per joint
__global__ void __launch_bounds__(256) lbs_blend_backward_kernel(const float* __restrict__ w, const float* __restrict__ g_b, int64_t vt,
                                                                 int nj, float* __restrict__ g_a) {
  __shared__ float s_red[8][12];
  const int j = blockIdx.x;
  float acc[12];
#pragma unroll
  for (int c = 0; c < 12; ++c) acc[c] = 0.f;
  for (int64_t v = threadIdx.x; v < vt; v += blockDim.x) {
    const float wj = __ldg(w + v * nj + j);
    if (wj == 0.f) continue;
#pragma unroll
    for (int c = 0; c < 12; ++c) acc[c] = fmaf(wj, __ldg(g_b + 12 * v + c), acc[c]);
  }
#pragma unroll
  for (int c = 0; c < 12; ++c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5][c] = acc[c];
  }
  __syncthreads();
  if (threadIdx.x < 16) {
    float s = 0.f;
    if (threadIdx.x < 12)
      for (int q = 0; q < 8; ++q) s += s_red[q][threadIdx.x];
    g_a[16 * j + threadIdx.x] = s;       // (last row of the 4x4: no gradient, the homogeneous row is not read)
  }
}

// ---------------------------------------------------------------------------------------------- nearest template vertex
struct NearestWs {
  int32_t* list;     // (P) ids of the rows that are not exactly zero
  int32_t* count;    // [0] number of listed rows, [1] nearest template vertex of the origin
};

__global__ void __launch_bounds__(256) lbs_compact_kernel(const float* __restrict__ pts, int64_t n, NearestWs ws) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool live = false;
  if (p < n) live = pts[3 * p] != 0.f || pts[3 * p + 1] != 0.f || pts[3 * p + 2] != 0.f;
  const unsigned m = __ballot_sync(0xffffffffu, live);
  if (m == 0u) return;
  const unsigned lane = threadIdx.x & 31u;
  int base = 0;
  if (lane == 0) base = atomicAdd(ws.count, __popc(m));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (live) ws.list[base + __popc(m & ((1u << lane) - 1u))] = (int32_t)p;
}

// entry i < count: point list[i]; entry i == count: the origin.  knn_points, K = 1: smallest squared distance.
__global__ void __launch_bounds__(256) lbs_nearest_kernel(const float* __restrict__ pts, const float* __restrict__ tmpl, int64_t vt,
                                                          NearestWs ws, int32_t* __restrict__ idx) {
  __shared__ float s_t[3 * kTile];
  const int count = ws.count[0];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if ((int64_t)blockIdx.x * blockDim.x > count) return;      // (whole CTA: nothing listed here)
  const bool live = i <= count;
  const int32_t p = (live && i < count) ? ws.list[i] : -1;
  float px = 0.f, py = 0.f, pz = 0.f;
  if (p >= 0) { px = pts[3ll * p]; py = pts[3ll * p + 1]; pz = pts[3ll * p + 2]; }
  float best = 3.4e38f;
  int best_i = 0;
  for (int64_t t0 = 0; t0 < vt; t0 += kTile) {
    const int nt = (int)min((int64_t)kTile, vt - t0);
    __syncthreads();
    for (int k = threadIdx.x; k < 3 * nt; k += blockDim.x) s_t[k] = __ldg(tmpl + 3 * t0 + k);
    __syncthreads();
    if (live) {
#pragma unroll 4
      for (int k = 0; k < nt; ++k) {
        const float dx = px - s_t[3 * k], dy = py - s_t[3 * k + 1], dz = pz - s_t[3 * k + 2];
        const float d = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        if (d < best) { best = d; best_i = (int)t0 + k; }
      }
    }
  }
  if (!live) return;
  if (p >= 0) idx[p] = best_i;
  else ws.count[1] = best_i;
}

__global__ void __launch_bounds__(256) lbs_fill_zero_kernel(const float* __restrict__ pts, int64_t n, NearestWs ws, int32_t* __restrict__ idx) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  if (pts[3 * p] == 0.f && pts[3 * p + 1] == 0.f && pts[3 * p + 2] == 0.f) idx[p] = ws.count[1];
}

// ---------------------------------------------------------------------------------------------- apply
__device__ __forceinline__ void load16(const float* __restrict__ tab, int v, float (&m)[16]) {
  const float4* q = reinterpret_cast<const float4*>(tab + 16ll * v);
  const float4 r0 = __ldg(q), r1 = __ldg(q + 1), r2 = __ldg(q + 2), r3 = __ldg(q + 3);
  m[0] = r0.x; m[1] = r0.y; m[2] = r0.z; m[3] = r0.w; m[4] = r1.x; m[5] = r1.y; m[6] = r1.z; m[7] = r1.w;
  m[8] = r2.x; m[9] = r2.y; m[10] = r2.z; m[11] = r2.w; m[12] = r3.x; m[13] = r3.y; m[14] = r3.z; m[15] = r3.w;
}

__global__ void __launch_bounds__(256) lbs_apply_kernel(const float* __restrict__ pts, int64_t n, const int32_t* __restrict__ idx,
                                                        const float* __restrict__ binv, const float* __restrict__ bpose,
                                                        const float* __restrict__ trans, float* __restrict__ can,
                                                        float* __restrict__ posed) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int v = idx[p];
  float m[16];
  load16(binv, v, m);
  const float x = pts[3 * p], y = pts[3 * p + 1], z = pts[3 * p + 2];
  // torch.matmul(M_p_inv, pts_h)[..., :3, 0]  (:417-419): rows 0..2 of the homogeneous product
  const float cx = fmaf(m[0], x, fmaf(m[1], y, fmaf(m[2], z, m[3])));
  const float cy = fmaf(m[4], x, fmaf(m[5], y, fmaf(m[6], z, m[7])));
  const float cz = fmaf(m[8], x, fmaf(m[9], y, fmaf(m[10], z, m[11])));
  can[3 * p] = cx; can[3 * p + 1] = cy; can[3 * p + 2] = cz;
  if (bpose == nullptr) return;
  load16(bpose, v, m);
  const float tx = trans ? trans[0] : 0.f, ty = trans ? trans[1] : 0.f, tz = trans ? trans[2] : 0.f;
  posed[3 * p] = fmaf(m[0], cx, fmaf(m[1], cy, fmaf(m[2], cz, m[3]))) + tx;
  posed[3 * p + 1] = fmaf(m[4], cx, fmaf(m[5], cy, fmaf(m[6], cz, m[7]))) + ty;
  posed[3 * p + 2] = fmaf(m[8], cx, fmaf(m[9], cy, fmaf(m[10], cz, m[11]))) + tz;
}

// Zero rows (the bulk of verts_aug) all hit the same table row: their share of g_b is (sum of their upstream gradients)
// (x) [can_0; 1], reduced per CTA in shared memory instead of through 12 atomics per point on one address.  The first zero
// row to claim s_zero_v names the CTA's table row; a zero row with another idx (possible through the ABI, never from
// d3h_lbs_nearest on the same points) takes the per-row atomics like a live row.
__global__ void __launch_bounds__(256) lbs_apply_backward_kernel(const float* __restrict__ g, int64_t n, const int32_t* __restrict__ idx,
                                                                 const float* __restrict__ binv, const float* __restrict__ bpose,
                                                                 const float* __restrict__ can, const float* __restrict__ pts,
                                                                 float* __restrict__ g_pts, float* __restrict__ g_b,
                                                                 float* __restrict__ g_trans) {
  __shared__ float s_zero[3];     // sum of g over this CTA's zero rows (pts row exactly (0,0,0)) with idx == s_zero_v
  __shared__ float s_all[3];      // sum of g over all rows of the CTA
  __shared__ float s_can[3];      // canonical point of those zero rows (the same for all of them: it depends on idx only)
  __shared__ int s_zero_v;
  if (threadIdx.x < 3) { s_zero[threadIdx.x] = 0.f; s_all[threadIdx.x] = 0.f; }
  if (threadIdx.x == 0) s_zero_v = -1;
  __syncthreads();
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float gx = 0.f, gy = 0.f, gz = 0.f, cx = 0.f, cy = 0.f, cz = 0.f;
  bool zero_row = false;
  int v = 0;
  if (p < n) {
    gx = g[3 * p]; gy = g[3 * p + 1]; gz = g[3 * p + 2];
    v = idx[p];
    float mi[16], mp[16];
    load16(binv, v, mi);
    load16(bpose, v, mp);
    // total = B_pose B_inv, rows 0..2 x cols 0..2; g_pts = total^T g
    float out[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float t = fmaf(mp[4 * r], mi[c], fmaf(mp[4 * r + 1], mi[4 + c], fmaf(mp[4 * r + 2], mi[8 + c], mp[4 * r + 3] * mi[12 + c])));
        out[c] = fmaf(t, r == 0 ? gx : (r == 1 ? gy : gz), out[c]);
      }
    }
    g_pts[3 * p] = out[0]; g_pts[3 * p + 1] = out[1]; g_pts[3 * p + 2] = out[2];
    cx = can[3 * p]; cy = can[3 * p + 1]; cz = can[3 * p + 2];
    zero_row = pts != nullptr && pts[3 * p] == 0.f && pts[3 * p + 1] == 0.f && pts[3 * p + 2] == 0.f;
    if (zero_row && atomicCAS(&s_zero_v, -1, v) == -1) { s_can[0] = cx; s_can[1] = cy; s_can[2] = cz; }
  }
  __syncthreads();
  zero_row = zero_row && v == s_zero_v;
  if (p < n && !zero_row && (gx != 0.f || gy != 0.f || gz != 0.f)) {
    float* row = g_b + 12ll * v;
    atomicAdd(row + 0, gx * cx); atomicAdd(row + 1, gx * cy); atomicAdd(row + 2, gx * cz); atomicAdd(row + 3, gx);
    atomicAdd(row + 4, gy * cx); atomicAdd(row + 5, gy * cy); atomicAdd(row + 6, gy * cz); atomicAdd(row + 7, gy);
    atomicAdd(row + 8, gz * cx); atomicAdd(row + 9, gz * cy); atomicAdd(row + 10, gz * cz); atomicAdd(row + 11, gz);
  }
  // CTA sums: all rows (translation gradient) and the zero rows of s_zero_v
  float all[3] = {gx, gy, gz}, zr[3] = {zero_row ? gx : 0.f, zero_row ? gy : 0.f, zero_row ? gz : 0.f};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      all[c] += __shfl_xor_sync(0xffffffffu, all[c], o);
      zr[c] += __shfl_xor_sync(0xffffffffu, zr[c], o);
    }
    if ((threadIdx.x & 31) == 0) {
      if (all[c] != 0.f) atomicAdd(&s_all[c], all[c]);
      if (zr[c] != 0.f) atomicAdd(&s_zero[c], zr[c]);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (g_trans != nullptr)
      for (int c = 0; c < 3; ++c)
        if (s_all[c] != 0.f) atomicAdd(g_trans + c, s_all[c]);
    if (s_zero_v >= 0 && (s_zero[0] != 0.f || s_zero[1] != 0.f || s_zero[2] != 0.f)) {
      float* row = g_b + 12ll * s_zero_v;
      const float cx = s_can[0], cy = s_can[1], cz = s_can[2];
      for (int r = 0; r < 3; ++r) {
        atomicAdd(row + 4 * r, s_zero[r] * cx); atomicAdd(row + 4 * r + 1, s_zero[r] * cy);
        atomicAdd(row + 4 * r + 2, s_zero[r] * cz); atomicAdd(row + 4 * r + 3, s_zero[r]);
      }
    }
  }
}

}  // namespace lbs
}  // namespace d3h

using namespace d3h;
using namespace d3h::lbs;

static int lbs_done(const char* who) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("%s: %s", who, cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}
static bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

extern "C" int d3h_lbs_blend(const float* lbs_weights, const float* a, int64_t n_template, int32_t n_joints, int32_t invert,
                             float* out, d3h_stream_t stream) {
  if (!lbs_weights || !a || !out || n_template < 0 || n_joints <= 0 || n_joints > kMaxJoints || !al16(out)) {
    set_error("d3h_lbs_blend: bad argument (1 <= J <= 128, out 16-byte aligned)");
    return D3H_E_BADARG;
  }
  if (n_template == 0) return D3H_OK;
#ifndef D3H_CPU_EMU
  lbs_blend_kernel<<<(unsigned)((n_template + 127) / 128), 128, 0, (cudaStream_t)stream>>>(lbs_weights, a, n_template, n_joints, invert, out);
#else   // tests/emu: g++ has no <<< >>>
  launch_k(lbs_blend_kernel, (unsigned)((n_template + 127) / 128), 128u, (cudaStream_t)stream, kLaunchStream, lbs_weights, a, n_template,
           n_joints, invert, out);
#endif
  return lbs_done("d3h_lbs_blend");
}

extern "C" int d3h_lbs_blend_backward(const float* lbs_weights, const float* g_b, int64_t n_template, int32_t n_joints, float* g_a,
                                      d3h_stream_t stream) {
  if (!lbs_weights || !g_b || !g_a || n_template < 0 || n_joints <= 0 || n_joints > kMaxJoints) {
    set_error("d3h_lbs_blend_backward: bad argument");
    return D3H_E_BADARG;
  }
#ifndef D3H_CPU_EMU
  lbs_blend_backward_kernel<<<(unsigned)n_joints, 256, 0, (cudaStream_t)stream>>>(lbs_weights, g_b, n_template, n_joints, g_a);
#else
  launch_k(lbs_blend_backward_kernel, (unsigned)n_joints, 256u, (cudaStream_t)stream, kLaunchStream, lbs_weights, g_b, n_template, n_joints, g_a);
#endif
  return lbs_done("d3h_lbs_blend_backward");
}

extern "C" int64_t d3h_lbs_nearest_workspace_bytes(int64_t n_points) { return n_points < 0 ? 0 : (4 * n_points + 64 + 15) / 16 * 16; }

extern "C" int d3h_lbs_nearest(const float* pts, int64_t n_points, const float* tmpl, int64_t n_template, int32_t* idx,
                               void* workspace, int64_t workspace_bytes, d3h_stream_t stream) {
  if (n_points < 0 || n_template <= 0 || n_template >= (1ll << 31) || n_points >= (1ll << 31) || !tmpl ||
      (n_points > 0 && (!pts || !idx)) || !workspace || !al16(workspace) || workspace_bytes < d3h_lbs_nearest_workspace_bytes(n_points)) {
    set_error("d3h_lbs_nearest: bad argument (null pointer, sizes outside [0, 2^31), or workspace too small)");
    return D3H_E_BADARG;
  }
  if (n_points == 0) return D3H_OK;
  cudaStream_t st = (cudaStream_t)stream;
  NearestWs ws;
  ws.count = reinterpret_cast<int32_t*>(workspace);                 // 16 words of counters, then the list
  ws.list = ws.count + 16;
  cudaMemsetAsync(ws.count, 0, 64, st);
  const unsigned blocks = (unsigned)((n_points + 255) / 256);
#ifndef D3H_CPU_EMU
  lbs_compact_kernel<<<blocks, 256, 0, st>>>(pts, n_points, ws);
  lbs_nearest_kernel<<<(unsigned)((n_points + 1 + 255) / 256), 256, 0, st>>>(pts, tmpl, n_template, ws, idx);
  lbs_fill_zero_kernel<<<blocks, 256, 0, st>>>(pts, n_points, ws, idx);
#else
  launch_k(lbs_compact_kernel, blocks, 256u, st, kLaunchStream, pts, n_points, ws);
  launch_k(lbs_nearest_kernel, (unsigned)((n_points + 1 + 255) / 256), 256u, st, kLaunchStream, pts, tmpl, n_template, ws, idx);
  launch_k(lbs_fill_zero_kernel, blocks, 256u, st, kLaunchStream, pts, n_points, ws, idx);
#endif
  return lbs_done("d3h_lbs_nearest");
}

extern "C" int d3h_lbs_apply(const float* pts, int64_t n_points, const int32_t* idx, const float* b_init_inv, const float* b_pose,
                             const float* trans, float* canonical, float* posed, d3h_stream_t stream) {
  if (n_points < 0 || !b_init_inv || !al16(b_init_inv) || !al16(b_pose) ||
      (n_points > 0 && (!pts || !idx || !canonical || (b_pose && !posed)))) {
    set_error("d3h_lbs_apply: bad argument (tables 16-byte aligned; posed required with b_pose)");
    return D3H_E_BADARG;
  }
  if (n_points == 0) return D3H_OK;
#ifndef D3H_CPU_EMU
  lbs_apply_kernel<<<(unsigned)((n_points + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pts, n_points, idx, b_init_inv, b_pose, trans,
                                                                                     canonical, posed);
#else
  launch_k(lbs_apply_kernel, (unsigned)((n_points + 255) / 256), 256u, (cudaStream_t)stream, kLaunchStream, pts, n_points, idx, b_init_inv,
           b_pose, trans, canonical, posed);
#endif
  return lbs_done("d3h_lbs_apply");
}

extern "C" int d3h_lbs_apply_backward(const float* g_posed, int64_t n_points, const int32_t* idx, const float* b_init_inv,
                                      const float* b_pose, const float* canonical, const float* pts, float* g_pts, float* g_b,
                                      float* g_trans, d3h_stream_t stream) {
  if (n_points < 0 || !b_init_inv || !b_pose || !al16(b_init_inv) || !al16(b_pose) || !g_b ||
      (n_points > 0 && (!g_posed || !idx || !canonical || !g_pts))) {
    set_error("d3h_lbs_apply_backward: bad argument");
    return D3H_E_BADARG;
  }
  if (n_points == 0) return D3H_OK;
#ifndef D3H_CPU_EMU
  lbs_apply_backward_kernel<<<(unsigned)((n_points + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      g_posed, n_points, idx, b_init_inv, b_pose, canonical, pts, g_pts, g_b, g_trans);
#else
  launch_k(lbs_apply_backward_kernel, (unsigned)((n_points + 255) / 256), 256u, (cudaStream_t)stream, kLaunchStream, g_posed, n_points, idx,
           b_init_inv, b_pose, canonical, pts, g_pts, g_b, g_trans);
#endif
  return lbs_done("d3h_lbs_apply_backward");
}
