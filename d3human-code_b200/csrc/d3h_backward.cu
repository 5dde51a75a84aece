// Backward of the float pipeline (the reference relies on autograd through gshell_tets.py:291-303, 342-397, 427).
//
//   zero_rows_kernel : dense (N,3)+(N)+(N) gradients of every frame of a backward call whose buffers were not pre-zeroed,
//                    ONE launch (grid.y = frame) ahead of the adjoints, 16-byte stores.  A training step's host work
//                    between two extractions leaves the GPU idle around the backward call, while the forward rounds are
//                    its critical path, so the fill runs here.  The forward call can still do it instead
//                    (d3h_forward_args.zero_g_*, zero_block_kernel; single calls and the tet-sharded path do).
//   adjoint_kernel : one thread per watertight vertex v (= crossing edge (a,b), sorted by a).  The forward sort left, for
//                    every vertex, the list of polygon corners that reference it (tape_runs / tape_slots), so the
//                    boundary-vertex adjoints are GATHERED: for each corner the thread evaluates the two polygon edges
//                    that meet there and pulls g_verts_aug / g_msdf_aug of their boundary rows onto v -- no atomics, no
//                    accumulator buffer, a fixed summation order.  It then adds its own upstream rows and scatters into
//                    pos / sdf / msdf of the two grid vertices.  Edges are sorted by `a`, so lanes that share `a` are
//                    adjacent: their a-side contributions are combined with a segmented warp reduction before one
//                    atomic per run; b-side contributions use plain float atomics (fan-in ~4, max 11).
//
//   adjoint_poly_kernel : calls that ran on the static edge table have no per-vertex corner lists on their tape; for them
//                    the boundary adjoints are SCATTERED (one thread per polygon, one vector atomic per corner) into a
//                    (V,8) accumulator that adjoint_kernel reads and clears.
//   The adjoints of up to 16 frames are one launch each (grid.y = frame).
//
// v2 scattered the boundary adjoints with float atomics into an (V,8) accumulator that a third kernel consumed
// (zero 8.7 + boundary 5.2 + crossing 5.4 us at 128^3); the gather form replaced it on the sort path.
//
// Gradient formulas: SURVEY.md appendix A.5 (verified against the reference's autograd in tests/).
#include <cstdlib>
#include <unordered_set>

#include "d3h_internal.cuh"

namespace d3h {

// Zero-fill of `len` floats at any 4-byte aligned address: scalar head up to the first 16-byte boundary, 16-byte
// stores for the body, scalar tail (rows of a stacked (B,N,3) gradient start at arbitrary multiples of 4 bytes).
__device__ __forceinline__ void zero_span(float* __restrict__ p, int64_t len, int64_t tid, int64_t stride) {
  if (p == nullptr || len <= 0) return;
  int64_t head = (int64_t)(((16u - (unsigned)(reinterpret_cast<uintptr_t>(p) & 15u)) & 15u) >> 2);
  if (head > len) head = len;
  if (tid < head) p[tid] = 0.f;
  float4* __restrict__ body = reinterpret_cast<float4*>(p + head);
  const int64_t n4 = (len - head) >> 2;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t i = tid; i < n4; i += stride) body[i] = z;
  const int64_t t0 = head + 4 * n4;
  if (tid < len - t0) p[t0 + tid] = 0.f;
}

// One row of the backward zero-fill: the gradient buffers one frame of the call zeroes (nullptr: none, or another row
// has it) and their grid size.
struct ZeroRow {
  float *g_pos, *g_sdf, *g_msdf;
  int64_t n;
};
constexpr int kZeroRows = 128;     // rows per launch (4 KB of kernel parameters): the largest batch extract.py makes
struct ZeroBatch {
  ZeroRow r[kZeroRows];
};

// grid.y = row
__global__ void __launch_bounds__(256) zero_rows_kernel(const __grid_constant__ ZeroBatch zb) {
  const ZeroRow& r = zb.r[blockIdx.y];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  zero_span(r.g_pos, 3 * r.n, tid, stride);
  zero_span(r.g_sdf, r.n, tid, stride);
  zero_span(r.g_msdf, r.n, tid, stride);
}

// Forward-side variant: the three pointers come from the argument block (they change from call to call, the launch
// shape does not).
__global__ void __launch_bounds__(256) zero_block_kernel(const FwdBlock* __restrict__ blk, int64_t n, const __grid_constant__ FrameSet fs) {
  blk = frame_ptr(blk, fs.off[blockIdx.y]);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long* tr = trace_begin(blk->trace, (unsigned)blk->a.seq, K_ZERO);
  zero_span(blk->a.zero_g_pos, 3 * n, tid, stride);
  zero_span(blk->a.zero_g_sdf, n, tid, stride);
  zero_span(blk->a.zero_g_msdf, n, tid, stride);
  trace_end(tr);
}

void launch_zero_grads_from_block(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream) {
  int64_t blocks = (5 * a.n_grid / 16 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 8) blocks = 148 * 8;
  // A fused batch runs the fill on a side stream next to the latency-bound kernels of the main chain.  A small launch (a
  // few CTAs per SM that keep HBM busy without taking the CTA slots of those kernels) was measured and is SLOWER: 1.51 /
  // 1.34-1.40 / 1.27 ms per step with 148 / 296 / 592 CTAs against 1.22 ms with 1184 or the full grid (r02at).
  // D3H_ZERO_CTAS = CTAs of the whole launch (A/B of this forward placement, which batches take with
  // D3H_ZERO_IN_FORWARD=1; extract.py); default: no cap.
  const int frames = batch_ctx().frames;
  if (frames > 1) {
    static int total = -1;
    if (total < 0) {
      const char* env = getenv("D3H_ZERO_CTAS");
      total = (env && atoi(env) > 0) ? atoi(env) : 0;
    }
    if (total > 0) {
      const int64_t per = total / frames > 0 ? total / frames : 1;
      if (blocks > per) blocks = per;
    }
  }
  ProfScope ps(K_ZERO, stream);
  launch_k(zero_block_kernel, (unsigned)blocks, 256u, stream, kLaunchLatency, ws.blk, a.n_grid, batch_ctx().fs);
}

static void launch_zero_rows(const ZeroBatch& zb, int m, int64_t max_n, cudaStream_t stream) {
  int64_t blocks = (5 * max_n / 16 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 8) blocks = 148 * 8;
  ProfScope ps(K_ZERO, stream);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)blocks, (unsigned)m, 1);
  cfg.blockDim = dim3(256, 1, 1);
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributePriority;
  at[0].val.priority = launch_priority(kLaunchStream);   // HBM-bound: the latency-bound kernels of other streams go first
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, zero_rows_kernel, zb);
}

// Zero-fill of the gradient buffers of every frame with grads_prezeroed = 0, in ONE launch per kZeroRows frames ahead of
// the adjoints.  A buffer several frames share (sdf / msdf of a batch of video frames) is zeroed once, by its first frame.
static void launch_zero_grads(const d3h_backward_args* a, int64_t n, cudaStream_t stream) {
  ZeroBatch zb;
  memset(&zb, 0, sizeof(zb));
  int m = 0;
  int64_t max_n = 0;
  std::unordered_set<const float*> seen;
  auto first = [&](float* p) { return (p != nullptr && seen.insert(p).second) ? p : nullptr; };
  for (int64_t i = 0; i < n; ++i) {
    if (a[i].grads_prezeroed) continue;
    ZeroRow r;
    r.g_pos = first(a[i].g_pos);
    r.g_sdf = first(a[i].g_sdf);
    r.g_msdf = first(a[i].g_msdf);
    r.n = a[i].n_grid;
    if (!r.g_pos && !r.g_sdf && !r.g_msdf) continue;
    zb.r[m++] = r;
    if (r.n > max_n) max_n = r.n;
    if (m == kZeroRows) {
      launch_zero_rows(zb, m, max_n, stream);
      memset(&zb, 0, sizeof(zb));
      m = 0;
      max_n = 0;
    }
  }
  if (m > 0) launch_zero_rows(zb, m, max_n, stream);
}

// segmented (by key) inclusive suffix-sum inside a warp; lanes with equal key must be contiguous.
// returns the run total in the first lane of every run.
__device__ __forceinline__ float seg_reduce_to_head(float v, int key, unsigned active) {
  const unsigned lane = lane_id();
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float nv = __shfl_down_sync(active, v, o);
    const int nk = __shfl_down_sync(active, key, o);
    if (lane + o < 32 && ((active >> (lane + o)) & 1u) && nk == key) v += nv;
  }
  return v;
}

struct EdgePull {  // what one polygon edge i -> j contributes to its two end vertices
  float gx_i, gy_i, gz_i, gsg_i, gmv_i;
  float gx_j, gy_j, gz_j, gsg_j, gmv_j;
};

// One frame's view of d3h_backward_args as the kernel needs it (passed by value, kAdjBatch frames per launch).
struct AdjFrame {
  const int32_t *edges, *corners, *slots, *runs;
  const float *pos, *sdf, *msdf, *verts_wt, *msdf_wt;
  const float *g_verts_aug, *g_msdf_aug, *g_msdf_bnd, *g_verts_wt, *g_msdf_wt;
  const float *g_verts_tng, *g_mvert_tng;   // through the tangent branch (d3h_tangent_backward), or nullptr
  float *g_pos, *g_sdf, *g_msdf;
  float* vacc;  // scatter form (static edge table calls): (nv,8) accumulator [gx gy gz gsg | gmv - - -], zero on entry
  int64_t nv, t1, t2;
  int msdf_negate, pad;
};
constexpr int kAdjBatch = 16;
struct AdjBatch {
  AdjFrame f[kAdjBatch];
};

// upstream gradient of extra['msdf'] at augmented row `row`: the caller may hand it over whole (g_msdf_aug, Va rows)
// and / or as the boundary slice extra['msdf_boundary'] = msdf[V:] (g_msdf_bnd, Va - V rows)
__device__ __forceinline__ float upstream_msdf(const AdjFrame& f, int64_t row) {
  float g = 0.f;
  if (f.g_msdf_aug != nullptr) g = __ldg(f.g_msdf_aug + row);
  if (f.g_msdf_bnd != nullptr && row >= f.nv) g += __ldg(f.g_msdf_bnd + (row - f.nv));
  return g;
}

// Adjoint of the boundary vertex on polygon edge i -> j whose row in the augmented arrays is `row`
// (gshell_tets.py:353-385 forward; SURVEY A.5).
__device__ __forceinline__ EdgePull pull_edge(const AdjFrame& f, int64_t row, float mi, float mj,
                                              const float* __restrict__ vi, const float* __restrict__ vj) {
  EdgePull r = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float u0, u1, D;
  const bool nz = boundary_weights(mi, mj, u0, u1, D);
  // the row is zeroed in forward unless its polygon's cut references it (gshell_tets.py:423-427):
  // that is exactly when the mSDF sign changes across the edge
  const bool used = (mi > 0.f) != (mj > 0.f);
  float gx = 0.f, gy = 0.f, gz = 0.f;
  if (f.g_verts_aug != nullptr && used) {
    gx = __ldg(f.g_verts_aug + 3 * row);
    gy = __ldg(f.g_verts_aug + 3 * row + 1);
    gz = __ldg(f.g_verts_aug + 3 * row + 2);
  }
  const float gm = upstream_msdf(f, row);
  r.gx_i = gx * u0; r.gy_i = gy * u0; r.gz_i = gz * u0; r.gsg_i = gm * u0;
  r.gx_j = gx * u1; r.gy_j = gy * u1; r.gz_j = gz * u1; r.gsg_j = gm * u1;
  if (nz) {
    // gu1/D - (gu0*u0 + gu1*u1)/D is u0 * g.(vj - vi) / D with gu0 ~ gu1: in fp32 the cancellation costs ~|v| / |vj - vi|
    // (the grid resolution) of relative accuracy, so the per-edge terms are formed in fp64 (inputs and result fp32)
    const double gu0 = (double)gx * vi[0] + (double)gy * vi[1] + (double)gz * vi[2];
    const double gu1 = (double)gx * vj[0] + (double)gy * vj[1] + (double)gz * vj[2];
    const double inv = 1.0 / (double)D;
    const double gD = -(gu0 * (double)u0 + gu1 * (double)u1) * inv;
    r.gmv_i = (float)(gu1 * inv + gD);
    r.gmv_j = (float)(-(gu0 * inv + gD));
  }
  return r;
}

// Scatter form of the boundary-vertex adjoints, for calls that ran on the static edge table (no per-vertex corner lists
// on the tape): one thread per polygon evaluates its 3-4 edges and adds what they contribute to its corners into the
// per-vertex accumulator (one 16-byte vector atomic + one scalar atomic per corner).  adjoint_kernel then reads and
// clears the accumulator.  grid.y = frame.
__global__ void __launch_bounds__(256) adjoint_poly_kernel(const __grid_constant__ AdjBatch batch) {
  const AdjFrame& f = batch.f[blockIdx.y];
  if (f.slots != nullptr || f.vacc == nullptr) return;          // gather-form frame
  if (f.g_verts_aug == nullptr && f.g_msdf_aug == nullptr && f.g_msdf_bnd == nullptr) return;
  const int64_t npoly = f.t1 + f.t2;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npoly) return;
  const bool quad = i >= f.t1;
  const int n = quad ? 4 : 3;
  const int64_t p0 = quad ? (3 * f.t1 + 4 * (i - f.t1)) : 3 * i;
  int L[4];
  float pv[4][3], mv[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    L[k] = (k < n) ? __ldg(f.corners + p0 + k) : 0;
    if (k < n) {
      pv[k][0] = __ldg(f.verts_wt + 3ll * L[k]); pv[k][1] = __ldg(f.verts_wt + 3ll * L[k] + 1);
      pv[k][2] = __ldg(f.verts_wt + 3ll * L[k] + 2);
      mv[k] = __ldg(f.msdf_wt + L[k]);
    } else {
      pv[k][0] = pv[k][1] = pv[k][2] = 0.f; mv[k] = 0.f;
    }
  }
  float acc[4][5];
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int c = 0; c < 5; ++c) acc[k][c] = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k >= n) break;
    const int kn = (k + 1 == n) ? 0 : k + 1;
    // select the next corner without dynamic register indexing
    float pn[3], mn;
#pragma unroll
    for (int c = 0; c < 3; ++c) pn[c] = (kn == 0) ? pv[0][c] : (kn == 1) ? pv[1][c] : (kn == 2) ? pv[2][c] : pv[3][c];
    mn = (kn == 0) ? mv[0] : (kn == 1) ? mv[1] : (kn == 2) ? mv[2] : mv[3];
    const EdgePull e = pull_edge(f, f.nv + p0 + k, mv[k], mn, pv[k], pn);
    acc[k][0] += e.gx_i; acc[k][1] += e.gy_i; acc[k][2] += e.gz_i; acc[k][3] += e.gsg_i; acc[k][4] += e.gmv_i;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (q == kn) {
        acc[q][0] += e.gx_j; acc[q][1] += e.gy_j; acc[q][2] += e.gz_j; acc[q][3] += e.gsg_j; acc[q][4] += e.gmv_j;
      }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k >= n) break;
    float* row = f.vacc + 8ll * L[k];
    atomicAdd(reinterpret_cast<float4*>(row), make_float4(acc[k][0], acc[k][1], acc[k][2], acc[k][3]));
    if (acc[k][4] != 0.f) atomicAdd(row + 4, acc[k][4]);
  }
}

// grid.y = frame of the batch: the adjoints of all frames are one launch (their blocks run side by side)
__global__ void __launch_bounds__(256) adjoint_kernel(const __grid_constant__ AdjBatch batch) {
  const AdjFrame& f = batch.f[blockIdx.y];
  const int64_t nv = f.nv, t1 = f.t1;
  if ((int64_t)blockIdx.x * blockDim.x >= nv) return;
  const int32_t* __restrict__ edges = f.edges;
  const int32_t* __restrict__ corners = f.corners;
  const int32_t* __restrict__ slots = f.slots;
  const int32_t* __restrict__ runs = f.runs;
  const float* __restrict__ pos = f.pos;
  const float* __restrict__ sdf = f.sdf;
  const float* __restrict__ msdf = f.msdf;
  const float* __restrict__ verts_wt = f.verts_wt;
  const float* __restrict__ msdf_wt = f.msdf_wt;
  const float* __restrict__ g_verts_aug = f.g_verts_aug;
  const float* __restrict__ g_verts_wt = f.g_verts_wt;
  const float* __restrict__ g_msdf_wt = f.g_msdf_wt;
  float* __restrict__ g_pos = f.g_pos;
  float* __restrict__ g_sdf = f.g_sdf;
  float* __restrict__ g_msdf = f.g_msdf;
  const int msdf_negate = f.msdf_negate;
  const bool any_msdf_up = f.g_msdf_aug != nullptr || f.g_msdf_bnd != nullptr;
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = v < nv;
  const unsigned active = __ballot_sync(0xffffffffu, live);
  if (!live) return;
  const float mv = __ldg(msdf_wt + v);
  const float pv[3] = {__ldg(verts_wt + 3 * v), __ldg(verts_wt + 3 * v + 1), __ldg(verts_wt + 3 * v + 2)};
  // g_vert, g_sg (stop-grad mSDF attribute), g_mv (mSDF through the boundary coefficients)
  float gx = 0.f, gy = 0.f, gz = 0.f, gsg = 0.f, gmv = 0.f;

  if (slots == nullptr && f.vacc != nullptr) {
    // scatter form: adjoint_poly_kernel has summed the boundary contributions of all corners on v; take and clear
    float4* row = reinterpret_cast<float4*>(f.vacc + 8ll * v);
    const float4 a0 = row[0], a1 = row[1];
    gx = a0.x; gy = a0.y; gz = a0.z; gsg = a0.w; gmv = a1.x;
    row[0] = make_float4(0.f, 0.f, 0.f, 0.f);
    row[1] = make_float4(0.f, 0.f, 0.f, 0.f);
  } else if (g_verts_aug != nullptr || any_msdf_up) {
    const int s0 = __ldg(runs + v), s1 = __ldg(runs + v + 1);
    for (int s = s0; s < s1; ++s) {
      const int64_t p = __ldg(slots + s);  // a corner of some polygon that sits on vertex v
      int64_t pbase;
      int n, k;
      if (p < 3 * t1) { k = (int)(p % 3); pbase = p - k; n = 3; }
      else { const int64_t q = p - 3 * t1; k = (int)(q & 3); pbase = p - k; n = 4; }
      const int64_t pn = pbase + (k + 1 == n ? 0 : k + 1), pp = pbase + (k == 0 ? n - 1 : k - 1);
      const int64_t jn = __ldg(corners + pn), jp = __ldg(corners + pp);
      const float vn[3] = {__ldg(verts_wt + 3 * jn), __ldg(verts_wt + 3 * jn + 1), __ldg(verts_wt + 3 * jn + 2)};
      const float vp[3] = {__ldg(verts_wt + 3 * jp), __ldg(verts_wt + 3 * jp + 1), __ldg(verts_wt + 3 * jp + 2)};
      // edge p -> pn: v is the i end (row nv + p); edge pp -> p: v is the j end (row nv + pp)
      const EdgePull e0 = pull_edge(f, nv + p, mv, __ldg(msdf_wt + jn), pv, vn);
      const EdgePull e1 = pull_edge(f, nv + pp, __ldg(msdf_wt + jp), mv, vp, pv);
      gx += e0.gx_i + e1.gx_j;
      gy += e0.gy_i + e1.gy_j;
      gz += e0.gz_i + e1.gz_j;
      gsg += e0.gsg_i + e1.gsg_j;
      gmv += e0.gmv_i + e1.gmv_j;
    }
  }

  const int a = edges[2 * v], b = edges[2 * v + 1];
  const bool used = mv > 0.f;  // verts_aug[v] was zeroed in forward otherwise
  if (g_verts_aug != nullptr && used) {
    gx += __ldg(g_verts_aug + 3 * v); gy += __ldg(g_verts_aug + 3 * v + 1); gz += __ldg(g_verts_aug + 3 * v + 2);
  }
  if (g_verts_wt != nullptr) {
    gx += __ldg(g_verts_wt + 3 * v); gy += __ldg(g_verts_wt + 3 * v + 1); gz += __ldg(g_verts_wt + 3 * v + 2);
  }
  if (f.g_msdf_aug != nullptr) gsg += __ldg(f.g_msdf_aug + v);
  if (g_msdf_wt != nullptr) gsg += __ldg(g_msdf_wt + v);
  if (f.g_verts_tng != nullptr) {
    gx += __ldg(f.g_verts_tng + 3 * v); gy += __ldg(f.g_verts_tng + 3 * v + 1); gz += __ldg(f.g_verts_tng + 3 * v + 2);
  }
  if (f.g_mvert_tng != nullptr) gmv += __ldg(f.g_mvert_tng + v);
  float w0, w1, dd;
  crossing_weights(__ldg(sdf + a), __ldg(sdf + b), w0, w1, dd);
  float ma = __ldg(msdf + a), mb = __ldg(msdf + b);
  if (msdf_negate) { ma = -ma; mb = -mb; }
  const float pax = __ldg(pos + 3ll * a), pay = __ldg(pos + 3ll * a + 1), paz = __ldg(pos + 3ll * a + 2);
  const float pbx = __ldg(pos + 3ll * b), pby = __ldg(pos + 3ll * b + 1), pbz = __ldg(pos + 3ll * b + 2);
  // g_sdf = gw1/dd - (gw0*w0 + gw1*w1)/dd = w0 * (gw1 - gw0) / dd with gw0 ~ gw1 (both ~ g.pos, their difference
  // ~ g.edge): fp32 loses |pos| / |edge| = the grid resolution in relative accuracy (4.6e-5 at 256^3, measured), so
  // the per-edge terms are formed in fp64 from the fp32 inputs; the accumulation into g_sdf stays fp32 atomics
  const double gw0 = (double)gx * pax + (double)gy * pay + (double)gz * paz + (double)gmv * ma;
  const double gw1 = (double)gx * pbx + (double)gy * pby + (double)gz * pbz + (double)gmv * mb;
  const double inv = 1.0 / (double)dd;
  const double gdd = -(gw0 * (double)w0 + gw1 * (double)w1) * inv;
  const float gs_a = (float)(gw1 * inv + gdd), gs_b = (float)(-(gw0 * inv + gdd));
  const float gm_in = gmv + gsg;

  // a side: runs of equal `a` are contiguous (edges sorted lexicographically) -> one atomic per run and warp
  float sax = seg_reduce_to_head(gx * w0, a, active);
  float say = seg_reduce_to_head(gy * w0, a, active);
  float saz = seg_reduce_to_head(gz * w0, a, active);
  float sas = seg_reduce_to_head(gs_a, a, active);
  float sam = seg_reduce_to_head(gm_in * w0, a, active);
  const unsigned lane = lane_id();
  const int a_prev = __shfl_up_sync(active, a, 1);
  const bool head = (lane == 0) || !((active >> (lane - 1)) & 1u) || (a_prev != a);
  if (head) {
    atomicAdd(g_pos + 3ll * a, sax); atomicAdd(g_pos + 3ll * a + 1, say); atomicAdd(g_pos + 3ll * a + 2, saz);
    atomicAdd(g_sdf + a, sas);
    if (g_msdf != nullptr) atomicAdd(g_msdf + a, sam);
  }
  // b side
  atomicAdd(g_pos + 3ll * b, gx * w1); atomicAdd(g_pos + 3ll * b + 1, gy * w1); atomicAdd(g_pos + 3ll * b + 2, gz * w1);
  atomicAdd(g_sdf + b, gs_b);
  if (g_msdf != nullptr) atomicAdd(g_msdf + b, gm_in * w1);
}

static AdjFrame adj_frame(const d3h_backward_args& a) {
  AdjFrame f;
  f.edges = a.tape_edges; f.corners = a.tape_corners; f.slots = a.tape_slots; f.runs = a.tape_runs;
  f.pos = a.pos; f.sdf = a.sdf; f.msdf = a.msdf; f.verts_wt = a.verts_wt; f.msdf_wt = a.msdf_wt;
  f.g_verts_aug = a.g_verts_aug; f.g_msdf_aug = a.g_msdf_aug; f.g_msdf_bnd = a.g_msdf_boundary;
  f.g_verts_wt = a.g_verts_wt; f.g_msdf_wt = a.g_msdf_wt;
  f.g_verts_tng = a.g_verts_tng; f.g_mvert_tng = a.g_mvert_tng;
  f.g_pos = a.g_pos; f.g_sdf = a.g_sdf; f.g_msdf = a.g_msdf;
  f.vacc = a.vacc;
  f.nv = a.n_verts; f.t1 = a.n_tri_tets; f.t2 = a.n_quad_tets;
  f.msdf_negate = a.msdf_negate; f.pad = 0;
  return f;
}

static bool has_upstream(const d3h_backward_args& a) {
  return a.g_verts_aug || a.g_msdf_aug || a.g_msdf_boundary || a.g_verts_wt || a.g_msdf_wt || a.g_verts_tng ||
         a.g_mvert_tng;
}

// Adjoints of n frames: the zero-fill first (frames that were not pre-zeroed), then ONE adjoint launch per kAdjBatch
// consecutive frames (grid.y = frame).  A frame with no surface or no upstream gradient gets no row of the launch, so a
// call of blocks without upstream gradients is a zero-fill alone (extract.py zeroes a batch's buffers that way).
void launch_backward_batch(const d3h_backward_args* a, int64_t n, cudaStream_t stream) {
  launch_zero_grads(a, n, stream);
  for (int64_t i0 = 0; i0 < n; i0 += kAdjBatch) {
    AdjBatch batch;
    memset(&batch, 0, sizeof(batch));
    int m = 0;
    int64_t max_nv = 0, max_poly = 0;
    for (int64_t i = i0; i < n && i < i0 + kAdjBatch; ++i) {
      if (a[i].n_verts <= 0 || !has_upstream(a[i])) continue;
      batch.f[m++] = adj_frame(a[i]);
      if (a[i].n_verts > max_nv) max_nv = a[i].n_verts;
      const bool scatter = a[i].tape_slots == nullptr && a[i].vacc != nullptr;
      if (scatter && a[i].n_tri_tets + a[i].n_quad_tets > max_poly) max_poly = a[i].n_tri_tets + a[i].n_quad_tets;
    }
    if (m == 0) continue;
    if (max_poly > 0) {
      ProfScope ps(K_ADJOINT_POLY, stream);
      cudaLaunchConfig_t cfg;
      memset(&cfg, 0, sizeof(cfg));
      cfg.gridDim = dim3((unsigned)((max_poly + 255) / 256), (unsigned)m, 1);
      cfg.blockDim = dim3(256, 1, 1);
      cfg.stream = stream;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributePriority;
      at[0].val.priority = launch_priority(kLaunchLatency);
      cfg.attrs = at;
      cfg.numAttrs = 1;
      cudaLaunchKernelEx(&cfg, adjoint_poly_kernel, batch);
    }
    ProfScope ps(K_ADJOINT, stream);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)((max_nv + 255) / 256), (unsigned)m, 1);
    cfg.blockDim = dim3(256, 1, 1);
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributePriority;
    at[0].val.priority = launch_priority(kLaunchLatency);
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, adjoint_kernel, batch);
  }
}

void launch_backward(const d3h_backward_args& a, cudaStream_t stream) { launch_backward_batch(&a, 1, stream); }

// out[i][:] = src[ids[i]][:], rows of `width` floats (compact gradient return, see d3h_gather_rows)
__global__ void __launch_bounds__(256) gather_rows_kernel(const int32_t* __restrict__ ids, int64_t n_ids,
                                                          const float* __restrict__ src, int64_t n_rows, int width,
                                                          float* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t total = n_ids * width;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride) {
    const int64_t i = k / width;
    const int c = (int)(k - i * width);
    const int64_t r = (int64_t)__ldg(ids + i);
    out[k] = (r >= 0 && r < n_rows) ? __ldg(src + r * width + c) : 0.f;
  }
}

}  // namespace d3h

using namespace d3h;

extern "C" int d3h_gather_rows(const int32_t* ids, int64_t n_ids, const float* src, int64_t n_rows, int32_t width,
                               float* out, d3h_stream_t stream) {
  if (n_ids < 0 || n_rows < 0 || width <= 0 || width > 16 || (n_ids > 0 && (!ids || !src || !out))) {
    set_error("d3h_gather_rows: bad argument (null pointer, negative size, or width outside [1, 16])");
    return D3H_E_BADARG;
  }
  if (n_ids == 0) return D3H_OK;
  int64_t blocks = (n_ids * width + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(gather_rows_kernel, (unsigned)blocks, 256u, (cudaStream_t)stream, kLaunchLatency, ids, n_ids, src, n_rows,
           (int)width, out);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("d3h_gather_rows: %s", cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}
