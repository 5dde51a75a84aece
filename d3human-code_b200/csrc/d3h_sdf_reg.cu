// The SDF sign-change regulariser (compute_sdf_reg_loss, hmsdf.py:162-170; include/d3h_tets.h, geometry/sdf_reg.py).
//
// The reference gathers both end points of every grid edge (30 M floats at 128^3 from a 237 MB int64 edge list), keeps
// the edges whose end points differ in torch.sign (a boolean-mask compaction: one device -> host sync) and runs two BCE
// kernels on them.  Here the edge list is one of the static tables of the extraction's edge scan (d3h_scan.cu), read with
// two sign bitmaps instead of the field:
//   sdf_reg_bits_kernel   one pass over sdf: a `> 0` and a `< 0` bitmap (__ballot_sync), and a flag for NaN
//   sdf_reg_runs_kernel   run-length tables: a thread per (chunk, d, mask) entry; the three-valued sign differs exactly
//                         where the `> 0` bits or the `< 0` bits differ, so x = ((win_pos ^ own_pos) | (win_neg ^ own_neg))
//                         & mask flags 32 edges.  Warps that flag nothing (all but a few per cent) leave; the entries that
//                         flag something are expanded by the whole warp, lane l = lane l of the entry: sdf[32c + l] and
//                         sdf[32c + l + d] are two coalesced loads, no id row is read
//   sdf_reg_rows_kernel   transposed rows (grids without that structure): a warp per chunk of 32 vertices, the same test
//                         per (a, b) row entry; padding entries (b == a) never differ
//   sdf_reg_final_kernel  one CTA: the per-warp partial sums (float64) and counts in a fixed order -> loss, M
// The backward pass runs the same scan on the bitmaps the forward pass left in the workspace and scatters
// g (sigmoid(s) - target) / M with float atomics.  No kernel's shape depends on M, and g and M are read on the device: the
// host never waits.
//
// Compiled as part of d3h_scan.cu (included at its end), not as a translation unit of its own.

#include "../../include/d3h_tets.h"
#include "d3h_internal.cuh"

namespace d3h {
namespace sdfreg {

constexpr int kThreads = 256;
constexpr int kFinalThreads = 512;

// Workspace, carved from one caller-owned allocation (every region 256-byte aligned relative to its start):
struct Ws {
  unsigned* nan_flag;      // 1: sdf holds a NaN
  int64_t* count;          // M of the last forward call (read by the backward pass)
  unsigned* pos;           // ceil(N/32) + 1 words: sdf > 0 (the last word is zero: sign_window reads behind the last vertex)
  unsigned* neg;           // ceil(N/32) + 1 words: sdf < 0
  double* part_sum;        // per warp of the scan: sum of the BCE terms of its edges
  unsigned* part_cnt;      // per warp of the scan: its selected edges
};

static int64_t al256(int64_t b) { return (b + 255) & ~(int64_t)255; }

// warps of the scan: a thread per run-length entry, or a warp per chunk of 32 vertices
static int64_t scan_warps(int64_t n_grid, int64_t n_runs, bool runs) {
  const int64_t n_chunks = (n_grid + 31) >> 5;
  return runs ? (n_runs + kThreads - 1) / kThreads * (kThreads / 32) : n_chunks;
}

static Ws carve(void* base, int64_t n_grid, int64_t n_entries, int64_t* total) {
  const int64_t words = ((n_grid + 31) >> 5) + 1;
  const int64_t slots = scan_warps(n_grid, n_entries, true) > scan_warps(n_grid, n_entries, false)
                            ? scan_warps(n_grid, n_entries, true) : scan_warps(n_grid, n_entries, false);
  char* p = static_cast<char*>(base);
  int64_t off = 0;
  auto take = [&](int64_t bytes) { char* r = p ? p + off : nullptr; off += al256(bytes); return r; };
  Ws w;
  char* head = take(16);
  w.nan_flag = reinterpret_cast<unsigned*>(head);
  w.count = reinterpret_cast<int64_t*>(head ? head + 8 : nullptr);
  w.pos = reinterpret_cast<unsigned*>(take(4 * words));
  w.neg = reinterpret_cast<unsigned*>(take(4 * words));
  w.part_sum = reinterpret_cast<double*>(take(8 * slots));
  w.part_cnt = reinterpret_cast<unsigned*>(take(4 * slots));
  *total = off;
  return w;
}

// torch's binary_cross_entropy_with_logits per element: (1 - t) x - log_sigmoid(x), log_sigmoid(x) = min(x, 0) -
// log1p(exp(-|x|)); precise expf / log1pf (the build takes no fast-math)
__device__ __forceinline__ float bce(float x, float t) {
  return (1.f - t) * x - (fminf(x, 0.f) - log1pf(expf(-fabsf(x))));
}
__device__ __forceinline__ float sigmoid(float x) { return 1.f / (1.f + expf(-x)); }

__global__ void __launch_bounds__(kThreads) sdf_reg_bits_kernel(const float* __restrict__ sdf, int64_t n_grid, int64_t words, Ws w) {
  const int64_t v = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if ((v >> 5) >= words) return;   // (warp-uniform)
  const float s = v < n_grid ? sdf[v] : 0.f;
  const unsigned p = __ballot_sync(0xffffffffu, s > 0.f), q = __ballot_sync(0xffffffffu, s < 0.f);
  const bool nan = __any_sync(0xffffffffu, s != s);
  if (lane_id() == 0) {
    w.pos[v >> 5] = p;
    w.neg[v >> 5] = q;
    if (nan) atomicOr(w.nan_flag, 1u);
  }
}

// One selected edge (a, b): its two BCE terms (forward) or its two gradient contributions (backward).
template <bool BWD>
__device__ __forceinline__ void edge_term(const float* __restrict__ sdf, int64_t a, int64_t b, float scale, float* __restrict__ g_sdf,
                                          double& acc) {
  const float sa = __ldg(sdf + a), sb = __ldg(sdf + b);
  const float ta = sa > 0.f ? 1.f : 0.f, tb = sb > 0.f ? 1.f : 0.f;
  if (BWD) {
    atomicAdd(g_sdf + a, scale * (sigmoid(sa) - tb));
    atomicAdd(g_sdf + b, scale * (sigmoid(sb) - ta));
  } else {
    acc += (double)bce(sa, tb) + (double)bce(sb, ta);
  }
}

// the warp's partial sum and count, in a fixed shuffle order (the loss is the same bit for bit on every run)
__device__ __forceinline__ void warp_partial(const Ws& w, int64_t warp, double acc, unsigned cnt) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane_id() == 0) {
    w.part_sum[warp] = acc;
    w.part_cnt[warp] = cnt;
  }
}

__device__ __forceinline__ float grad_scale(const Ws& w, const float* __restrict__ g_loss) {
  const int64_t m = *w.count;
  return m > 0 ? (float)((double)__ldg(g_loss) / (double)m) : 0.f;
}

template <bool BWD>
__global__ void __launch_bounds__(kThreads)
sdf_reg_runs_kernel(const float* __restrict__ sdf, const int2* __restrict__ runs, const int32_t* __restrict__ run_chunk, int64_t n_runs,
                    Ws w, const float* __restrict__ g_loss, float* __restrict__ g_sdf) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;   // entry
  const unsigned lane = lane_id();
  unsigned x = 0u;       // bit l: the edge (32c + l, 32c + l + d) exists and its end points differ in sign
  int c = 0, d = 0;
  if (i < n_runs) {
    c = __ldg(run_chunk + i);
    const int2 e = __ldg(runs + i);
    d = e.x;
    const int64_t b0 = ((int64_t)c << 5) + d;
    x = ((sign_window(w.pos, b0) ^ __ldg(w.pos + c)) | (sign_window(w.neg, b0) ^ __ldg(w.neg + c))) & (unsigned)e.y;
  }
  const unsigned live = __ballot_sync(0xffffffffu, x != 0u);
  if (live == 0u) {
    if (!BWD && lane == 0) { w.part_sum[i >> 5] = 0.0; w.part_cnt[i >> 5] = 0u; }
    return;
  }
  const float scale = BWD ? grad_scale(w, g_loss) : 0.f;
  double acc = 0.0;
  for (unsigned m = live; m != 0u; m &= m - 1u) {
    const int src = __ffs((int)m) - 1;
    const unsigned xs = __shfl_sync(0xffffffffu, x, src);
    const int cs = __shfl_sync(0xffffffffu, c, src), ds = __shfl_sync(0xffffffffu, d, src);
    if ((xs >> lane) & 1u) {
      const int64_t a = ((int64_t)cs << 5) + lane;
      edge_term<BWD>(sdf, a, a + ds, scale, g_sdf, acc);
    }
  }
  if (!BWD) warp_partial(w, i >> 5, acc, (unsigned)__popc(x));
}

template <bool BWD>
__global__ void __launch_bounds__(kThreads)
sdf_reg_rows_kernel(const float* __restrict__ sdf, int64_t n_grid, const int32_t* __restrict__ rows, const int32_t* __restrict__ row_off,
                    Ws w, const float* __restrict__ g_loss, float* __restrict__ g_sdf) {
  const int64_t c = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5;   // chunk = warp
  const int64_t n_chunks = (n_grid + 31) >> 5;
  if (c >= n_chunks) return;   // (warp-uniform)
  const unsigned lane = lane_id();
  const int64_t a = (c << 5) + lane;
  const bool in = a < n_grid;
  const unsigned own_p = (__ldg(w.pos + c) >> lane) & 1u, own_n = (__ldg(w.neg + c) >> lane) & 1u;
  const int r0 = __ldg(row_off + c), r1 = __ldg(row_off + c + 1);
  const float scale = BWD ? grad_scale(w, g_loss) : 0.f;
  double acc = 0.0;
  unsigned cnt = 0u;
#pragma unroll 4
  for (int r = r0; r < r1; ++r) {
    const int b = ld_stream_s32(rows + ((int64_t)r << 5) + lane);
    const bool hit = in && b != a && ((occ_of(w.pos, b) ^ own_p) | (occ_of(w.neg, b) ^ own_n)) != 0u;
    if (hit) {
      edge_term<BWD>(sdf, a, b, scale, g_sdf, acc);
      ++cnt;
    }
  }
  if (!BWD) warp_partial(w, c, acc, cnt);
}

__global__ void __launch_bounds__(kFinalThreads) sdf_reg_final_kernel(Ws w, int64_t n_warps, float* __restrict__ loss) {
  __shared__ double s_sum[kFinalThreads];
  __shared__ unsigned long long s_cnt[kFinalThreads];
  const int t = threadIdx.x;
  double s = 0.0;
  unsigned long long n = 0ull;
  for (int64_t j = t; j < n_warps; j += kFinalThreads) {
    s += w.part_sum[j];
    n += w.part_cnt[j];
  }
  s_sum[t] = s;
  s_cnt[t] = n;
  __syncthreads();
  for (int o = kFinalThreads / 2; o > 0; o >>= 1) {
    if (t < o) {
      s_sum[t] += s_sum[t + o];
      s_cnt[t] += s_cnt[t + o];
    }
    __syncthreads();
  }
  if (t == 0) {
    const unsigned long long m = s_cnt[0];
    *w.count = (int64_t)m;
    // torch: the mean of an empty selection is NaN; a NaN end point is selected (NaN != x) and makes its terms NaN
    *loss = (m == 0ull || *w.nan_flag != 0u) ? nanf("") : (float)(s_sum[0] / (double)m);
  }
}

}  // namespace sdfreg
}  // namespace d3h

using namespace d3h;
using namespace d3h::sdfreg;

static int sdf_reg_done(const char* who) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("%s: %s", who, cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}

extern "C" int64_t d3h_sdf_reg_workspace_bytes(int64_t n_grid, int64_t n_entries) {
  if (n_grid < 0 || n_entries < 0) return 0;
  int64_t total = 0;
  carve(nullptr, n_grid, n_entries, &total);
  return total;
}

// common argument check; -> 1 run-length form, 0 rows form, -1 refused (message set)
static int sdf_reg_form(const char* who, const float* sdf, int64_t n_grid, const int32_t* edge_runs, const int32_t* edge_run_chunk,
                        int64_t n_edge_runs, const int32_t* edge_rows, const int32_t* edge_row_off, const void* workspace,
                        int64_t workspace_bytes) {
  const bool runs = edge_runs != nullptr || edge_run_chunk != nullptr;
  const bool rows = edge_rows != nullptr || edge_row_off != nullptr;
  if (runs == rows || (runs && (!edge_runs || !edge_run_chunk || (reinterpret_cast<uintptr_t>(edge_runs) & 7))) ||
      (rows && (!edge_rows || !edge_row_off))) {
    set_error("%s: bad argument (exactly one table form: edge_runs + edge_run_chunk, 8-byte aligned, or edge_rows + edge_row_off)", who);
    return -1;
  }
  if (n_grid < 0 || n_grid >= (1ll << 31) || (n_grid > 0 && !sdf) || n_edge_runs < 0 || n_edge_runs >= (1ll << 26) ||
      (rows && n_edge_runs != 0) || !workspace || (reinterpret_cast<uintptr_t>(workspace) & 15) ||
      workspace_bytes < d3h_sdf_reg_workspace_bytes(n_grid, n_edge_runs)) {
    set_error("%s: bad argument (N in [0, 2^31), n_edge_runs in [0, 2^26) and 0 with the rows form, workspace 16-byte aligned "
              "and at least d3h_sdf_reg_workspace_bytes(N, n_edge_runs))", who);
    return -1;
  }
  return runs ? 1 : 0;
}

extern "C" int d3h_sdf_reg_forward(const float* sdf, int64_t n_grid, const int32_t* edge_runs, const int32_t* edge_run_chunk,
                                   int64_t n_edge_runs, const int32_t* edge_rows, const int32_t* edge_row_off, void* workspace,
                                   int64_t workspace_bytes, float* loss, d3h_stream_t stream) {
  const int form = sdf_reg_form("d3h_sdf_reg_forward", sdf, n_grid, edge_runs, edge_run_chunk, n_edge_runs, edge_rows, edge_row_off,
                                workspace, workspace_bytes);
  if (form < 0) return D3H_E_BADARG;
  if (!loss) {
    set_error("d3h_sdf_reg_forward: bad argument (loss is NULL)");
    return D3H_E_BADARG;
  }
  cudaStream_t st = (cudaStream_t)stream;
  int64_t total = 0;
  const Ws w = carve(workspace, n_grid, n_edge_runs, &total);
  const int64_t words = ((n_grid + 31) >> 5) + 1;
  cudaMemsetAsync(w.nan_flag, 0, 4, st);
  launch_k(sdf_reg_bits_kernel, (unsigned)((words * 32 + kThreads - 1) / kThreads), (unsigned)kThreads, st, kLaunchStream, sdf, n_grid,
           words, w);
  const int64_t n_warps = scan_warps(n_grid, n_edge_runs, form == 1);
  const unsigned grid = (unsigned)((n_warps * 32 + kThreads - 1) / kThreads);
  if (grid > 0) {
    if (form == 1)
      launch_k(sdf_reg_runs_kernel<false>, grid, (unsigned)kThreads, st, kLaunchStream, sdf, reinterpret_cast<const int2*>(edge_runs),
               edge_run_chunk, n_edge_runs, w, (const float*)nullptr, (float*)nullptr);
    else
      launch_k(sdf_reg_rows_kernel<false>, grid, (unsigned)kThreads, st, kLaunchStream, sdf, n_grid, edge_rows, edge_row_off, w,
               (const float*)nullptr, (float*)nullptr);
  }
  launch_k(sdf_reg_final_kernel, 1u, (unsigned)kFinalThreads, st, kLaunchLatency, w, n_warps, loss);
  return sdf_reg_done("d3h_sdf_reg_forward");
}

extern "C" int d3h_sdf_reg_backward(const float* sdf, int64_t n_grid, const int32_t* edge_runs, const int32_t* edge_run_chunk,
                                    int64_t n_edge_runs, const int32_t* edge_rows, const int32_t* edge_row_off, const float* g_loss,
                                    void* workspace, int64_t workspace_bytes, float* g_sdf, d3h_stream_t stream) {
  const int form = sdf_reg_form("d3h_sdf_reg_backward", sdf, n_grid, edge_runs, edge_run_chunk, n_edge_runs, edge_rows, edge_row_off,
                                workspace, workspace_bytes);
  if (form < 0) return D3H_E_BADARG;
  if (!g_loss || (n_grid > 0 && !g_sdf)) {
    set_error("d3h_sdf_reg_backward: bad argument (g_loss or g_sdf is NULL)");
    return D3H_E_BADARG;
  }
  cudaStream_t st = (cudaStream_t)stream;
  int64_t total = 0;
  const Ws w = carve(workspace, n_grid, n_edge_runs, &total);
  const int64_t n_warps = scan_warps(n_grid, n_edge_runs, form == 1);
  const unsigned grid = (unsigned)((n_warps * 32 + kThreads - 1) / kThreads);
  if (grid > 0) {
    if (form == 1)
      launch_k(sdf_reg_runs_kernel<true>, grid, (unsigned)kThreads, st, kLaunchStream, sdf, reinterpret_cast<const int2*>(edge_runs),
               edge_run_chunk, n_edge_runs, w, g_loss, g_sdf);
    else
      launch_k(sdf_reg_rows_kernel<true>, grid, (unsigned)kThreads, st, kLaunchStream, sdf, n_grid, edge_rows, edge_row_off, w, g_loss,
               g_sdf);
  }
  return sdf_reg_done("d3h_sdf_reg_backward");
}
