// Stage 3: per-polygon work on the O(surface) records.
//
//   poly_faces_kernel : watertight faces from triangle_table (gshell_tets.py:322-325), face normals / tangents
//                       splatted to the watertight vertices (auto_normals :9-34, compute_tangents :40-78 with the
//                       "UV indexed by vertex id" quirk of :327), mSDF cut case per polygon (:338-339, :401-404) and
//                       the number of polygons per faces_aug bucket in every 256-polygon tile.  The last CTA to finish
//                       scans those tile counts and PUBLISHES the final sizes of the call to the host (d3h_counts in
//                       mapped pinned memory): the host wakes up while the kernel below is still running.
//   poly_cut_kernel   : per-corner vertex frame (normalised normal, averaged + Gram-Schmidt tangent, :28-29, :69-73),
//                       boundary vertices on every polygon edge (:342-397), zeroing of unreferenced rows (:423-427),
//                       faces_aug emission in the reference's 6-bucket order (:406-420) from in-tile ballot ranks.
#include "d3h_internal.cuh"

namespace d3h {

struct UvParams {
  int nuv;      // ceil(sqrt(F)), gshell_tets.py:220 with max_idx = 2F
  float step;   // linspace step, end / (nuv - 1) in fp32
  float end;    // fp32(1 - 1/nuv)
  float pad;    // fp32(0.9 / nuv), :226
};

// torch.linspace(0, 1 - 1/nuv, nuv)[i] as ATen's CPU kernel evaluates it: lower half start + step*i, upper half
// end - step*(n-1-i) with a single rounding (vectorised fmadd); pinned against torch in the oracle tests.
__device__ __forceinline__ float uv_lin(const UvParams& p, int i) {
  return (i < p.nuv / 2) ? __fmul_rn(p.step, (float)i) : __fmaf_rn(-p.step, (float)(p.nuv - 1 - i), p.end);
}
// UV the reference reads for *vertex id* k (uvs_pre[faces], :327 -> :228-233)
__device__ __forceinline__ float2 vertex_uv(const UvParams& p, int k) {
  const int cell = k >> 2, c = k & 3;
  const int ix = cell % p.nuv, iy = cell / p.nuv;
  float u = uv_lin(p, ix), v = uv_lin(p, iy);
  if (c == 1 || c == 2) u = __fadd_rn(u, p.pad);
  if (c == 2 || c == 3) v = __fadd_rn(v, p.pad);
  return make_float2(u, v);
}

__device__ __forceinline__ int pos_in_loop(int code, int edge) {
  int r = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (c_loop_edge[code][k] == edge) r = k;
  return r;
}

// torch.cross on CPU: component = fma(a_i, b_j, -fl(a_j * b_i)) (pinned in the oracle tests)
__device__ __forceinline__ float cross_comp(float ai, float bj, float aj, float bi) {
  return __fmaf_rn(ai, bj, -__fmul_rn(aj, bi));
}

// mSDF cut case of a polygon from the interpolated mSDF at its corners (gshell_tets.py:338-339, 401-404) and the
// faces_aug bucket it lands in: tri polygons cut into 1,2 triangles -> buckets 0,1; quad into 1..4 -> buckets 2..5.
__device__ __forceinline__ int cut_case(bool quad, float m0, float m1, float m2, float m3, unsigned& mcase, int& ncut) {
  const unsigned mo0 = m0 > 0.f, mo1 = m1 > 0.f, mo2 = m2 > 0.f, mo3 = m3 > 0.f;
  if (quad) {
    mcase = (mo0 << 3) | (mo1 << 2) | (mo2 << 1) | mo3;
    ncut = c_num_cut_quad[mcase];
    return ncut ? (1 + ncut) : -1;
  }
  mcase = (mo0 << 2) | (mo1 << 1) | mo2;
  ncut = c_num_cut_tri[mcase];
  return ncut ? (ncut - 1) : -1;
}

// poly_cut_kernel: four lanes per polygon (lane k = corner k; the fourth lane of a triangle polygon idles): a 256-thread
// CTA takes 64 polygons = two of poly_faces_kernel's 32-polygon groups.  Every lane evaluates ONE vertex frame and ONE
// boundary vertex and writes at most one cut triangle; the values of the neighbouring corner travel by warp shuffles.
// (v1 gave a whole polygon to one thread: four vertex frames in sequence on 226 CTAs, 14 us for 58 k polygons.)
constexpr int kCutPolysPerCta = kPolyThreads / 4;

// cut tables as shared-memory words (the case code differs from lane to lane: __constant__ would serialise)
struct CutTables {
  unsigned long long quad[16];   // 12 locals x 4 bits
  unsigned tri[8];               //  6 locals x 4 bits
  unsigned char nq[16], nt[8];   // number of cut triangles
  unsigned char uq[16], ut[8];   // locals referenced by the cut triangles (bit mask)
};

__device__ __forceinline__ void load_cut_tables(CutTables& T) {
  const unsigned t = threadIdx.x;
  if (t < 16u) {
    unsigned long long w = 0ull;
    unsigned used = 0u;
    const int n = c_num_cut_quad[t];
    for (int e = 0; e < 12; ++e) {
      const int loc = c_cut_quad[t][e];
      w |= (unsigned long long)(loc & 0xf) << (4 * e);
      if (e < 3 * n) used |= 1u << loc;
    }
    T.quad[t] = w; T.nq[t] = (unsigned char)n; T.uq[t] = (unsigned char)used;
  } else if (t < 24u) {
    const unsigned c = t - 16u;
    unsigned w = 0u, used = 0u;
    const int n = c_num_cut_tri[c];
    for (int e = 0; e < 6; ++e) {
      const int loc = c_cut_tri[c][e];
      w |= (unsigned)(loc & 0xf) << (4 * e);
      if (e < 3 * n) used |= 1u << loc;
    }
    T.tri[c] = w; T.nt[c] = (unsigned char)n; T.ut[c] = (unsigned char)used;
  }
}

// what the topology CTAs of poly_cut_kernel write for one frame
struct CutOut {
  int64_t* faces_aug;
  float* verts_aug;
  float* msdf_aug;
  int64_t cap_faces_aug, cap_verts_aug;
};

// REPLAY = second extraction of a cloth / body pair (d3h_forward_args.pair_*): `blk` is the pair's argument block (its
// outputs, the opposite msdf_negate), the interpolated mSDF of every vertex is the exact negation of the stored one,
// normals / tangents were accumulated by the first extraction and are not splatted again.
//
// Both surface kernels have two kinds of CTAs.  Frames that share sdf and msdf share one topology (BatchCtx), and all of
// a polygon that follows from its corner ids and the interpolated mSDF alone -- the corner ids on the tape, the watertight
// faces, the mSDF cut case, the rank in its faces_aug bucket, the faces_aug rows, the boundary mSDF -- is the same for each
// of them.  CTAs [0, topo_ctas) of a row are TOPOLOGY CTAs: they do that work once per topology and store the result into
// every frame of the launch that uses it.  When all `topo_rows` rows of the launch share one topology they split its tiles
// (row r takes tiles [r * topo_ctas, (r + 1) * topo_ctas)); otherwise topo_rows = 1 and every row does its own.  The
// other CTAs of a row are the frame's own and do only what needs its positions: normals, tangents, boundary vertices.
// resident CTAs per SM the compiler has to leave room for (register cap): A/B by -D at build time
#ifndef D3H_FACES_MINB
#define D3H_FACES_MINB 4   // 64 registers instead of 80
#endif
#ifndef D3H_CUT_MINB
#define D3H_CUT_MINB 5     // 48 registers, no spill: five CTAs per SM (4 allows 49 and leaves four)
#endif

// vertex id of a corner on the static edge table paths = number of marked edges before its edge in the static edge list
__device__ __forceinline__ int edge_vertex(const unsigned* __restrict__ edge_bits, const unsigned* __restrict__ word_prefix,
                                           unsigned r) {
  return (int)(__ldcg(word_prefix + (r >> 5)) + __popc(__ldcg(edge_bits + (r >> 5)) & ((1u << (r & 31u)) - 1u)));
}

// corner ids of a polygon: on the tape ([3*T1 | 4*T2], gshell_tets.py:406-407), or from the static edge ranks
__device__ __forceinline__ void polygon_corners(bool static_edges, const int32_t* __restrict__ corners,
                                                const unsigned* __restrict__ corner_rank, const unsigned* __restrict__ edge_bits,
                                                const unsigned* __restrict__ word_prefix, int64_t i, int64_t p0, int n,
                                                int (&L)[4]) {
  if (static_edges) {
    const uint4 rk = __ldcg(reinterpret_cast<const uint4*>(corner_rank) + i);
    const unsigned rr[4] = {rk.x, rk.y, rk.z, rk.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) L[k] = (k < n) ? edge_vertex(edge_bits, word_prefix, rr[k]) : 0;
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) L[k] = (k < n) ? corners[p0 + k] : 0;
  }
}

// the watertight triangle t of a polygon: its corners in face order (select without dynamic register indexing)
template <typename T>
__device__ __forceinline__ void triangle_corners(int code, int t, const T (&in)[4], T (&out)[3]) {
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int lp = pos_in_loop(code, c_tri_edge[code][3 * t + c]);
    out[c] = lp == 0 ? in[0] : lp == 1 ? in[1] : lp == 2 ? in[2] : in[3];
  }
}

template <bool REPLAY>
__global__ void __launch_bounds__(kPolyThreads, D3H_FACES_MINB)
poly_faces_kernel(const FwdBlock* __restrict__ blk, const d3h_tet_record* __restrict__ records,
                  DevCounters* __restrict__ ctr, const float4* __restrict__ w_vert, float* __restrict__ w_acc,
                  unsigned* __restrict__ poly_cnt, unsigned* __restrict__ poly_gcnt, unsigned* __restrict__ poly_excl,
                  unsigned char* __restrict__ poly_used, UvParams uvp,
                  d3h_counts* __restrict__ counts_dev, const unsigned* __restrict__ corner_rank,
                  const unsigned* __restrict__ edge_bits, const unsigned* __restrict__ word_prefix, unsigned topo_ctas,
                  unsigned topo_rows, const __grid_constant__ FrameSet fs, const __grid_constant__ FrameSet topo) {
  pdl_enter();
  constexpr int WARPS = kPolyThreads / 32;
  const int64_t shift = fs.off[blockIdx.y], tshift = topo.off[blockIdx.y];
  // the topology: records, corner ids (on the tape of its frame) and static edge ranks
  records = frame_ptr(records, tshift);
  corner_rank = frame_ptr(corner_rank, tshift); edge_bits = frame_ptr(edge_bits, tshift);
  word_prefix = frame_ptr(word_prefix, tshift);
  const FwdBlock* __restrict__ tblk = frame_ptr(blk, tshift);
  int32_t* __restrict__ corners = tblk->a.tape_corners;
  // a replay finds the corner array on the tape, and so does the edge-scan path (scan_emit_kernel wrote it)
  const bool static_edges = !REPLAY && tblk->a.edge_off != nullptr && tblk->a.etets == nullptr;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;

  if (blockIdx.x >= topo_ctas) {
    // ---- the frame's own CTAs: face normals / tangents of its positions, splatted to the watertight vertices ----
    if (REPLAY) return;   // (not launched: normals / tangents were accumulated by the first extraction of the pair)
    const DevCounters* __restrict__ fc = frame_ptr(ctr, shift);
    w_vert = frame_ptr(w_vert, shift); w_acc = frame_ptr(w_acc, shift);
    const unsigned t1 = fc->work_tri, t2 = fc->work_quad;
    unsigned long long* tr = trace_begin(fc->trace, fc->trace_frame, K_POLY_FACES);
    const int64_t npoly = (int64_t)t1 + t2;
    const int64_t i = (int64_t)(blockIdx.x - topo_ctas) * kPolyThreads + threadIdx.x;
    const bool cross_quirk = ((int64_t)t1 + 2ll * t2 == 3);  // torch.cross without dim on a (3,3) tensor, gshell_tets.py:19
    if (i < npoly) {
      const int4 meta = reinterpret_cast<const int4*>(records + i)[1];
      const int code = meta.x, rank = meta.y;
      const bool quad = __popc((unsigned)code) == 2;
      const int n = quad ? 4 : 3;
      const int64_t p0 = quad ? (3ll * t1 + 4ll * rank) : 3ll * rank;
      int L[4];
      float4 P[4];
      polygon_corners(static_edges, corners, corner_rank, edge_bits, word_prefix, i, p0, n, L);
#pragma unroll
      for (int k = 0; k < 4; ++k) P[k] = (k < n) ? w_vert[L[k]] : make_float4(0.f, 0.f, 0.f, 0.f);
      const int ntri = quad ? 2 : 1;
      for (int t = 0; t < ntri; ++t) {
        int vi[3];
        float4 pv[3];
        triangle_corners(code, t, L, vi);
        triangle_corners(code, t, P, pv);
        const float ax = __fsub_rn(pv[1].x, pv[0].x), ay = __fsub_rn(pv[1].y, pv[0].y), az = __fsub_rn(pv[1].z, pv[0].z);
        const float bx = __fsub_rn(pv[2].x, pv[0].x), by = __fsub_rn(pv[2].y, pv[0].y), bz = __fsub_rn(pv[2].z, pv[0].z);
        // accumulator row of a vertex: [nx ny nz count | tx ty tz -]; one 16-byte vector atomic per half (sm_90+)
        float nx = 0.f, ny = 0.f, nz = 0.f;
        if (!cross_quirk) {
          nx = cross_comp(ay, bz, az, by);
          ny = cross_comp(az, bx, ax, bz);
          nz = cross_comp(ax, by, ay, bx);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c)
          atomicAdd(reinterpret_cast<float4*>(w_acc + 8ll * vi[c]), make_float4(nx, ny, nz, 1.f));
        // tangent of this face
        const float2 uv0 = vertex_uv(uvp, vi[0]), uv1 = vertex_uv(uvp, vi[1]), uv2 = vertex_uv(uvp, vi[2]);
        const float u1x = __fsub_rn(uv1.x, uv0.x), u1y = __fsub_rn(uv1.y, uv0.y);
        const float u2x = __fsub_rn(uv2.x, uv0.x), u2y = __fsub_rn(uv2.y, uv0.y);
        float den = __fsub_rn(__fmul_rn(u1x, u2y), __fmul_rn(u1y, u2x));
        den = (den > 0.f) ? fmaxf(den, 1e-6f) : fminf(den, -1e-6f);
        const float tx = __fdiv_rn(__fsub_rn(__fmul_rn(ax, u2y), __fmul_rn(bx, u1y)), den);
        const float ty = __fdiv_rn(__fsub_rn(__fmul_rn(ay, u2y), __fmul_rn(by, u1y)), den);
        const float tz = __fdiv_rn(__fsub_rn(__fmul_rn(az, u2y), __fmul_rn(bz, u1y)), den);
#pragma unroll
        for (int c = 0; c < 3; ++c)
          atomicAdd(reinterpret_cast<float4*>(w_acc + 8ll * vi[c]) + 1, make_float4(tx, ty, tz, 0.f));
      }
    }
    // the (3,3) torch.cross quirk: the three face normals are crossed along the *face* axis
    if (cross_quirk && i == 0) {
      float a[3][3], b[3][3];
      int fv[3][3];
      for (int64_t q = 0; q < npoly; ++q) {
        const int4 meta = reinterpret_cast<const int4*>(records + q)[1];
        const int code = meta.x, rank = meta.y;
        const bool quad = __popc((unsigned)code) == 2;
        const int64_t p0 = quad ? (3ll * t1 + 4ll * rank) : 3ll * rank;
        for (int t = 0; t < (quad ? 2 : 1); ++t) {
          const int64_t row = quad ? ((int64_t)t1 + 2ll * rank + t) : (int64_t)rank;
          float4 pv[3];
          for (int c = 0; c < 3; ++c) {
            const int kk = pos_in_loop(code, c_tri_edge[code][3 * t + c]);
            fv[row][c] = static_edges ? edge_vertex(edge_bits, word_prefix, __ldcg(corner_rank + 4 * q + kk)) : corners[p0 + kk];
            pv[c] = w_vert[fv[row][c]];
          }
          a[row][0] = __fsub_rn(pv[1].x, pv[0].x); a[row][1] = __fsub_rn(pv[1].y, pv[0].y); a[row][2] = __fsub_rn(pv[1].z, pv[0].z);
          b[row][0] = __fsub_rn(pv[2].x, pv[0].x); b[row][1] = __fsub_rn(pv[2].y, pv[0].y); b[row][2] = __fsub_rn(pv[2].z, pv[0].z);
        }
      }
      for (int c = 0; c < 3; ++c) {  // column c: vectors (a[0][c], a[1][c], a[2][c]) x (b[0][c], b[1][c], b[2][c])
        float fn[3];
        fn[0] = cross_comp(a[1][c], b[2][c], a[2][c], b[1][c]);
        fn[1] = cross_comp(a[2][c], b[0][c], a[0][c], b[2][c]);
        fn[2] = cross_comp(a[0][c], b[1][c], a[1][c], b[0][c]);
        for (int r = 0; r < 3; ++r)
          for (int k = 0; k < 3; ++k) atomicAdd(w_acc + 8ll * fv[r][k] + c, fn[r]);  // counts were added above
      }
    }
    if (tr != nullptr) __syncthreads();
    trace_end(tr);
    return;
  }

  // ---- topology CTAs: corner ids and watertight faces of every frame, mSDF cut case and the polygons per faces_aug
  // bucket of every group and tile (poly_cut_kernel ranks with them); the last one out scans the tiles and publishes ----
  DevCounters* __restrict__ tc = frame_ptr(ctr, tshift);
  w_vert = frame_ptr(w_vert, tshift);
  poly_cnt = frame_ptr(poly_cnt, tshift); poly_gcnt = frame_ptr(poly_gcnt, tshift); poly_excl = frame_ptr(poly_excl, tshift);
  poly_used = frame_ptr(poly_used, tshift);
  __shared__ unsigned s_cnt[8][WARPS];
  __shared__ unsigned s_last;
  __shared__ unsigned long long s_scan[3][32];
  __shared__ CutTables s_tab;
  __shared__ int32_t* s_corners[kMaxFused];   // outputs of the frames of this topology
  __shared__ int64_t* s_fwt[kMaxFused];
  __shared__ int64_t s_cap_fwt[kMaxFused];
  __shared__ int s_nf;
  load_cut_tables(s_tab);
  if (threadIdx.x == 32) {
    int nf = 0;
    for (unsigned f = 0; f < gridDim.y; ++f) {
      if (topo.off[f] != tshift) continue;
      const FwdBlock* b = frame_ptr(blk, fs.off[f]);
      s_corners[nf] = b->a.tape_corners; s_fwt[nf] = b->a.faces_wt; s_cap_fwt[nf] = b->a.cap_faces_wt;
      ++nf;
    }
    s_nf = nf;
  }
  __syncthreads();
  const int nf = s_nf;
  const unsigned t1 = tc->work_tri, t2 = tc->work_quad;
  unsigned long long* tr = trace_begin(tc->trace, tc->trace_frame, K_POLY_FACES);
  const int64_t npoly = (int64_t)t1 + t2;
  const int64_t ntiles = (npoly + kPolyThreads - 1) / kPolyThreads;
  const unsigned ntopo = topo_rows * topo_ctas;
  const unsigned tile = (blockIdx.y % topo_rows) * topo_ctas + blockIdx.x;
  // CTAs past the data still take part in the "last CTA out" count (the grid is sized from the capacity)
  const int64_t i = (int64_t)tile * kPolyThreads + threadIdx.x;

  if ((int64_t)tile < ntiles) {
    int bucket = -1;
    if (i < npoly) {
      const int4 meta = reinterpret_cast<const int4*>(records + i)[1];
      const int code = meta.x, rank = meta.y;
      const bool quad = __popc((unsigned)code) == 2;
      const int n = quad ? 4 : 3;
      const int64_t p0 = quad ? (3ll * t1 + 4ll * rank) : 3ll * rank;
      int L[4];
      float m[4];
      polygon_corners(static_edges, corners, corner_rank, edge_bits, word_prefix, i, p0, n, L);
      // the corner array of every frame's tape (poly_cut_kernel and the backward pass read it there)
      for (int f = 0; f < nf; ++f) {
        int32_t* __restrict__ dst = s_corners[f];
        if (static_edges || dst != corners) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (k < n) dst[p0 + k] = L[k];
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) m[k] = (k < n) ? reinterpret_cast<const float*>(w_vert + L[k])[3] : 0.f;
      // ---- watertight faces ----
      const int ntri = quad ? 2 : 1;
      for (int t = 0; t < ntri; ++t) {
        const int64_t row = quad ? ((int64_t)t1 + 2ll * rank + t) : (int64_t)rank;
        int vi[3];
        triangle_corners(code, t, L, vi);
        for (int f = 0; f < nf; ++f) {
          if (row < s_cap_fwt[f]) {
            int64_t* __restrict__ faces_wt = s_fwt[f];
            faces_wt[3 * row + 0] = vi[0];
            faces_wt[3 * row + 1] = vi[1];
            faces_wt[3 * row + 2] = vi[2];
          }
        }
      }
      unsigned mcase;
      int ncut;
      const float sg = REPLAY ? -1.f : 1.f;  // exact: the pair's interpolated mSDF is the negation (SURVEY A.4)
      bucket = cut_case(quad, sg * m[0], sg * m[1], sg * m[2], sg * m[3], mcase, ncut);
      // boundary vertices the cut references (bit k: the one on polygon edge k -> k+1), for the frames' poly_cut CTAs
      poly_used[i] = (unsigned char)(((quad ? s_tab.uq[mcase] : s_tab.ut[mcase]) >> n) & 0xfu);
    }
    // ---- polygons per bucket: per group of 32 polygons (one warp; poly_cut_kernel ranks inside a tile with them) and
    // per tile of 256 (scanned below by the last CTA).  Lane b keeps the count of bucket b ----
    unsigned mine = 0u;
#pragma unroll
    for (int b = 0; b < 6; ++b) {
      const unsigned msk = __ballot_sync(0xffffffffu, bucket == b);
      if (lane == (unsigned)b) mine = __popc(msk);
    }
    if (lane < 8u) {   // (entries 6, 7: zero)
      poly_gcnt[((int64_t)tile * WARPS + warp) * 8 + lane] = mine;
      s_cnt[lane][warp] = mine;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
      unsigned run = 0;
#pragma unroll
      for (int w = 0; w < WARPS; ++w) run += s_cnt[threadIdx.x][w];
      poly_cnt[(int64_t)tile * 8 + threadIdx.x] = run;
    }
  }

  // ---- last topology CTA out: scan the tile counts, finalise and publish the sizes of every frame of the topology ----
  __threadfence();
  __syncthreads();
  trace_end(tr);
  if (threadIdx.x == 0) s_last = (atomicAdd(REPLAY ? &tc->poly_done2 : &tc->poly_done, 1u) == ntopo - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // thread t owns tiles [t*per, (t+1)*per); buckets are scanned as three pairs packed in 64-bit words
  const int64_t per = (ntiles + kPolyThreads - 1) / kPolyThreads;
  const int64_t tl0 = (int64_t)threadIdx.x * per;
  unsigned long long sum[3] = {0ull, 0ull, 0ull};
  for (int64_t q = 0; q < per; ++q) {
    if (tl0 + q < ntiles) {
      const uint4 c03 = __ldcg(reinterpret_cast<const uint4*>(poly_cnt + (tl0 + q) * 8));
      const uint2 c45 = __ldcg(reinterpret_cast<const uint2*>(poly_cnt + (tl0 + q) * 8 + 4));
      sum[0] += (unsigned long long)c03.x | ((unsigned long long)c03.y << 32);
      sum[1] += (unsigned long long)c03.z | ((unsigned long long)c03.w << 32);
      sum[2] += (unsigned long long)c45.x | ((unsigned long long)c45.y << 32);
    }
  }
  unsigned long long incl[3], run[3], total[3];
#pragma unroll
  for (int wd = 0; wd < 3; ++wd) {
    incl[wd] = sum[wd];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long nb = __shfl_up_sync(0xffffffffu, incl[wd], o);
      if (lane >= (unsigned)o) incl[wd] += nb;
    }
    if (lane == 31) s_scan[wd][warp] = incl[wd];
  }
  __syncthreads();
#pragma unroll
  for (int wd = 0; wd < 3; ++wd) {
    unsigned long long wpre = 0ull, tot = 0ull;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) {
      if (w < (int)warp) wpre += s_scan[wd][w];
      tot += s_scan[wd][w];
    }
    run[wd] = wpre + incl[wd] - sum[wd];
    total[wd] = tot;
  }
  for (int64_t q = 0; q < per; ++q) {
    if (tl0 + q < ntiles) {
      const uint4 c03 = __ldcg(reinterpret_cast<const uint4*>(poly_cnt + (tl0 + q) * 8));
      const uint2 c45 = __ldcg(reinterpret_cast<const uint2*>(poly_cnt + (tl0 + q) * 8 + 4));
      unsigned* e = poly_excl + (tl0 + q) * 8;
      e[0] = (unsigned)run[0]; e[1] = (unsigned)(run[0] >> 32);
      e[2] = (unsigned)run[1]; e[3] = (unsigned)(run[1] >> 32);
      e[4] = (unsigned)run[2]; e[5] = (unsigned)(run[2] >> 32);
      run[0] += (unsigned long long)c03.x | ((unsigned long long)c03.y << 32);
      run[1] += (unsigned long long)c03.z | ((unsigned long long)c03.w << 32);
      run[2] += (unsigned long long)c45.x | ((unsigned long long)c45.y << 32);
    }
  }
  // thread f publishes frame f of the launch (if it uses this topology)
  if (threadIdx.x < gridDim.y && topo.off[threadIdx.x] == tshift) {
    const int64_t off = fs.off[threadIdx.x];
    DevCounters* __restrict__ fc = frame_ptr(ctr, off);
    const FwdBlock* __restrict__ fb = frame_ptr(blk, off);
    unsigned bk[6];
#pragma unroll
    for (int wd = 0; wd < 3; ++wd) {
      bk[2 * wd] = (unsigned)total[wd];
      bk[2 * wd + 1] = (unsigned)(total[wd] >> 32);
    }
    const int ncut_of[6] = {1, 2, 1, 2, 3, 4};
    int64_t fa = 0;
    d3h_counts c;
    for (int b = 0; b < 6; ++b) {
      if (REPLAY) fc->bucket2[b] = bk[b]; else fc->bucket[b] = bk[b];
      c.bucket_polys[b] = bk[b];
      fa += (int64_t)bk[b] * ncut_of[b];
    }
    c.n_valid_tets = fc->n_valid;
    c.n_tri_tets = fc->n_tri;
    c.n_quad_tets = fc->n_quad;
    c.n_corners = 3ll * fc->n_tri + 4ll * fc->n_quad;
    c.n_verts = fc->n_verts;
    c.n_faces_aug = fa;
    c.bad_index = 0;
    c.overflow = (fc->n_valid != fc->work_tri + fc->work_quad) ? 1 : 0;  // record buffer overflowed: surface stages skipped
    const int64_t seq = fb->a.seq;
    d3h_counts* counts_mapped = fb->counts_mapped;
    c.seq = seq;
    c.reserved = 0;
    *frame_ptr(counts_dev, off) = c;
    if (counts_mapped != nullptr) {  // straight into pinned host memory; `seq` last, after a system-scope fence
      volatile int64_t* dst = reinterpret_cast<volatile int64_t*>(counts_mapped);
      const int64_t* src = reinterpret_cast<const int64_t*>(&c);
      constexpr int kSeqWord = (int)(offsetof(d3h_counts, seq) / 8);
      for (int w = 0; w < (int)(sizeof(d3h_counts) / 8); ++w)
        if (w != kSeqWord) dst[w] = src[w];
      __threadfence_system();
      dst[kSeqWord] = seq;
    }
  }
}

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float3 safe_normalize3(float x, float y, float z) {  // render/util.py:25-29
  const float d = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
  const float len = __fsqrt_rn(fmaxf(d, 1e-20f));
  return make_float3(__fdiv_rn(x, len), __fdiv_rn(y, len), __fdiv_rn(z, len));
}

// Tangent of one watertight vertex from its splat accumulators: auto_normals tail (gshell_tets.py:28-29) and
// compute_tangents tail (:69-73).  Every corner of the vertex evaluates the same expression on the same inputs.
__device__ __forceinline__ float3 vertex_tangent(const float* __restrict__ w_acc, int v) {
  const float4 a0 = __ldcg(reinterpret_cast<const float4*>(w_acc + 8ll * v));
  const float4 a1 = __ldcg(reinterpret_cast<const float4*>(w_acc + 8ll * v) + 1);
  float nx = a0.x, ny = a0.y, nz = a0.z;
  const float d = __fadd_rn(__fadd_rn(__fmul_rn(nx, nx), __fmul_rn(ny, ny)), __fmul_rn(nz, nz));
  if (!(d > 1e-20f)) { nx = 0.f; ny = 0.f; nz = 1.f; }
  const float3 n = safe_normalize3(nx, ny, nz);
  const float cnt = a0.w;
  float3 t = safe_normalize3(__fdiv_rn(a1.x, cnt), __fdiv_rn(a1.y, cnt), __fdiv_rn(a1.z, cnt));
  const float dp = __fadd_rn(__fadd_rn(__fmul_rn(t.x, n.x), __fmul_rn(t.y, n.y)), __fmul_rn(t.z, n.z));
  return safe_normalize3(__fsub_rn(t.x, __fmul_rn(dp, n.x)), __fsub_rn(t.y, __fmul_rn(dp, n.y)),
                         __fsub_rn(t.z, __fmul_rn(dp, n.z)));
}

template <bool REPLAY>
__global__ void __launch_bounds__(kPolyThreads, D3H_CUT_MINB)
poly_cut_kernel(const FwdBlock* __restrict__ blk, const d3h_tet_record* __restrict__ records,
                const DevCounters* __restrict__ ctr, const float4* __restrict__ w_vert,
                const float* __restrict__ w_acc, const int32_t* __restrict__ owner,
                const unsigned* __restrict__ poly_gcnt, const unsigned* __restrict__ poly_excl,
                const unsigned char* __restrict__ poly_used, unsigned topo_ctas, unsigned topo_rows,
                const __grid_constant__ FrameSet fs, const __grid_constant__ FrameSet topo) {
  pdl_enter();
  constexpr int WARPS = kPolyThreads / 32;
  constexpr unsigned FULL = 0xffffffffu;
  const int64_t shift = fs.off[blockIdx.y], tshift = topo.off[blockIdx.y];
  records = frame_ptr(records, tshift);   // (shared topology: the first frame's records and corner ids)
  const int32_t* __restrict__ corners = frame_ptr(blk, tshift)->a.tape_corners;
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned k = lane & 3u, lane0 = lane & ~3u;                 // corner of this lane, first lane of its polygon

  if (blockIdx.x >= topo_ctas) {
    // ---- the frame's own CTAs: vertex frames, tangent rows and the boundary vertices' positions and tangents ----
    blk = frame_ptr(blk, shift); ctr = frame_ptr(ctr, shift);
    w_vert = frame_ptr(w_vert, shift); w_acc = frame_ptr(w_acc, shift); owner = frame_ptr(owner, shift);
    poly_used = frame_ptr(poly_used, tshift);
    float* __restrict__ verts_aug = blk->a.verts_aug;
    float* __restrict__ v_tng_aug = blk->a.v_tng_aug;
    float* __restrict__ v_tng_wt = blk->a.v_tng_wt;
    const int64_t cap_verts_aug = blk->a.cap_verts_aug, cap_verts = blk->a.cap_verts;
    const bool static_edges = blk->a.edge_off != nullptr;
    const unsigned t1 = ctr->work_tri, t2 = ctr->work_quad;
    unsigned long long* tr = trace_begin(ctr->trace, ctr->trace_frame, K_POLY_CUT);
    const int64_t npoly = (int64_t)t1 + t2;
    const unsigned tile = blockIdx.x - topo_ctas;
    if ((int64_t)tile * kCutPolysPerCta >= npoly) return;
    const int64_t nv = ctr->n_verts;
    const int64_t i = (int64_t)tile * kCutPolysPerCta + warp * 8 + (lane >> 2);
    bool corner = false;
    int n = 3;
    int64_t p0 = 0;
    unsigned used = 0u;
    float4 P = make_float4(0.f, 0.f, 0.f, 0.f);
    float3 T = make_float3(0.f, 0.f, 0.f);
    if (i < npoly) {
      const int4 meta = reinterpret_cast<const int4*>(records + i)[1];
      const int code = meta.x, rank = meta.y;
      const bool quad = __popc((unsigned)code) == 2;
      n = quad ? 4 : 3;
      p0 = quad ? (3ll * t1 + 4ll * rank) : 3ll * rank;
      corner = (int)k < n;
      if (corner) {
        used = (poly_used[i] >> k) & 1u;
        const int L = corners[p0 + k];
        P = w_vert[L];
        if (REPLAY) P.w = -P.w;  // the pair's interpolated mSDF: exact negation
        T = vertex_tangent(w_acc, L);
        // the corner that opened the vertex's run in the sorted key array writes the vertex's own tangent rows
        // (static edge table paths: no owner is known, every corner writes the same value)
        if (static_edges || owner[L] == (int32_t)(p0 + k)) {
          const int64_t v = L;
          if (v < cap_verts) {
            store_same_value(v_tng_wt + 3 * v, T.x);
            store_same_value(v_tng_wt + 3 * v + 1, T.y);
            store_same_value(v_tng_wt + 3 * v + 2, T.z);
          }
          if (v < cap_verts_aug) {
            store_same_value(v_tng_aug + 3 * v, T.x);
            store_same_value(v_tng_aug + 3 * v + 1, T.y);
            store_same_value(v_tng_aug + 3 * v + 2, T.z);
          }
        }
      }
    }
    // ---- boundary vertex on polygon edge k -> k+1: this lane's corner and the next one's ----
    const unsigned kn = ((int)k + 1 == n) ? 0u : k + 1u;
    const unsigned src = lane0 + (corner ? kn : k);
    float4 Pj;
    float3 Tj;
    Pj.x = __shfl_sync(FULL, P.x, src); Pj.y = __shfl_sync(FULL, P.y, src);
    Pj.z = __shfl_sync(FULL, P.z, src); Pj.w = __shfl_sync(FULL, P.w, src);
    Tj.x = __shfl_sync(FULL, T.x, src); Tj.y = __shfl_sync(FULL, T.y, src); Tj.z = __shfl_sync(FULL, T.z, src);
    if (corner) {
      float u0, u1, D;
      boundary_weights(P.w, Pj.w, u0, u1, D);
      const int64_t row = nv + p0 + k;
      if (row < cap_verts_aug) {
        if (used) {   // (the topology CTAs zero the rows of the others)
          verts_aug[3 * row + 0] = lerp2(P.x, u0, Pj.x, u1);
          verts_aug[3 * row + 1] = lerp2(P.y, u0, Pj.y, u1);
          verts_aug[3 * row + 2] = lerp2(P.z, u0, Pj.z, u1);
        }
        v_tng_aug[3 * row + 0] = lerp2(T.x, u0, Tj.x, u1);
        v_tng_aug[3 * row + 1] = lerp2(T.y, u0, Tj.y, u1);
        v_tng_aug[3 * row + 2] = lerp2(T.z, u0, Tj.z, u1);
      }
    }
    trace_end(tr);
    return;
  }

  // ---- topology CTAs: cut case, rank of the polygon in its bucket, and for every frame of the topology its faces_aug
  // rows, the boundary mSDF and the zero rows of the boundary vertices no cut triangle references ----
  ctr = frame_ptr(ctr, tshift); w_vert = frame_ptr(w_vert, tshift);
  poly_gcnt = frame_ptr(poly_gcnt, tshift); poly_excl = frame_ptr(poly_excl, tshift);
  __shared__ unsigned s_cnt[6][WARPS];
  __shared__ CutTables s_tab;
  __shared__ CutOut s_out[kMaxFused];
  __shared__ int s_nf;
  const unsigned t1 = ctr->work_tri, t2 = ctr->work_quad;
  unsigned long long* tr = trace_begin(ctr->trace, ctr->trace_frame, K_POLY_CUT);
  const int64_t npoly = (int64_t)t1 + t2;
  const unsigned tile = (blockIdx.y % topo_rows) * topo_ctas + blockIdx.x;
  if ((int64_t)tile * kCutPolysPerCta >= npoly) return;
  load_cut_tables(s_tab);
  if (threadIdx.x == 32) {
    int nf = 0;
    for (unsigned f = 0; f < gridDim.y; ++f) {
      if (topo.off[f] != tshift) continue;
      const FwdBlock* b = frame_ptr(blk, fs.off[f]);
      s_out[nf] = CutOut{b->a.faces_aug, b->a.verts_aug, b->a.msdf_aug, b->a.cap_faces_aug, b->a.cap_verts_aug};
      ++nf;
    }
    s_nf = nf;
  }
  const int64_t nv = ctr->n_verts;
  const int64_t i = (int64_t)tile * kCutPolysPerCta + warp * 8 + (lane >> 2);
  const bool live = i < npoly;

  bool quad = false, corner = false;
  int n = 3, L = 0;
  int64_t p0 = 0;
  float m = 0.f;
  if (live) {
    const int4 meta = reinterpret_cast<const int4*>(records + i)[1];
    const int code = meta.x, rank = meta.y;
    quad = __popc((unsigned)code) == 2;
    n = quad ? 4 : 3;
    p0 = quad ? (3ll * t1 + 4ll * rank) : 3ll * rank;
    corner = (int)k < n;
    if (corner) {
      L = corners[p0 + k];
      m = reinterpret_cast<const float*>(w_vert + L)[3];
      if (REPLAY) m = -m;  // the pair's interpolated mSDF: exact negation
    }
  }
  __syncthreads();   // the tables and the outputs
  // ---- mSDF cut case from the four corner signs (gshell_tets.py:338-339, 401-404) ----
  const unsigned mo = (__ballot_sync(FULL, corner && m > 0.f) >> lane0) & 0xfu;   // bit c = corner c
  unsigned mcase;
  int ncut = 0, bucket = -1;
  unsigned used_mask = 0u;
  unsigned long long cut = 0ull;
  if (quad) {
    mcase = ((mo & 1u) << 3) | ((mo & 2u) << 1) | ((mo & 4u) >> 1) | ((mo & 8u) >> 3);
    if (live) { ncut = s_tab.nq[mcase]; used_mask = s_tab.uq[mcase]; cut = s_tab.quad[mcase]; }
    bucket = ncut ? (1 + ncut) : -1;
  } else {
    mcase = ((mo & 1u) << 2) | (mo & 2u) | ((mo & 4u) >> 2);
    if (live) { ncut = s_tab.nt[mcase]; used_mask = s_tab.ut[mcase]; cut = s_tab.tri[mcase]; }
    bucket = ncut ? (ncut - 1) : -1;
  }
  // ---- ordered rank of the polygon inside its bucket: group prefix + warps of the group before + polygons before ----
  unsigned my_ballot = 0;
#pragma unroll
  for (int b = 0; b < 6; ++b) {
    const unsigned msk = __ballot_sync(FULL, bucket == b && k == 0u);
    if (bucket == b) my_ballot = msk;
    if (lane == 0) s_cnt[b][warp] = __popc(msk);
  }
  __syncthreads();
  int64_t row0 = 0;
  if (bucket >= 0) {
    const int ncut_of[6] = {1, 2, 1, 2, 3, 4};
    int64_t fbase = 0;
#pragma unroll
    for (int b = 0; b < 6; ++b)
      if (b < bucket) fbase += (int64_t)(REPLAY ? ctr->bucket2[b] : ctr->bucket[b]) * ncut_of[b];
    // polygons of this bucket before this one: tiles of 256 before (scanned by poly_faces_kernel), groups of 32 before
    // inside the tile, warps of this kernel before inside the group (4 warps = one group)
    const int64_t grp = i >> 5;
    unsigned before = poly_excl[(grp >> 3) * 8 + bucket];
    for (int64_t q = grp & ~int64_t(7); q < grp; ++q) before += __ldg(poly_gcnt + q * 8 + bucket);
    for (unsigned w = warp & ~3u; w < warp; ++w) before += s_cnt[bucket][w];
    row0 = fbase + ((int64_t)before + __popc(my_ballot & ((1u << lane0) - 1u))) * ncut;   // polygons before this one
  }
  const int nf = s_nf;
  // ---- boundary vertex on polygon edge k -> k+1: its mSDF, and a zero row where no cut triangle references it ----
  const unsigned kn = ((int)k + 1 == n) ? 0u : k + 1u;
  const float mj = __shfl_sync(FULL, m, lane0 + (corner ? kn : k));
  if (corner) {
    float u0, u1, D;
    boundary_weights(m, mj, u0, u1, D);
    const int64_t row = nv + p0 + k;
    const bool used = (used_mask >> (n + k)) & 1u;
    const float mb = lerp2(m, u0, mj, u1);
    for (int f = 0; f < nf; ++f) {
      const CutOut o = s_out[f];
      if (row < o.cap_verts_aug) {
        if (!used) {
          o.verts_aug[3 * row + 0] = 0.f;
          o.verts_aug[3 * row + 1] = 0.f;
          o.verts_aug[3 * row + 2] = 0.f;
        }
        o.msdf_aug[row] = mb;
      }
    }
  }
  // ---- cut triangles: lane k writes triangle k of its polygon ----
  const bool tri_here = (int)k < ncut;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int loc = (int)((cut >> (4 * (3 * k + c))) & 0xfull);
    const bool is_corner = tri_here && loc < n;
    const int Lv = __shfl_sync(FULL, L, lane0 + (is_corner ? (unsigned)loc : k));
    if (tri_here) {
      const int64_t g = is_corner ? (int64_t)Lv : nv + p0 + (loc - n);
      const int64_t frow = row0 + k;
      for (int f = 0; f < nf; ++f)
        if (frow < s_out[f].cap_faces_aug) s_out[f].faces_aug[3 * frow + c] = g;
    }
  }
  trace_end(tr);
}

// Sizes of a call whose surface stages do not run at all (cap_valid_tets == 0: counting run).
__global__ void publish_counts_kernel(const FwdBlock* __restrict__ blk, const DevCounters* __restrict__ ctr,
                                      d3h_counts* __restrict__ counts_dev) {
  const int64_t seq = blk->a.seq;
  d3h_counts* counts_mapped = blk->counts_mapped;
  d3h_counts c;
  memset(&c, 0, sizeof(c));
  c.n_valid_tets = ctr->n_valid;
  c.n_tri_tets = ctr->n_tri;
  c.n_quad_tets = ctr->n_quad;
  c.n_corners = 3ll * ctr->n_tri + 4ll * ctr->n_quad;
  c.overflow = (ctr->n_valid != ctr->work_tri + ctr->work_quad) ? 1 : 0;
  c.seq = seq;
  *counts_dev = c;
  if (counts_mapped != nullptr) {
    volatile int64_t* dst = reinterpret_cast<volatile int64_t*>(counts_mapped);
    const int64_t* src = reinterpret_cast<const int64_t*>(&c);
    constexpr int kSeqWord = (int)(offsetof(d3h_counts, seq) / 8);
    for (int w = 0; w < (int)(sizeof(d3h_counts) / 8); ++w)
      if (w != kSeqWord) dst[w] = src[w];
    __threadfence_system();
    dst[kSeqWord] = seq;
  }
}

// ------------------------------------------------------------------------------------------------
static UvParams uv_params(int64_t n_tets) {
  UvParams uvp;
  // map_uv(face_gidx_pre, num_tets*2): N = int(ceil(sqrt((max_idx+1)//2))), gshell_tets.py:220,319
  const int64_t half = (2 * n_tets + 1) / 2;
  uvp.nuv = (int)ceil(sqrt((double)half));
  if (uvp.nuv < 1) uvp.nuv = 1;
  uvp.end = (float)(1.0 - (1.0 / (double)uvp.nuv));
  uvp.step = (uvp.nuv > 1) ? uvp.end / (float)(uvp.nuv - 1) : 0.f;
  uvp.pad = (float)(0.9 / (double)uvp.nuv);
  return uvp;
}

static unsigned cut_blocks(const Workspace& ws) {
  const int64_t n = (ws.cap_tets + kCutPolysPerCta - 1) / kCutPolysPerCta;
  return (unsigned)(n > 0 ? n : 1);
}

// Rows of the launch that split the tiles of one topology (all of them when the frames share it, see poly_faces_kernel),
// and the topology CTAs each of them takes out of `tiles`.
static unsigned topo_rows() {
  const BatchCtx& ctx = batch_ctx();
  return ctx.topo_frames == 1 ? (unsigned)ctx.frames : 1u;
}
static unsigned topo_ctas(unsigned tiles, unsigned rows) { return (tiles + rows - 1) / rows; }

void launch_surface(const d3h_forward_args& a, const Workspace& ws, const d3h_tet_record* records,
                    cudaStream_t stream) {
  const UvParams uvp = uv_params(a.n_tets);
  if (ws.cap_tets <= 0) {
    ProfScope ps(K_POLY_FACES, stream);
    launch_k(publish_counts_kernel, 1u, 1u, stream, kLaunchLatency, ws.blk, ws.ctr, ws.counts);
    return;
  }
  const unsigned rows = topo_rows();
  const unsigned nblk = (unsigned)(ws.ntiles_poly > 0 ? ws.ntiles_poly : 1), ncut = cut_blocks(ws);
  const unsigned tfaces = topo_ctas(nblk, rows), tcut = topo_ctas(ncut, rows);
  {
    ProfScope ps(K_POLY_FACES, stream);
    launch_k_dep(poly_faces_kernel<false>, tfaces + nblk, (unsigned)kPolyThreads, stream, kLaunchLatency, ws.blk, records,
                 ws.ctr, ws.vert, ws.acc, ws.poly_cnt, ws.poly_gcnt, ws.poly_excl, ws.poly_used, uvp, ws.counts,
                 ws.corner_rank, ws.edge_bits, ws.word_prefix, tfaces, rows, batch_ctx().fs, batch_ctx().topo);
  }
  ProfScope ps(K_POLY_CUT, stream);
  launch_k_dep(poly_cut_kernel<false>, tcut + ncut, (unsigned)kPolyThreads, stream, kLaunchLatency, ws.blk, records, ws.ctr,
               ws.vert, ws.acc, ws.owner, ws.poly_gcnt, ws.poly_excl, ws.poly_used, tcut, rows, batch_ctx().fs,
               batch_ctx().topo);
}

// ------------------------------------------------------------------------------------------------
// tangent branch of the backward pass (d3h_tangent_backward; optional, SURVEY A.5)
//
// workspace rows, 16 floats per watertight vertex:  [0..2] sum of face normals N   [3] face count c
//   [4..6] sum of face tangents S   [8..10] upstream gradient of the final tangent g_T   [12..14] g_N   -- then reused:
//   [4..6] g_S after the vertex pass.  g_mvert / g_verts are the outputs.
// Per-vertex chain in double: the gradients of the normalisations divide by |N| and |W| (small where faces cancel).
// ------------------------------------------------------------------------------------------------
struct TngArgs {
  d3h_tangent_backward_args a;
  float* ws;
  UvParams uvp;
};

// boundary vertices (gshell_tets.py:380-385): thread per polygon, rows V + p0 + k of v_tng_aug
__global__ void __launch_bounds__(256) tng_boundary_kernel(TngArgs g) {
  const d3h_tangent_backward_args& a = g.a;
  const int64_t t1 = a.n_tri_tets, npoly = a.n_tri_tets + a.n_quad_tets;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npoly) return;
  const bool quad = i >= t1;
  const int n = quad ? 4 : 3;
  const int64_t p0 = quad ? (3 * t1 + 4 * (i - t1)) : 3 * i;
  for (int k = 0; k < n; ++k) {
    const int kn = (k + 1 == n) ? 0 : k + 1;
    const int vi = __ldg(a.tape_corners + p0 + k), vj = __ldg(a.tape_corners + p0 + kn);
    const int64_t row = a.n_verts + p0 + k;
    const float gx = __ldg(a.g_tng_aug + 3 * row), gy = __ldg(a.g_tng_aug + 3 * row + 1), gz = __ldg(a.g_tng_aug + 3 * row + 2);
    if (gx == 0.f && gy == 0.f && gz == 0.f) continue;
    float u0, u1, D;
    const bool nz = boundary_weights(__ldg(a.msdf_wt + vi), __ldg(a.msdf_wt + vj), u0, u1, D);
    float* ri = g.ws + 16ll * vi + 8;
    float* rj = g.ws + 16ll * vj + 8;
    atomicAdd(ri, gx * u0); atomicAdd(ri + 1, gy * u0); atomicAdd(ri + 2, gz * u0);
    atomicAdd(rj, gx * u1); atomicAdd(rj + 1, gy * u1); atomicAdd(rj + 2, gz * u1);
    if (nz) {
      const double gu0 = (double)gx * a.v_tng_wt[3ll * vi] + (double)gy * a.v_tng_wt[3ll * vi + 1] + (double)gz * a.v_tng_wt[3ll * vi + 2];
      const double gu1 = (double)gx * a.v_tng_wt[3ll * vj] + (double)gy * a.v_tng_wt[3ll * vj + 1] + (double)gz * a.v_tng_wt[3ll * vj + 2];
      const double inv = 1.0 / (double)D;
      const double gD = -(gu0 * (double)u0 + gu1 * (double)u1) * inv;
      atomicAdd(a.g_mvert + vi, (float)(gu1 * inv + gD));
      atomicAdd(a.g_mvert + vj, (float)(-(gu0 * inv + gD)));
    }
  }
}

struct FaceGeom {
  int v[3];
  float e1[3], e2[3];
  float u1y, u2y, den;
};
__device__ __forceinline__ FaceGeom face_geom(const TngArgs& g, int64_t f) {
  FaceGeom r;
#pragma unroll
  for (int c = 0; c < 3; ++c) r.v[c] = (int)g.a.faces_wt[3 * f + c];
  const float* p = g.a.verts_wt;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    r.e1[c] = __fsub_rn(p[3ll * r.v[1] + c], p[3ll * r.v[0] + c]);
    r.e2[c] = __fsub_rn(p[3ll * r.v[2] + c], p[3ll * r.v[0] + c]);
  }
  const float2 uv0 = vertex_uv(g.uvp, r.v[0]), uv1 = vertex_uv(g.uvp, r.v[1]), uv2 = vertex_uv(g.uvp, r.v[2]);
  const float u1x = __fsub_rn(uv1.x, uv0.x), u2x = __fsub_rn(uv2.x, uv0.x);
  r.u1y = __fsub_rn(uv1.y, uv0.y);
  r.u2y = __fsub_rn(uv2.y, uv0.y);
  float den = __fsub_rn(__fmul_rn(u1x, r.u2y), __fmul_rn(r.u1y, u2x));
  r.den = (den > 0.f) ? fmaxf(den, 1e-6f) : fminf(den, -1e-6f);
  return r;
}

// forward sums again: N, c, S per vertex (thread per watertight face)
__global__ void __launch_bounds__(256) tng_accumulate_kernel(TngArgs g, int64_t n_faces) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_faces) return;
  const FaceGeom q = face_geom(g, f);
  const float nx = cross_comp(q.e1[1], q.e2[2], q.e1[2], q.e2[1]);
  const float ny = cross_comp(q.e1[2], q.e2[0], q.e1[0], q.e2[2]);
  const float nz = cross_comp(q.e1[0], q.e2[1], q.e1[1], q.e2[0]);
  const float tx = __fdiv_rn(__fsub_rn(__fmul_rn(q.e1[0], q.u2y), __fmul_rn(q.e2[0], q.u1y)), q.den);
  const float ty = __fdiv_rn(__fsub_rn(__fmul_rn(q.e1[1], q.u2y), __fmul_rn(q.e2[1], q.u1y)), q.den);
  const float tz = __fdiv_rn(__fsub_rn(__fmul_rn(q.e1[2], q.u2y), __fmul_rn(q.e2[2], q.u1y)), q.den);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float* row = g.ws + 16ll * q.v[c];
    atomicAdd(reinterpret_cast<float4*>(row), make_float4(nx, ny, nz, 1.f));
    atomicAdd(reinterpret_cast<float4*>(row) + 1, make_float4(tx, ty, tz, 0.f));
  }
}

// y = x / sqrt(max(x.x, 1e-20)) (render/util.py:25-29) and its adjoint
__device__ __forceinline__ void normalize_fwd(const double (&x)[3], double (&y)[3], double& len, bool& free) {
  const double d = x[0] * x[0] + x[1] * x[1] + x[2] * x[2];
  free = d > 1e-20;
  len = sqrt(free ? d : 1e-20);
  y[0] = x[0] / len; y[1] = x[1] / len; y[2] = x[2] / len;
}
__device__ __forceinline__ void normalize_bwd(const double (&y)[3], double len, bool free, const double (&gy)[3], double (&gx)[3]) {
  const double dot = free ? (y[0] * gy[0] + y[1] * gy[1] + y[2] * gy[2]) : 0.0;   // (clamped: the length is a constant)
#pragma unroll
  for (int c = 0; c < 3; ++c) gx[c] = (gy[c] - y[c] * dot) / len;
}

// thread per vertex: through normalise -> Gram-Schmidt -> normalise -> mean (tangent) and normalise (normal)
__global__ void __launch_bounds__(256) tng_vertex_kernel(TngArgs g) {
  const d3h_tangent_backward_args& a = g.a;
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= a.n_verts) return;
  float* row = g.ws + 16ll * v;
  double gt[3] = {row[8], row[9], row[10]};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (a.g_tng_wt != nullptr) gt[c] += a.g_tng_wt[3 * v + c];
    if (a.g_tng_aug != nullptr) gt[c] += a.g_tng_aug[3 * v + c];
  }
  const double cnt = row[3];
  double gs[3] = {0.0, 0.0, 0.0}, gn_sum[3] = {0.0, 0.0, 0.0};
  if (cnt > 0.0 && (gt[0] != 0.0 || gt[1] != 0.0 || gt[2] != 0.0)) {
    const double ns[3] = {row[0], row[1], row[2]};
    const bool nondeg = ns[0] * ns[0] + ns[1] * ns[1] + ns[2] * ns[2] > 1e-20;       // else (0,0,1): a constant
    const double nin[3] = {nondeg ? ns[0] : 0.0, nondeg ? ns[1] : 0.0, nondeg ? ns[2] : 1.0};
    const double am[3] = {row[4] / cnt, row[5] / cnt, row[6] / cnt};
    double n[3], t1[3], w[3], t2[3], ln, lt, lw;
    bool fn, ft, fw;
    normalize_fwd(nin, n, ln, fn);
    normalize_fwd(am, t1, lt, ft);
    const double proj = t1[0] * n[0] + t1[1] * n[1] + t1[2] * n[2];
#pragma unroll
    for (int c = 0; c < 3; ++c) w[c] = t1[c] - proj * n[c];
    normalize_fwd(w, t2, lw, fw);
    double gw[3], gt1[3], gn[3], ga[3], gnin[3];
    normalize_bwd(t2, lw, fw, gt, gw);
    const double ngw = n[0] * gw[0] + n[1] * gw[1] + n[2] * gw[2];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      gt1[c] = gw[c] - n[c] * ngw;
      gn[c] = -(proj * gw[c] + ngw * t1[c]);
    }
    normalize_bwd(t1, lt, ft, gt1, ga);
    normalize_bwd(n, ln, fn, gn, gnin);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      gs[c] = ga[c] / cnt;
      gn_sum[c] = nondeg ? gnin[c] : 0.0;
    }
  }
  row[4] = (float)gs[0]; row[5] = (float)gs[1]; row[6] = (float)gs[2];
  row[12] = (float)gn_sum[0]; row[13] = (float)gn_sum[1]; row[14] = (float)gn_sum[2];
}

// thread per face: g_S and g_N of its three vertices -> the edge vectors -> the vertex positions
__global__ void __launch_bounds__(256) tng_scatter_kernel(TngArgs g, int64_t n_faces) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_faces) return;
  const FaceGeom q = face_geom(g, f);
  double gt[3] = {0.0, 0.0, 0.0}, gf[3] = {0.0, 0.0, 0.0};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float* row = g.ws + 16ll * q.v[c];
    gt[0] += row[4]; gt[1] += row[5]; gt[2] += row[6];
    gf[0] += row[12]; gf[1] += row[13]; gf[2] += row[14];
  }
  if (gt[0] == 0.0 && gt[1] == 0.0 && gt[2] == 0.0 && gf[0] == 0.0 && gf[1] == 0.0 && gf[2] == 0.0) return;
  const double e1[3] = {q.e1[0], q.e1[1], q.e1[2]}, e2[3] = {q.e2[0], q.e2[1], q.e2[2]};
  // fn = e1 x e2: g_e1 = e2 x g_fn, g_e2 = g_fn x e1;  tang = (e1 u2y - e2 u1y) / den
  const double c1[3] = {e2[1] * gf[2] - e2[2] * gf[1], e2[2] * gf[0] - e2[0] * gf[2], e2[0] * gf[1] - e2[1] * gf[0]};
  const double c2[3] = {gf[1] * e1[2] - gf[2] * e1[1], gf[2] * e1[0] - gf[0] * e1[2], gf[0] * e1[1] - gf[1] * e1[0]};
  float* out = g.a.g_verts;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const double gnom = gt[c] / (double)q.den;
    const double g1 = gnom * (double)q.u2y + c1[c], g2 = -gnom * (double)q.u1y + c2[c];
    atomicAdd(out + 3ll * q.v[1] + c, (float)g1);
    atomicAdd(out + 3ll * q.v[2] + c, (float)g2);
    atomicAdd(out + 3ll * q.v[0] + c, (float)(-(g1 + g2)));
  }
}

// ------------------------------------------------------------------------------------------------
// second extraction of a cloth / body pair
// ------------------------------------------------------------------------------------------------
// Stores the pair's argument block and writes everything of the second extraction that hangs off a watertight vertex:
// same position, mSDF negated, verts_aug row kept iff the negated mSDF is positive (gshell_tets.py:423-427).
__global__ void __launch_bounds__(256) pair_vertex_kernel(FwdBlock src, Workspace ws) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  if (tid == 0) *ws.blk2 = src;
  const d3h_forward_args& a = src.a;
  const int64_t nv = ws.ctr->n_verts;
  const float4* __restrict__ w_vert = ws.vert;
  float4* __restrict__ vacc = reinterpret_cast<float4*>(a.vacc);
  for (int64_t v = tid; v < nv; v += nthreads) {
    const float4 p = w_vert[v];
    const float m = -p.w;
    if (v < a.cap_verts) {
      a.verts_wt[3 * v] = p.x; a.verts_wt[3 * v + 1] = p.y; a.verts_wt[3 * v + 2] = p.z;
      a.msdf_wt[v] = m;
      if (vacc != nullptr) {
        vacc[2 * v] = make_float4(0.f, 0.f, 0.f, 0.f);
        vacc[2 * v + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    if (v < a.cap_verts_aug) {
      const bool used = m > 0.f;
      a.verts_aug[3 * v] = used ? p.x : 0.f;
      a.verts_aug[3 * v + 1] = used ? p.y : 0.f;
      a.verts_aug[3 * v + 2] = used ? p.z : 0.f;
      a.msdf_aug[v] = m;
    }
  }
}

void launch_pair_replay(const d3h_forward_args& a, const Workspace& ws, const d3h_tet_record* records,
                        cudaStream_t stream) {
  FwdBlock blk2;
  blk2.a = a;
  blk2.a.msdf_negate = a.msdf_negate ? 0 : 1;
  blk2.a.verts_aug = a.pair_verts_aug; blk2.a.v_tng_aug = a.pair_v_tng_aug; blk2.a.msdf_aug = a.pair_msdf_aug;
  blk2.a.faces_aug = a.pair_faces_aug; blk2.a.verts_wt = a.pair_verts_wt; blk2.a.v_tng_wt = a.pair_v_tng_wt;
  blk2.a.msdf_wt = a.pair_msdf_wt; blk2.a.faces_wt = a.pair_faces_wt; blk2.a.vacc = a.pair_vacc;
  blk2.a.counts_host = a.pair_counts_host;
  blk2.a.seq = a.pair_seq;
  blk2.a.zero_g_pos = blk2.a.zero_g_sdf = blk2.a.zero_g_msdf = nullptr;
  blk2.counts_mapped = mapped_counts_pointer(a.pair_counts_host);
  blk2.trace = nullptr;
  ProfScope ps(K_PAIR_REPLAY, stream);
  int64_t vblocks = (ws.cap_corners + 255) / 256;
  if (vblocks < 1) vblocks = 1;
  if (vblocks > 148 * 4) vblocks = 148 * 4;
  launch_k(pair_vertex_kernel, (unsigned)vblocks, 256u, stream, kLaunchLatency, blk2, ws);
  if (ws.cap_tets <= 0) {
    launch_k(publish_counts_kernel, 1u, 1u, stream, kLaunchLatency, ws.blk2, ws.ctr, ws.counts2);
    return;
  }
  const UvParams uvp = uv_params(a.n_tets);
  // one frame: topology CTAs only in poly_faces_kernel (no normals / tangents to splat), both kinds in poly_cut_kernel
  const unsigned nblk = (unsigned)(ws.ntiles_poly > 0 ? ws.ntiles_poly : 1), ncut = cut_blocks(ws);
  launch_k(poly_faces_kernel<true>, nblk, (unsigned)kPolyThreads, stream, kLaunchLatency, ws.blk2, records, ws.ctr, ws.vert,
           ws.acc, ws.poly_cnt, ws.poly_gcnt, ws.poly_excl, ws.poly_used, uvp, ws.counts2, ws.corner_rank, ws.edge_bits,
           ws.word_prefix, nblk, 1u, FrameSet{}, FrameSet{});
  launch_k(poly_cut_kernel<true>, 2 * ncut, (unsigned)kPolyThreads, stream, kLaunchLatency, ws.blk2, records, ws.ctr,
           ws.vert, ws.acc, ws.owner, ws.poly_gcnt, ws.poly_excl, ws.poly_used, ncut, 1u, FrameSet{}, FrameSet{});
}

}  // namespace d3h


extern "C" int d3h_tangent_backward(const d3h_tangent_backward_args* a, d3h_stream_t s) {
  using namespace d3h;
  if (!a) { set_error("d3h_tangent_backward: null argument struct"); return D3H_E_BADARG; }
  const int64_t nv = a->n_verts, npoly = a->n_tri_tets + a->n_quad_tets, nf = a->n_tri_tets + 2 * a->n_quad_tets;
  if (nv < 0 || a->n_tri_tets < 0 || a->n_quad_tets < 0 || a->n_tets <= 0 || (nv > 0 && (!a->verts_wt || !a->msdf_wt ||
      !a->v_tng_wt || !a->g_verts || !a->g_mvert || !a->workspace)) || (nf > 0 && !a->faces_wt) || (npoly > 0 && !a->tape_corners) ||
      (reinterpret_cast<uintptr_t>(a->workspace) & 15) || a->workspace_bytes < 64 * nv) {
    set_error("d3h_tangent_backward: bad argument (null pointer, negative size, or workspace smaller than 64 bytes per vertex)");
    return D3H_E_BADARG;
  }
  if (nf == 3) {
    set_error("d3h_tangent_backward: a watertight mesh of exactly three faces (torch.cross without dim, gshell_tets.py:19) is not supported");
    return D3H_E_BADARG;
  }
  cudaStream_t stream = (cudaStream_t)s;
  if (nv == 0) return D3H_OK;
  cudaMemsetAsync(a->workspace, 0, (size_t)64 * nv, stream);
  cudaMemsetAsync(a->g_verts, 0, (size_t)12 * nv, stream);
  cudaMemsetAsync(a->g_mvert, 0, (size_t)4 * nv, stream);
  TngArgs g;
  g.a = *a;
  g.ws = reinterpret_cast<float*>(a->workspace);
  g.uvp = uv_params(a->n_tets);
  if (a->g_tng_aug != nullptr && npoly > 0)
    launch_k(tng_boundary_kernel, (unsigned)((npoly + 255) / 256), 256u, stream, kLaunchLatency, g);
  if (nf > 0) launch_k(tng_accumulate_kernel, (unsigned)((nf + 255) / 256), 256u, stream, kLaunchLatency, g, nf);
  launch_k(tng_vertex_kernel, (unsigned)((nv + 255) / 256), 256u, stream, kLaunchLatency, g);
  if (nf > 0) launch_k(tng_scatter_kernel, (unsigned)((nf + 255) / 256), 256u, stream, kLaunchLatency, g, nf);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("d3h_tangent_backward: %s", cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}
