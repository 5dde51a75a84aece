// The edge-scan path: stage 1 and 2 of the extraction WITHOUT streaming the tet array.
//
// A training run extracts from the same tet grid every iteration (hmsdf.py:207-212), so the host builds, once per
// grid, the sorted list of all distinct tet edges (edge_off / edge_b: CSR by smaller endpoint), the tets around every
// edge (etet_off / etets) and the rank of every tet's six edges in that list (tet_edge_rank).  With them:
//
//   edge_scan_kernel   one thread per grid vertex a walks the larger neighbours b of a (4 bytes per EDGE instead of the
//                      16 bytes per TET of classify_kernel: 68 MB instead of 201 MB at 128^3).  sign(sdf[a]) !=
//                      sign(sdf[b]) is exactly the crossing mask of gshell_tets.py:281.  Crossing edges go to work queues.
//   edge_mark_kernel   one thread per crossing edge walks the tets around it, 8 at a time with all loads of a batch in
//                      flight: the tets around a crossing edge are exactly the valid tets of :261-275 (a tet has mixed
//                      signs iff one of its edges crosses).  Marks the edge in the bitmap over the edge list and the
//                      tets in the T1 / T2 bitmaps; the first marker of a tet counts it for its 8192-tet tile and
//                      queues it.
//   scan_prefix_kernel one CTA per non-empty tile / edge block: exclusive prefix of the popcounts of its 256 bitmap
//                      words, on top of the sum of the counters of the earlier tiles / blocks (no look-back chain).
//                      rank among the marked tets = record id (tet order, the order of the boolean-mask compaction
//                      :277, :323-324); rank among the marked edges = vertex id (the order of torch.unique(dim=0), :279).
//   scan_emit_kernel   one thread per queue entry, whatever tile or block it sits in (balanced): a valid tet becomes its
//                      record + the vertex ids of its polygon corners (tape_corners), a crossing edge becomes its
//                      interpolated vertex (:291-303).
//
// Work queues: the order of the entries does not matter, so every warp appends with ONE atomic -- but ~1500 warps
// reserving on the same counter serialise at ~18 ns per atomic (measured: 27 us for the marking kernel, all of it
// waiting for that one address).  The queues are therefore split in kQueues sub-queues, a warp uses sub-queue
// (global warp id) % kQueues, and the consumers give every sub-queue its own CTAs.
//
// poly_faces_kernel / poly_cut_kernel / the adjoint are shared with the other paths.
//
// Forms of the static edge list, chosen once per grid by the host (extract.build_edge_table):
//   run-length tables  scan_runs_kernel + runs_expand_kernel (DEFAULT on grids numbered along the axes of a lattice; with the
//                      compressed tet array they also find the valid tets, and edge_mark_kernel is not launched)
//   transposed rows    edge_scan_rows_kernel (grids without that structure; edge_scan_pipe_kernel: opt-in persistent variant)
//   CSR walk           edge_scan_kernel (D3H_SCAN_ROWS=0)
// Kernels that a batch runs with gridDim.y = frame take the frame's workspace by offset (FrameSet, d3h_internal.cuh).
#include <cstdlib>

#include "d3h_internal.cuh"

namespace d3h {

constexpr int kEScanThreads = 256;
// vertices per thread of the stream (x 8 neighbour loads in flight each): D3H_SCAN_VPT = 1, 2 or 4 (default)
static int scan_vpt() {
  static int v = 0;
  if (v == 0) {
    const char* env = getenv("D3H_SCAN_VPT");
    v = (env && (env[0] == '1' || env[0] == '2')) ? (env[0] - '0') : 4;
  }
  return v;
}

struct ScanLists {
  unsigned* tile_cnt;     // valid tets per 8192-tet compaction tile: T1 class | T2 class << 16
  unsigned* eblock_cnt;   // crossing edges per 8192-edge block
  unsigned* q_cnt;        // [3][kQueues] x kQStride words: entries appended to every sub-queue (true counts, may exceed the
                          //   capacity), one counter per 128-byte line (atomics on one line serialise):
                          //   0 crossing edges as the stream found them, 1 valid tets, 2 edges that survive the prefilter
  int32_t* elist_raw;     // kQueues x cap_qe
  int2* vlist;            // kQueues x cap_qv: (tet id, occupancy code)
  int32_t* elist;         // kQueues x cap_qe; == elist_raw without the open-mesh prefilter
  int64_t cap_qe, cap_qv; // entries per sub-queue
};

__device__ __forceinline__ void shift_lists(ScanLists& L, int64_t shift) {
  L.tile_cnt = frame_ptr(L.tile_cnt, shift);
  L.eblock_cnt = frame_ptr(L.eblock_cnt, shift);
  L.q_cnt = frame_ptr(L.q_cnt, shift);
  L.elist_raw = frame_ptr(L.elist_raw, shift);
  L.vlist = frame_ptr(L.vlist, shift);
  L.elist = frame_ptr(L.elist, shift);
}

// One reservation per warp: `n` entries of this lane -> first slot of the lane in sub-queue q (all 32 lanes call).
__device__ __forceinline__ int64_t warp_reserve(unsigned* __restrict__ counter, unsigned n) {
  const unsigned lane = lane_id();
  unsigned incl = n;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned nb = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= (unsigned)o) incl += nb;
  }
  const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
  if (total == 0u) return -1;
  unsigned base = 0u;
  if (lane == 31) base = atomicAdd(counter, total);
  return (int64_t)__shfl_sync(0xffffffffu, base, 31) + incl - n;
}

// The stream.  A warp takes 32 * VPT consecutive vertices (lane l: vertices base + l, base + l + 32, ...: coalesced offset
// loads) and all neighbour loads of a thread's vertices are in flight together.  No shared memory, no barrier: a warp
// that found crossing edges (rare: the surface touches < 2 % of the vertices) reserves their slots in its sub-queue
// with one atomic and retires on its own.
template <int VPT>
__global__ void __launch_bounds__(kEScanThreads)
edge_scan_kernel(const FwdBlock* __restrict__ blk, const unsigned* __restrict__ occ_bits, ScanLists L) {
  pdl_enter();
  const d3h_forward_args& a = blk->a;
  const int32_t* __restrict__ edge_off = a.edge_off;
  const int32_t* __restrict__ edge_b = a.edge_b;
  const int64_t n_grid = a.n_grid;
  unsigned long long* tr = trace_begin(blk->trace, (unsigned)a.seq, K_EDGE_SCAN);
  const unsigned lane = lane_id();
  const int64_t gwarp = (int64_t)blockIdx.x * (kEScanThreads / 32) + (threadIdx.x >> 5);
  const int64_t wbase = gwarp * (32 * VPT);
  int e0[VPT], e1[VPT];
  unsigned oa[VPT];
#pragma unroll
  for (int k = 0; k < VPT; ++k) {
    const int64_t v = wbase + k * 32 + lane;
    e0[k] = e1[k] = 0;
    oa[k] = 0u;
    if (v < n_grid) {
      e0[k] = __ldg(edge_off + v);
      e1[k] = __ldg(edge_off + v + 1);
      oa[k] = occ_of(occ_bits, (int)v);
    }
  }
  int b[VPT][8];
#pragma unroll
  for (int k = 0; k < VPT; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) b[k][j] = (e0[k] + j < e1[k]) ? __ldg(edge_b + e0[k] + j) : -1;
  unsigned x[VPT];      // bit j: neighbour j of vertex k has the other sign
  unsigned cnt = 0u;
  bool more = false;    // a vertex with more than 8 larger neighbours (unstructured grids)
#pragma unroll
  for (int k = 0; k < VPT; ++k) {
    x[k] = 0u;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (b[k][j] >= 0) x[k] |= (occ_of(occ_bits, b[k][j]) ^ oa[k]) << j;
    cnt += __popc(x[k]);
    more = more || (e0[k] + 8 < e1[k]);
  }
  if (__any_sync(0xffffffffu, more)) {
    // the rest of the long neighbour lists: counted here, written below
#pragma unroll
    for (int k = 0; k < VPT; ++k)
      for (int e = e0[k] + 8; e < e1[k]; ++e) cnt += occ_of(occ_bits, __ldg(edge_b + e)) ^ oa[k];
  }
  const unsigned q = (unsigned)(gwarp % kQueues);
  int64_t slot = warp_reserve(L.q_cnt + kQStride * q, cnt);
  if (slot < 0) { trace_end(tr); return; }
  int32_t* __restrict__ out = L.elist_raw + (int64_t)q * L.cap_qe;
#pragma unroll
  for (int k = 0; k < VPT; ++k) {
    unsigned y = x[k];
    while (y) {
      const int e = e0[k] + (__ffs((int)y) - 1);
      y &= y - 1u;
      if (slot < L.cap_qe) out[slot] = e;
      ++slot;
    }
    for (int e = e0[k] + 8; e < e1[k]; ++e) {
      if ((occ_of(occ_bits, __ldg(edge_b + e)) ^ oa[k]) == 0u) continue;
      if (slot < L.cap_qe) out[slot] = e;
      ++slot;
    }
  }
  trace_end(tr);
}

// The stream over the TRANSPOSED edge list (d3h_forward_args.edge_rows, the default when the host built it).  The kernel
// above is bound by its instructions, not by DRAM (ncu r02q: 26 instructions per edge, issue slots 61 % busy at 3.1 TB/s):
// lane l's neighbours start at edge_off[v], 7 words apart from lane l+1's, so every load needs its own address, bound
// check and predicate, and one load instruction touches 7 cache lines.  Here a chunk of 32 consecutive vertices owns
// whole 128-byte rows (row j, lane l = the j-th larger neighbour of vertex 32c + l): one base address per chunk, row j at
// an immediate offset, one line per load.  Nothing is predicated: a lane always reads 8 rows -- past the chunk's last row
// lie the rows of the next chunk (8 spare rows close the table), valid vertex ids whose sign bits are fetched and then
// masked off by the chunk's row count; a missing neighbour inside the chunk is the vertex itself (same sign: never a
// crossing).  Six instructions per slot: row load, word index, address, sign word load, shift, funnel shift into the
// result mask.  edge_off is only read by the few lanes that found a crossing edge.
template <int CPW, bool PHASED>   // chunks per warp: 8 * CPW row loads in flight per lane
__global__ void __launch_bounds__(kEScanThreads, CPW == 4 ? 3 : (CPW == 2 ? 5 : 8))
edge_scan_rows_kernel(const FwdBlock* __restrict__ blk, const unsigned* __restrict__ occ_bits, ScanLists L) {
  pdl_enter();
  const d3h_forward_args& a = blk->a;
  const int32_t* __restrict__ rows = a.edge_rows;
  const int64_t n_grid = a.n_grid;
  const int64_t n_chunks = (n_grid + 31) >> 5;
  unsigned long long* tr = trace_begin(blk->trace, (unsigned)a.seq, K_EDGE_SCAN);
  const unsigned lane = lane_id();
  const int64_t gwarp = (int64_t)blockIdx.x * (kEScanThreads / 32) + (threadIdx.x >> 5);
  const int64_t c0 = gwarp * CPW;
  // row ranges of the warp's chunks: lanes 0 .. CPW fetch CPW + 1 consecutive offsets (clamped to the end of the
  // table: a chunk beyond the grid has no rows), everybody gets them by shuffle; the chunk's own signs are one word
  int roff, own = 0;
  {
    const int64_t c = c0 + lane < n_chunks ? c0 + lane : n_chunks;
    roff = __ldg(a.edge_row_off + c);
    if (lane < (unsigned)CPW && c < n_chunks) own = (int)__ldg(occ_bits + c);
  }
  int r0[CPW], w[CPW];
  unsigned oa[CPW];
#pragma unroll
  for (int k = 0; k < CPW; ++k) {
    r0[k] = __shfl_sync(0xffffffffu, roff, k);
    w[k] = __shfl_sync(0xffffffffu, roff, k + 1) - r0[k];
    oa[k] = ((unsigned)__shfl_sync(0xffffffffu, own, k) >> lane) & 1u;
  }
  int b[CPW][8];
  int all_b = 0;
#pragma unroll
  for (int k = 0; k < CPW; ++k) {
    const int32_t* __restrict__ p = rows + ((int64_t)r0[k] << 5) + lane;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      b[k][j] = ld_stream_s32(p + 32 * j);
      all_b |= b[k][j];
    }
  }
  // Three phases, each waiting for memory ONCE: all row loads, all sign-word loads, the bit arithmetic.  Left alone,
  // ptxas interleaves them in groups of four and a warp waits for DRAM eight times in a row (r02v: 21 us, every stall on
  // the first use of a load).  The phases are tied by data: vertex ids are non-negative, so `all_b >> 31` is a zero the
  // compiler cannot know -- added to the bitmap's address it makes every sign look-up depend on every row load, and-ed
  // with the OR of the sign words it seeds the result mask.
  const unsigned* __restrict__ occ = PHASED ? occ_bits + (all_b >> 31) : occ_bits;
  unsigned word[CPW][8];
  unsigned all_w = 0u;
#pragma unroll
  for (int k = 0; k < CPW; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      word[k][j] = __ldg(occ + (b[k][j] >> 5));
      all_w |= word[k][j];
    }
  const unsigned seed = PHASED ? (all_w & (unsigned)(all_b >> 31)) : 0u;
  unsigned x[CPW];      // bit j: neighbour j of the lane's vertex in chunk k has the other sign
  unsigned cnt = 0u;
  bool more = false;    // a chunk with more than 8 rows (unstructured grids)
#pragma unroll
  for (int k = 0; k < CPW; ++k) {
    unsigned acc = seed;   // the sign bit of slot j is pushed in at the top: slot 0 ends up in bit 24, slot 7 in bit 31
#pragma unroll
    for (int j = 0; j < 8; ++j) acc = __funnelshift_r(acc, word[k][j] >> (b[k][j] & 31), 1);
    acc = (acc >> 24) ^ (oa[k] ? 0xffu : 0u);
    const int wk = w[k] < 8 ? w[k] : 8;
    acc &= (1u << wk) - 1u;                                   // rows of the chunk only
    if (((c0 + k) << 5) + lane >= n_grid) acc = 0u;           // lanes beyond the grid in the last chunk
    x[k] = acc;
    cnt += __popc(acc);
    more = more || w[k] > 8;
  }
  if (more) {   // (warp-uniform) the rest of the long neighbour lists: counted here, written below
#pragma unroll
    for (int k = 0; k < CPW; ++k) {
      if (((c0 + k) << 5) + lane >= n_grid) continue;
      const int32_t* __restrict__ p = rows + ((int64_t)r0[k] << 5) + lane;
      for (int j = 8; j < w[k]; ++j) cnt += occ_of(occ_bits, ld_stream_s32(p + 32 * j)) ^ oa[k];
    }
  }
  const unsigned q = (unsigned)(gwarp % kQueues);
  int64_t slot = warp_reserve(L.q_cnt + kQStride * q, cnt);
  if (slot < 0) { trace_end(tr); return; }
  int32_t* __restrict__ out = L.elist_raw + (int64_t)q * L.cap_qe;
#pragma unroll
  for (int k = 0; k < CPW; ++k) {
    const int64_t v = ((c0 + k) << 5) + lane;
    unsigned y = x[k];
    if ((y == 0u && w[k] <= 8) || v >= n_grid) continue;
    const int e0 = __ldg(a.edge_off + v);
    while (y) {
      const int e = e0 + (__ffs((int)y) - 1);
      y &= y - 1u;
      if (slot < L.cap_qe) out[slot] = e;
      ++slot;
    }
    const int32_t* __restrict__ p = rows + ((int64_t)r0[k] << 5) + lane;
    for (int j = 8; j < w[k]; ++j) {
      if ((occ_of(occ_bits, ld_stream_s32(p + 32 * j)) ^ oa[k]) == 0u) continue;
      if (slot < L.cap_qe) out[slot] = e0 + j;
      ++slot;
    }
  }
  trace_end(tr);
}

// The same as a PERSISTENT, software-pipelined kernel (opt-in, D3H_SCAN_PIPE=1: measured 23.5 us against 22.7 us, r02x).  Timed alone, every one-shot variant above -- one, two or
// four chunks per warp, phased or not, and the CSR walk -- takes the same ~21 us (r02w): a warp lives ~5000 cycles (offset
// load, row loads, sign words, each a full memory latency) and has row loads in flight for a third of them, so the bytes in
// flight per SM are the same whatever the shape, and they are too few for DRAM.  Here a warp keeps streaming: while it
// looks up the signs of group g its row loads of group g + W (W = warps of the grid) and the row offsets of group g + 2W
// are already under way, so every resident warp has 8 * CPW rows in flight all the time.
template <int CPW>
__global__ void __launch_bounds__(kEScanThreads, CPW == 2 ? 3 : 5)
edge_scan_pipe_kernel(const FwdBlock* __restrict__ blk, const unsigned* __restrict__ occ_bits, ScanLists L) {
  pdl_enter();
  const d3h_forward_args& a = blk->a;
  const int32_t* __restrict__ rows = a.edge_rows;
  const int32_t* __restrict__ row_off = a.edge_row_off;
  const int64_t n_grid = a.n_grid;
  const int64_t n_chunks = (n_grid + 31) >> 5;
  const int64_t n_groups = (n_chunks + CPW - 1) / CPW;
  unsigned long long* tr = trace_begin(blk->trace, (unsigned)a.seq, K_EDGE_SCAN);
  const unsigned lane = lane_id();
  const int64_t gwarp = (int64_t)blockIdx.x * (kEScanThreads / 32) + (threadIdx.x >> 5);
  const int64_t W = (int64_t)gridDim.x * (kEScanThreads / 32);
  const unsigned q = (unsigned)(gwarp % kQueues);
  int32_t* __restrict__ out = L.elist_raw + (int64_t)q * L.cap_qe;
  // row offsets of a group: lanes 0 .. CPW hold CPW + 1 consecutive entries; a chunk beyond the grid has no rows (its
  // offsets are the end of the table: the 8 spare rows)
  auto load_off = [&](int64_t g) {
    int64_t c = g * CPW + lane;
    c = c < n_chunks ? c : n_chunks;
    return lane <= (unsigned)CPW ? __ldg(row_off + c) : 0;
  };
  int64_t g = gwarp;
  if (g >= n_groups) { trace_end(tr); return; }
  int roff = load_off(g), roff_next = load_off(g + W);
  int b[CPW][8];
#pragma unroll
  for (int k = 0; k < CPW; ++k) {
    const int32_t* __restrict__ p = rows + ((int64_t)__shfl_sync(0xffffffffu, roff, k) << 5) + lane;
#pragma unroll
    for (int j = 0; j < 8; ++j) b[k][j] = ld_stream_s32(p + 32 * j);
  }
  for (;;) {
    // ---- group g + W: rows; group g + 2W: offsets ----
    int bn[CPW][8];
#pragma unroll
    for (int k = 0; k < CPW; ++k) {
      const int32_t* __restrict__ p = rows + ((int64_t)__shfl_sync(0xffffffffu, roff_next, k) << 5) + lane;
#pragma unroll
      for (int j = 0; j < 8; ++j) bn[k][j] = ld_stream_s32(p + 32 * j);
    }
    const int roff_next2 = load_off(g + 2 * W);
    // ---- group g ----
    const int64_t c0 = g * CPW;
    int own = 0;
    if (lane < (unsigned)CPW && c0 + lane < n_chunks) own = (int)__ldg(occ_bits + c0 + lane);   // the chunk's own signs
    int r0[CPW], w[CPW];
    unsigned oa[CPW];
    int all_b = 0;
#pragma unroll
    for (int k = 0; k < CPW; ++k) {
      r0[k] = __shfl_sync(0xffffffffu, roff, k);
      w[k] = __shfl_sync(0xffffffffu, roff, k + 1) - r0[k];
      oa[k] = ((unsigned)__shfl_sync(0xffffffffu, own, k) >> lane) & 1u;
#pragma unroll
      for (int j = 0; j < 8; ++j) all_b |= b[k][j];
    }
    // (vertex ids are non-negative: `all_b >> 31` is a zero the compiler cannot know; it ties every sign look-up to
    // every row load of the group and seeds the result mask with the OR of the sign words, see edge_scan_rows_kernel)
    const unsigned* __restrict__ occ = occ_bits + (all_b >> 31);
    unsigned word[CPW][8];
    unsigned all_w = 0u;
#pragma unroll
    for (int k = 0; k < CPW; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        word[k][j] = __ldg(occ + (b[k][j] >> 5));
        all_w |= word[k][j];
      }
    const unsigned seed = all_w & (unsigned)(all_b >> 31);
    unsigned x[CPW];
    unsigned cnt = 0u;
    bool more = false;
#pragma unroll
    for (int k = 0; k < CPW; ++k) {
      unsigned acc = seed;
#pragma unroll
      for (int j = 0; j < 8; ++j) acc = __funnelshift_r(acc, word[k][j] >> (b[k][j] & 31), 1);
      acc = (acc >> 24) ^ (oa[k] ? 0xffu : 0u);
      const int wk = w[k] < 8 ? w[k] : 8;
      acc &= (1u << wk) - 1u;
      if (((c0 + k) << 5) + lane >= n_grid) acc = 0u;
      x[k] = acc;
      cnt += __popc(acc);
      more = more || w[k] > 8;
    }
    if (more) {   // (warp-uniform) the rest of the long neighbour lists: counted here, written below
#pragma unroll
      for (int k = 0; k < CPW; ++k) {
        if (((c0 + k) << 5) + lane >= n_grid) continue;
        const int32_t* __restrict__ p = rows + ((int64_t)r0[k] << 5) + lane;
        for (int j = 8; j < w[k]; ++j) cnt += occ_of(occ_bits, ld_stream_s32(p + 32 * j)) ^ oa[k];
      }
    }
    int64_t slot = warp_reserve(L.q_cnt + kQStride * q, cnt);
    if (slot >= 0) {
#pragma unroll
      for (int k = 0; k < CPW; ++k) {
        const int64_t v = ((c0 + k) << 5) + lane;
        unsigned y = x[k];
        if ((y == 0u && w[k] <= 8) || v >= n_grid) continue;
        const int e0 = __ldg(a.edge_off + v);
        while (y) {
          const int e = e0 + (__ffs((int)y) - 1);
          y &= y - 1u;
          if (slot < L.cap_qe) out[slot] = e;
          ++slot;
        }
        const int32_t* __restrict__ p = rows + ((int64_t)r0[k] << 5) + lane;
        for (int j = 8; j < w[k]; ++j) {
          if ((occ_of(occ_bits, ld_stream_s32(p + 32 * j)) ^ oa[k]) == 0u) continue;
          if (slot < L.cap_qe) out[slot] = e0 + j;
          ++slot;
        }
      }
    }
    g += W;
    if (g >= n_groups) break;
    roff = roff_next;
    roff_next = roff_next2;
#pragma unroll
    for (int k = 0; k < CPW; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) b[k][j] = bn[k][j];
  }
  trace_end(tr);
}

// The scan over the RUN-LENGTH compressed tables (d3h_forward_args.edge_runs / tet_runs; the default whenever the host
// built them).  Every kernel above spends its time on per-edge work: 6 to 26 instructions to fetch one sign bit, ~9 M warp
// instructions per call at an IPC bounded by the dependent look-ups -- ~20 us whatever the shape (r02w / r02x).  On a grid
// numbered along its axes the 32 vertices of a chunk have the same few end-point differences d, and the signs of the 32
// far end points 32c + l + d are 32 CONSECUTIVE bits of the sign bitmap: one funnel shift of two adjacent words.  A THREAD
// takes an entry (chunk, d, mask): one xor with the chunk's own word and an and with the mask give the crossing flags of
// 32 edges.  ~7 entries per chunk on the Kuhn lattice: 5.6 MB instead of 59 MB, ~0.5 M warp instructions.
//
// With the tet array compressed the same way (tet_runs; watertight template) the CTAs behind the edge entries find the
// VALID TETS (mixed signs, gshell_tets.py:261-275): a thread takes an entry (chunk of the first vertex, d1, d2, d3, mask),
// three windows beside the chunk's own word are the occupancy codes of 32 tets.  That replaces edge_mark_kernel (~22 us of
// dependent look-ups: edge -> incidence list -> tet -> signs -> returned atomics): every crossing edge and every valid tet
// is met exactly once, so marks and counts are fire-and-forget and only the queue slots cost one returned atomic per warp.
//
// The entries that found something (the surface: a few per cent) are expanded by the whole warp, lane l = lane l of the
// entry, eight entries at a time so that the loads of their id rows are in flight together (a lane expanding its own
// entries one after the other makes the kernel 47 us: r02y).  (sign_window: d3h_internal.cuh)
__device__ __forceinline__ int64_t shfl_i64(int64_t v, int src) {
  return (int64_t)__shfl_sync(0xffffffffu, (unsigned)(v & 0xffffffffll), src) |
         ((int64_t)__shfl_sync(0xffffffffu, (unsigned)(v >> 32), src) << 32);
}

// Work items of the expansion: an entry that found something.  Edge items live in the (otherwise unused) second edge
// queue, tet items in the record buffer (written later, by scan_emit_kernel); their counters are the first two words of
// the fourth counter group, the third word flags a dropped item (scan_prefix_kernel reports an overflow then).
struct EdgeItem { int entry_q; unsigned x; int64_t at; };                           // 16 bytes; entry | sub-queue << 26
struct TetItem { int entry_q; unsigned x; int64_t at; unsigned own, w1, w2, w3; };  // 32 bytes
constexpr int kItemEdges = 3 * kQueues, kItemTets = 3 * kQueues + 1, kItemDropped = 3 * kQueues + 2;

// One slot per lane with `has` in the item list behind `counter` (one atomic per warp); -1: no room
__device__ __forceinline__ int64_t item_slot(unsigned* __restrict__ counter, bool has, int64_t cap, unsigned* __restrict__ dropped) {
  const unsigned m = __ballot_sync(0xffffffffu, has);
  unsigned base = 0u;
  if (lane_id() == 0) base = atomicAdd(counter, (unsigned)__popc(m));
  base = __shfl_sync(0xffffffffu, base, 0);
  const int64_t s = (int64_t)base + __popc(m & ((1u << lane_id()) - 1u));
  if (has && s >= cap) { atomicOr(dropped, 1u); return -1; }
  return has ? s : -1;
}

// Pass A: a thread per entry.  The warps that find nothing (all but a few per cent) leave after the test.
template <bool MARK>   // MARK: with the compressed tet array (crossing edges are marked by the expansion, no edge_mark_kernel)
__global__ void __launch_bounds__(kEScanThreads)
scan_runs_kernel(const FwdBlock* __restrict__ blk, const unsigned* __restrict__ occ_bits, ScanLists L, EdgeItem* __restrict__ eitems,
                 int64_t cap_eitems, TetItem* __restrict__ titems, int64_t cap_titems, unsigned nb_edges, const __grid_constant__ FrameSet fs) {
  pdl_enter();
  const int64_t shift = fs.off[blockIdx.y];   // (the lists and item buffers are shifted by the few warps that need them)
  blk = frame_ptr(blk, shift);
  occ_bits = frame_ptr(occ_bits, shift);
  const d3h_forward_args& a = blk->a;
  unsigned long long* tr = trace_begin(blk->trace, (unsigned)a.seq, K_EDGE_SCAN);
  const bool edges = blockIdx.x < nb_edges;
  const int64_t i = (int64_t)(edges ? blockIdx.x : blockIdx.x - nb_edges) * kEScanThreads + threadIdx.x;   // entry
  const unsigned q = ((blockIdx.x * kEScanThreads + threadIdx.x) >> 5) % kQueues;
  if (edges) {
    unsigned x = 0u;     // crossing flags: bit l = the edge (32c + l, 32c + l + d) exists and its end points differ in sign
    if (i < a.n_edge_runs) {
      const int64_t c = __ldg(a.edge_run_chunk + i);
      const int2 e = __ldg(reinterpret_cast<const int2*>(a.edge_runs) + i);
      x = (sign_window(occ_bits, (c << 5) + e.x) ^ __ldg(occ_bits + c)) & (unsigned)e.y;
    }
    if (!__any_sync(0xffffffffu, x != 0u)) { trace_end(tr); return; }
    unsigned* __restrict__ q_cnt = frame_ptr(L.q_cnt, shift);
    const int64_t at = warp_reserve(q_cnt + kQStride * q, (unsigned)__popc(x));
    const int64_t s = item_slot(q_cnt + kQStride * kItemEdges, x != 0u, cap_eitems, q_cnt + kQStride * kItemDropped);
    if (s >= 0) frame_ptr(eitems, shift)[s] = EdgeItem{(int)i | (int)(q << 26), x, at};
  } else {
    unsigned x = 0u, own = 0u, w1 = 0u, w2 = 0u, w3 = 0u;   // x: tets of the entry whose signs are mixed
    if (i < a.n_tet_runs) {
      const int64_t c = __ldg(a.tet_run_chunk + i);
      const int4 e = __ldg(reinterpret_cast<const int4*>(a.tet_runs) + i);
      own = __ldg(occ_bits + c);
      w1 = sign_window(occ_bits, (c << 5) + e.x);
      w2 = sign_window(occ_bits, (c << 5) + e.y);
      w3 = sign_window(occ_bits, (c << 5) + e.z);
      x = ((own ^ w1) | (own ^ w2) | (own ^ w3)) & (unsigned)e.w;
    }
    if (!__any_sync(0xffffffffu, x != 0u)) { trace_end(tr); return; }
    unsigned* __restrict__ q_cnt = frame_ptr(L.q_cnt, shift);
    const int64_t at = warp_reserve(q_cnt + kQStride * (kQueues + q), (unsigned)__popc(x));
    const int64_t s = item_slot(q_cnt + kQStride * kItemTets, x != 0u, cap_titems, q_cnt + kQStride * kItemDropped);
    if (s >= 0) frame_ptr(titems, shift)[s] = TetItem{(int)i | (int)(q << 26), x, at, own, w1, w2, w3};
  }
  trace_end(tr);
}

// Pass B: a warp per item, lane l = lane l of the entry: one coalesced row of ids, the marks and counts (reductions: every
// crossing edge and every valid tet is met exactly once) and the queue entries.  Warps [0, warps_edges) of the grid take
// the edge items, the others the tet items, every CTA a contiguous piece of its list.
//
// The per-tile / per-block counts are the hot spot: a compaction tile on the surface collects ~2000 valid tets, and
// reductions on one address pass the L2 at ~18 ns each -- 21 us for this kernel, as for edge_mark_kernel before it (r02ab).
// Items come in entry order, so the few hundred tets of a CTA fall into one or two tiles: the counts are collected in a
// small shared table (key = counter index) and flushed with one reduction per key and CTA.
constexpr int kAggSlots = 64;
struct CountAgg {
  unsigned key[kAggSlots], val[kAggSlots];
};
__device__ __forceinline__ void agg_add(CountAgg& g, unsigned* __restrict__ counters, unsigned key, unsigned v) {
  const unsigned slot = key % kAggSlots;
  const unsigned old = atomicCAS(&g.key[slot], 0xffffffffu, key);
  if (old == 0xffffffffu || old == key) atomicAdd(&g.val[slot], v);
  else atomicAdd(counters + key, v);   // the slot belongs to another counter
}

template <bool MARK>
__global__ void __launch_bounds__(256)
runs_expand_kernel(const FwdBlock* __restrict__ blk, unsigned* __restrict__ m1_words, unsigned* __restrict__ m2_words,
                   unsigned* __restrict__ edge_bits, ScanLists L, const EdgeItem* __restrict__ eitems, int64_t cap_eitems,
                   const TetItem* __restrict__ titems, int64_t cap_titems, unsigned ctas_edges, const __grid_constant__ FrameSet fs) {
  pdl_enter();
  {
    const int64_t shift = fs.off[blockIdx.y];
    blk = frame_ptr(blk, shift); m1_words = frame_ptr(m1_words, shift); m2_words = frame_ptr(m2_words, shift);
    edge_bits = frame_ptr(edge_bits, shift); eitems = frame_ptr(eitems, shift); titems = frame_ptr(titems, shift);
    shift_lists(L, shift);
  }
  __shared__ CountAgg agg;
  const d3h_forward_args& a = blk->a;
  unsigned long long* tr = trace_begin(blk->trace, (unsigned)a.seq, K_EDGE_MARK);
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned below = (1u << lane) - 1u;
  if (threadIdx.x < kAggSlots) { agg.key[threadIdx.x] = 0xffffffffu; agg.val[threadIdx.x] = 0u; }
  __syncthreads();
  const bool edges = blockIdx.x < ctas_edges;
  unsigned* __restrict__ counters = edges ? L.eblock_cnt : L.tile_cnt;
  if (edges) {
    int64_t n = (int64_t)L.q_cnt[kQStride * kItemEdges];
    n = n < cap_eitems ? n : cap_eitems;
    const int64_t per = (n + ctas_edges - 1) / ctas_edges, j0 = per * blockIdx.x, j1 = j0 + per < n ? j0 + per : n;
    for (int64_t j = j0 + warp; j < j1; j += 8) {
      const EdgeItem it = eitems[j];
      if (!((it.x >> lane) & 1u)) continue;
      const unsigned e = (unsigned)__ldg(a.edge_run_ids + ((int64_t)(it.entry_q & 0x3ffffff) << 5) + lane);   // rank in the edge list
      if (MARK) {
        atomicOr(edge_bits + (e >> 5), 1u << (e & 31u));
        agg_add(agg, counters, e / (unsigned)kEdgeBlock, 1u);
      }
      const int64_t s = it.at + __popc(it.x & below);
      if (s < L.cap_qe) L.elist_raw[(int64_t)((unsigned)it.entry_q >> 26) * L.cap_qe + s] = (int)e;
    }
  } else if (MARK) {
    int64_t n = (int64_t)L.q_cnt[kQStride * kItemTets];
    n = n < cap_titems ? n : cap_titems;
    const unsigned ctas_tets = gridDim.x - ctas_edges;
    const int64_t per = (n + ctas_tets - 1) / ctas_tets, j0 = per * (blockIdx.x - ctas_edges), j1 = j0 + per < n ? j0 + per : n;
    for (int64_t j = j0 + warp; j < j1; j += 8) {
      const TetItem it = titems[j];
      if (!((it.x >> lane) & 1u)) continue;
      const int t = __ldg(a.tet_run_ids + ((int64_t)(it.entry_q & 0x3ffffff) << 5) + lane);
      // occupancy code: bit v = sign of the tet's vertex v
      const unsigned code = ((it.own >> lane) & 1u) | (((it.w1 >> lane) & 1u) << 1) | (((it.w2 >> lane) & 1u) << 2) |
                            (((it.w3 >> lane) & 1u) << 3);
      const bool quad = __popc(code) == 2;
      atomicOr((quad ? m2_words : m1_words) + (t >> 5), 1u << (t & 31));
      agg_add(agg, counters, (unsigned)t / (unsigned)kTileTets, quad ? 0x10000u : 1u);
      const int64_t s = it.at + __popc(it.x & below);
      if (s < L.cap_qv) L.vlist[(int64_t)((unsigned)it.entry_q >> 26) * L.cap_qv + s] = make_int2(t, (int)code);
    }
  }
  __syncthreads();
  if (threadIdx.x < kAggSlots && agg.key[threadIdx.x] != 0xffffffffu && agg.val[threadIdx.x] != 0u)
    atomicAdd(counters + agg.key[threadIdx.x], agg.val[threadIdx.x]);
  trace_end(tr);
}

// launch of the stream over the compressed or transposed edge list.  A/B switches: D3H_SCAN_PIPE=1 the persistent kernel
// instead of the one-shot one; D3H_SCAN_CPW = chunks per warp (pipe: 1 or 2 (default); one-shot: 1, 2 (default) or 4);
// D3H_SCAN_PHASED=0 leaves the instruction order of the one-shot kernel to the compiler
template <typename Launch>
static void launch_scan_rows(const d3h_forward_args& a, Launch&& launch) {
  static int cpw = 0, phased = 1, pipe = 0, grid1 = 0, grid2 = 0;
  if (cpw == 0) {
    const char* env = getenv("D3H_SCAN_CPW");
    cpw = (env && (env[0] == '1' || env[0] == '4')) ? (env[0] - '0') : 2;
    const char* ph = getenv("D3H_SCAN_PHASED");
    phased = !(ph && ph[0] == '0');
    const char* pp = getenv("D3H_SCAN_PIPE");
    pipe = pp && pp[0] == '1';
    grid1 = persistent_grid(reinterpret_cast<const void*>(edge_scan_pipe_kernel<1>), kEScanThreads, 0);
    grid2 = persistent_grid(reinterpret_cast<const void*>(edge_scan_pipe_kernel<2>), kEScanThreads, 0);
    const char* gg = getenv("D3H_SCAN_GRID");   // tests: a small grid makes every warp take many groups
    if (gg && atoi(gg) > 0) grid1 = grid2 = atoi(gg);
  }
  const int64_t n_chunks = (a.n_grid + 31) / 32;
  if (pipe) {
    const int c = cpw == 1 ? 1 : 2;
    const int64_t need = (n_chunks + 8 * c - 1) / (8 * c);   // CTAs of a one-shot launch
    const int64_t cap = c == 1 ? grid1 : grid2;
    const unsigned nblk = (unsigned)(need < cap ? need : cap);
    if (c == 1) launch(edge_scan_pipe_kernel<1>, nblk);
    else launch(edge_scan_pipe_kernel<2>, nblk);
    return;
  }
  const int64_t per_cta = (int64_t)(kEScanThreads / 32) * cpw;
  const unsigned nblk = (unsigned)((n_chunks + per_cta - 1) / per_cta);
  if (!phased) launch(edge_scan_rows_kernel<4, false>, (unsigned)((n_chunks + 31) / 32));
  else if (cpw == 1) launch(edge_scan_rows_kernel<1, true>, nblk);
  else if (cpw == 4) launch(edge_scan_rows_kernel<4, true>, nblk);
  else launch(edge_scan_rows_kernel<2, true>, nblk);
}

// One thread per crossing edge of the whole grid (all resident at once: the chain etet_off -> etets -> tets -> signs ->
// atomics is paid once).  CTA c serves sub-queue c % kQueues.  All loads of a batch of 8 tets are issued together.
template <bool MOCC>
__global__ void __launch_bounds__(256)
edge_mark_kernel(const FwdBlock* __restrict__ blk, const unsigned* __restrict__ occ_bits,
                 const unsigned* __restrict__ mocc_bits, unsigned* __restrict__ m1_words,
                 unsigned* __restrict__ m2_words, unsigned* __restrict__ edge_bits, ScanLists L) {
  pdl_enter();
  const d3h_forward_args& a = blk->a;
  const int32_t* __restrict__ etets = a.etets;
  const int4* __restrict__ tets = reinterpret_cast<const int4*>(a.tets);
  unsigned long long* tr = trace_begin(blk->trace, (unsigned)a.seq, K_EDGE_MARK);
  const unsigned lane = lane_id();
  const unsigned q = blockIdx.x % kQueues, part = blockIdx.x / kQueues, parts = gridDim.x / kQueues;
  const int64_t raw = (int64_t)L.q_cnt[kQStride * q];
  const int64_t n = raw < L.cap_qe ? raw : L.cap_qe;
  const int32_t* __restrict__ in = L.elist_raw + (int64_t)q * L.cap_qe;
  // the valid tets found by this warp go to sub-queue (its global warp id) % kQueues
  const unsigned qv = (unsigned)((blockIdx.x * 8u + (threadIdx.x >> 5)) % kQueues);
  int2* __restrict__ vout = L.vlist + (int64_t)qv * L.cap_qv;
  for (int64_t j0 = (int64_t)part * 256 + (threadIdx.x & ~31u); j0 < n; j0 += (int64_t)parts * 256) {   // warp-uniform
    const int64_t j = j0 + lane;
    const int e = j < n ? in[j] : -1;
    int t0 = 0, t1 = 0;
    if (e >= 0) { t0 = __ldg(a.etet_off + e); t1 = __ldg(a.etet_off + e + 1); }
    bool any = false;
    while (__any_sync(0xffffffffu, t0 < t1)) {
      int t[8];
      int4 v4[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) t[i] = (t0 + i < t1) ? __ldg(etets + t0 + i) : -1;
#pragma unroll
      for (int i = 0; i < 8; ++i) v4[i] = (t[i] >= 0) ? __ldg(tets + t[i]) : make_int4(0, 0, 0, 0);
      unsigned code[8], fresh = 0u;   // fresh: bit i = this lane marked tet i first
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        code[i] = occ_of(occ_bits, v4[i].x) | (occ_of(occ_bits, v4[i].y) << 1) | (occ_of(occ_bits, v4[i].z) << 2) |
                  (occ_of(occ_bits, v4[i].w) << 3);
        if (MOCC && t[i] >= 0) {   // open-mesh prefilter, gshell_tets.py:275: keep tets with a vertex of positive mSDF
          const unsigned keep = occ_of(mocc_bits, v4[i].x) | occ_of(mocc_bits, v4[i].y) | occ_of(mocc_bits, v4[i].z) |
                                occ_of(mocc_bits, v4[i].w);
          if (!keep) t[i] = -1;
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (t[i] < 0) continue;
        any = true;
        const bool quad = __popc(code[i]) == 2;
        const unsigned bit = 1u << (t[i] & 31);
        const unsigned old = atomicOr((quad ? m2_words : m1_words) + (t[i] >> 5), bit);
        if (!(old & bit)) fresh |= 1u << i;
      }
      // count the tet for its tile: the result is not used, so this is a fire-and-forget reduction (a tile on the
      // surface collects ~2000 of them; waiting for returned values was 40 % of this kernel's stall samples)
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if ((fresh >> i) & 1u)
          atomicAdd(L.tile_cnt + (unsigned)t[i] / (unsigned)kTileTets, __popc(code[i]) == 2 ? 0x10000u : 1u);
      int64_t slot = warp_reserve(L.q_cnt + kQStride * (kQueues + qv), (unsigned)__popc(fresh));
      if (slot >= 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (!((fresh >> i) & 1u)) continue;
          if (slot < L.cap_qv) vout[slot] = make_int2(t[i], (int)code[i]);
          ++slot;
        }
      }
      t0 += 8;
    }
    // the edge itself: a bit in the bitmap over the edge list and a count for its block.  With the prefilter `any` may
    // be false (no valid tet keeps the edge: torch.unique never sees it) and the surviving edges are queued again.
    if (any) {
      atomicOr(edge_bits + ((unsigned)e >> 5), 1u << ((unsigned)e & 31u));
      atomicAdd(L.eblock_cnt + (unsigned)e / (unsigned)kEdgeBlock, 1u);
    }
    if (MOCC) {
      const int64_t slot = warp_reserve(L.q_cnt + kQStride * (2 * kQueues + q), any ? 1u : 0u);
      if (any && slot >= 0 && slot < L.cap_qe) L.elist[(int64_t)q * L.cap_qe + slot] = e;
    }
  }
  trace_end(tr);
}

// The same with the fixed-width incidence rows (d3h_forward_args.etets8) and WITHOUT waiting for an atomic: which of the
// threads that meet a valid tet (one per crossing edge of the tet, 3 or 4) counts and queues it is decided by a rule
// instead of by the value an atomicOr returns -- the thread of the tet's FIRST crossing edge in the order of
// gshell_tets.py:187.  The first crossing edge always starts at the tet's vertex 0 (if the signs of vertices 1, 2, 3 all
// equalled the sign of vertex 0 the tet would not be valid), so the owner is the edge (vertex 0, first vertex j whose
// sign differs).  Also exact for tets that repeat a vertex: equal ids have equal signs, and the incidence lists name
// every (edge, tet) pair once.  Chain of dependent loads per thread: queue entry -> incidence row (+ end points, in
// parallel; both prefetched into L2 by the stream) -> tets -> sign bits; the marks and counts are fire-and-forget.
template <bool MOCC>
__global__ void __launch_bounds__(256)
edge_mark_rows_kernel(const FwdBlock* __restrict__ blk, const unsigned* __restrict__ occ_bits,
                      const unsigned* __restrict__ mocc_bits, unsigned* __restrict__ m1_words,
                      unsigned* __restrict__ m2_words, unsigned* __restrict__ edge_bits, ScanLists L) {
  pdl_enter();
  const d3h_forward_args& a = blk->a;
  const int32_t* __restrict__ etets = a.etets;
  const int4* __restrict__ rows = reinterpret_cast<const int4*>(a.etets8);
  const int2* __restrict__ edge_ab = reinterpret_cast<const int2*>(a.edge_ab);
  const int4* __restrict__ tets = reinterpret_cast<const int4*>(a.tets);
  unsigned long long* tr = trace_begin(blk->trace, (unsigned)a.seq, K_EDGE_MARK);
  const unsigned lane = lane_id();
  const unsigned q = blockIdx.x % kQueues, part = blockIdx.x / kQueues, parts = gridDim.x / kQueues;
  const int64_t raw = (int64_t)L.q_cnt[kQStride * q];
  const int64_t n = raw < L.cap_qe ? raw : L.cap_qe;
  const int32_t* __restrict__ in = L.elist_raw + (int64_t)q * L.cap_qe;
  const unsigned qv = (unsigned)((blockIdx.x * 8u + (threadIdx.x >> 5)) % kQueues);
  int2* __restrict__ vout = L.vlist + (int64_t)qv * L.cap_qv;
  for (int64_t j0 = (int64_t)part * 256 + (threadIdx.x & ~31u); j0 < n; j0 += (int64_t)parts * 256) {   // warp-uniform
    const int64_t j = j0 + lane;
    const int e = j < n ? in[j] : -1;
    int4 r0 = make_int4(-1, -1, -1, -1), r1 = r0;
    int2 ab = make_int2(-1, -1);
    if (e >= 0) {
      r0 = __ldg(rows + 2ll * e);
      r1 = __ldg(rows + 2ll * e + 1);
      ab = __ldg(edge_ab + e);
    }
    const bool crowded = r1.w == -2;    // more than 8 tets around the edge: walk the CSR list instead
    int t0 = 0, t1 = 0;
    if (crowded) { t0 = __ldg(a.etet_off + e); t1 = __ldg(a.etet_off + e + 1); }
    bool any = false, first = true;
    do {
      int t[8];
      if (!crowded) {
        t[0] = first ? r0.x : -1; t[1] = first ? r0.y : -1; t[2] = first ? r0.z : -1; t[3] = first ? r0.w : -1;
        t[4] = first ? r1.x : -1; t[5] = first ? r1.y : -1; t[6] = first ? r1.z : -1; t[7] = first ? r1.w : -1;
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) t[i] = (t0 + i < t1) ? __ldg(etets + t0 + i) : -1;
      }
      int4 v4[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v4[i] = (t[i] >= 0) ? __ldg(tets + t[i]) : make_int4(0, 0, 0, 0);
      unsigned code[8], own = 0u;   // own: bit i = this edge is the first crossing edge of tet i
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        code[i] = occ_of(occ_bits, v4[i].x) | (occ_of(occ_bits, v4[i].y) << 1) | (occ_of(occ_bits, v4[i].z) << 2) |
                  (occ_of(occ_bits, v4[i].w) << 3);
        if (MOCC && t[i] >= 0) {   // open-mesh prefilter, gshell_tets.py:275: keep tets with a vertex of positive mSDF
          const unsigned keep = occ_of(mocc_bits, v4[i].x) | occ_of(mocc_bits, v4[i].y) | occ_of(mocc_bits, v4[i].z) |
                                occ_of(mocc_bits, v4[i].w);
          if (!keep) t[i] = -1;
        }
        if (t[i] < 0) continue;
        // signs relative to vertex 0; the first vertex j in 1..3 that differs closes the tet's first crossing edge
        const unsigned rel = (code[i] & 1u) ? (~code[i] & 0xeu) : (code[i] & 0xeu);
        const int jf = __ffs((int)rel) - 1;                                        // 1..3
        const int other = (ab.x == v4[i].x) ? ab.y : ((ab.y == v4[i].x) ? ab.x : -1);   // -1: vertex 0 is not on this edge
        const int vj = jf == 1 ? v4[i].y : (jf == 2 ? v4[i].z : v4[i].w);
        // (first-match semantics: a vertex id that repeats inside the tet has the same sign everywhere, so if `other`
        // equals v_jf it is the first differing vertex whichever copy is meant)
        if (other >= 0 && other == vj) own |= 1u << i;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (t[i] < 0) continue;
        any = true;
        if (!((own >> i) & 1u)) continue;
        const bool quad = __popc(code[i]) == 2;
        atomicOr((quad ? m2_words : m1_words) + (t[i] >> 5), 1u << (t[i] & 31));          // (results unused: reductions)
        atomicAdd(L.tile_cnt + (unsigned)t[i] / (unsigned)kTileTets, quad ? 0x10000u : 1u);
      }
      int64_t slot = warp_reserve(L.q_cnt + kQStride * (kQueues + qv), (unsigned)__popc(own));
      if (slot >= 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (!((own >> i) & 1u)) continue;
          if (slot < L.cap_qv) vout[slot] = make_int2(t[i], (int)code[i]);
          ++slot;
        }
      }
      t0 += 8;
      first = false;
    } while (__any_sync(0xffffffffu, crowded && t0 < t1));
    if (any) {
      atomicOr(edge_bits + ((unsigned)e >> 5), 1u << ((unsigned)e & 31u));
      atomicAdd(L.eblock_cnt + (unsigned)e / (unsigned)kEdgeBlock, 1u);
    }
    if (MOCC) {
      const int64_t slot = warp_reserve(L.q_cnt + kQStride * (2 * kQueues + q), any ? 1u : 0u);
      if (any && slot >= 0 && slot < L.cap_qe) L.elist[(int64_t)q * L.cap_qe + slot] = e;
    }
  }
  trace_end(tr);
}

// ------------------------------------------------------------------------------------------------
// exclusive prefixes of the marked tets (per word of the T1 / T2 bitmaps) and of the marked edges (per word of the edge
// bitmap).  grid = grid_tiles + grid_blocks CTAs; a CTA of the first group takes the listed tiles li = blockIdx.x,
// + grid_tiles, ..., a CTA of the second group the listed edge blocks likewise.  The first CTA of each group also
// publishes the grid totals.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
scan_prefix_kernel(const unsigned* __restrict__ m1_words, const unsigned* __restrict__ m2_words,
                   const unsigned* __restrict__ tile_cnt, int64_t ntiles,
                   uint2* __restrict__ tet_word_prefix, const unsigned* __restrict__ edge_bits,
                   const unsigned* __restrict__ eblock_cnt, int64_t n_eblocks,
                   unsigned* __restrict__ word_prefix, DevCounters* __restrict__ ctr, int64_t cap_records,
                   const unsigned* __restrict__ q_cnt, int64_t cap_qe, int64_t cap_qv, unsigned grid_tiles,
                   const __grid_constant__ FrameSet fs, const __grid_constant__ FrameSet also, int n_also) {
  pdl_enter();
  {
    const int64_t shift = fs.off[blockIdx.y];
    m1_words = frame_ptr(m1_words, shift); m2_words = frame_ptr(m2_words, shift); tile_cnt = frame_ptr(tile_cnt, shift);
    tet_word_prefix = frame_ptr(tet_word_prefix, shift); edge_bits = frame_ptr(edge_bits, shift);
    eblock_cnt = frame_ptr(eblock_cnt, shift); word_prefix = frame_ptr(word_prefix, shift); ctr = frame_ptr(ctr, shift);
    q_cnt = frame_ptr(q_cnt, shift);
  }
  constexpr int WARPS = 256 / 32;
  __shared__ unsigned long long s_sum[WARPS];
  __shared__ unsigned long long s_w[WARPS];
  const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
  const bool tiles = blockIdx.x < grid_tiles;
  const unsigned first = tiles ? blockIdx.x : blockIdx.x - grid_tiles;
  const unsigned stride = tiles ? grid_tiles : gridDim.x - grid_tiles;
  const unsigned* __restrict__ cnt = tiles ? tile_cnt : eblock_cnt;
  const int64_t n_all = tiles ? ntiles : n_eblocks;
  unsigned long long* tr = trace_begin(ctr->trace, ctr->trace_frame, K_COMPACT);

  if (first == 0u) {   // totals of the whole grid
    unsigned long long sum = 0ull;
    for (int64_t i = threadIdx.x; i < n_all; i += 256) {
      const unsigned c = __ldcg(cnt + i);
      sum += tiles ? ((unsigned long long)(c & 0xffffu) | ((unsigned long long)(c >> 16) << 32)) : (unsigned long long)c;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) s_sum[warp] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long tot = 0ull;
      for (int w = 0; w < WARPS; ++w) tot += s_sum[w];
      if (tiles) {
        const unsigned t1 = (unsigned)(tot & 0xffffffffull), t2 = (unsigned)(tot >> 32);
        ctr->n_tri = t1;
        ctr->n_quad = t2;
        // a sub-queue that overflowed dropped entries: crossing edges whose tets were never marked, or valid tets that
        // never become records.  Report enough valid tets for the caller to grow (the counts of an overflowed call only
        // serve that purpose)
        int64_t raw = 0, max_e = 0, max_v = 0;
        for (int q = 0; q < kQueues; ++q) {
          const int64_t ne = (int64_t)q_cnt[kQStride * q], nt = (int64_t)q_cnt[kQStride * (kQueues + q)];
          raw += ne;
          max_e = ne > max_e ? ne : max_e;
          max_v = nt > max_v ? nt : max_v;
        }
        const bool dropped = q_cnt[kQStride * (3 * kQueues + 2)] != 0u;   // run-length tables: an item list was too small
        const bool queue_ok = max_e <= cap_qe && max_v <= cap_qv && !dropped;
        // records needed for every sub-queue to hold what it was offered (a sub-queue has 1/8 of the record capacity
        // for tets and 1/2 of it for edges), and the expected number of valid tets when none could be marked yet
        int64_t need = 2 * raw;
        need = 8 * max_v > need ? 8 * max_v : need;
        need = 2 * max_e > need ? 2 * max_e : need;
        need = cap_records + 1 > need ? cap_records + 1 : need;
        if (dropped) need = 2 * cap_records > need ? 2 * cap_records : need;
        ctr->n_valid = queue_ok ? t1 + t2 : max(t1 + t2, (unsigned)need);
        const bool fits = queue_ok && (int64_t)t1 + t2 <= cap_records;
        ctr->work_tri = fits ? t1 : 0u;
        ctr->work_quad = fits ? t2 : 0u;
        for (int f = 1; f < n_also; ++f) {   // frames that share this topology (BatchCtx): the totals into their counters too
          DevCounters* c2 = frame_ptr(ctr, also.off[f] - also.off[0]);
          c2->n_tri = t1; c2->n_quad = t2; c2->n_valid = ctr->n_valid; c2->work_tri = ctr->work_tri; c2->work_quad = ctr->work_quad;
        }
      } else {
        ctr->n_verts = (unsigned)tot;
        for (int f = 1; f < n_also; ++f) frame_ptr(ctr, also.off[f] - also.off[0])->n_verts = (unsigned)tot;
      }
    }
    __syncthreads();
  }

  for (int64_t id = first; id < n_all; id += stride) {
    if (__ldcg(cnt + id) == 0u) continue;   // most tiles / blocks hold no surface (block-uniform)
    unsigned long long sum = 0ull;   // tiles: T1 in the low half, T2 in the high half
    for (int64_t i = threadIdx.x; i < id; i += 256) {
      const unsigned c = __ldcg(cnt + i);
      sum += tiles ? ((unsigned long long)(c & 0xffffu) | ((unsigned long long)(c >> 16) << 32)) : (unsigned long long)c;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const int64_t w = id * 256 + threadIdx.x;
    unsigned long long c;
    if (tiles) c = (unsigned long long)__popc(__ldcg(m1_words + w)) | ((unsigned long long)__popc(__ldcg(m2_words + w)) << 32);
    else c = (unsigned long long)__popc(__ldcg(edge_bits + w));
    unsigned long long incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long nb = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (unsigned)o) incl += nb;
    }
    if (lane == 0) s_sum[warp] = sum;
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    unsigned long long excl = 0ull, wpre = 0ull;
#pragma unroll
    for (int q = 0; q < WARPS; ++q) {
      excl += s_sum[q];
      if (q < (int)warp) wpre += s_w[q];
    }
    const unsigned long long pre = excl + wpre + incl - c;
    if (tiles) tet_word_prefix[w] = make_uint2((unsigned)(pre & 0xffffffffull), (unsigned)(pre >> 32));
    else if (c) word_prefix[w] = (unsigned)pre;
    __syncthreads();   // s_sum / s_w are rewritten by the next trip
  }
  trace_end(tr);
}

// ------------------------------------------------------------------------------------------------
// one thread per queue entry.  CTAs [0, grid_tets) take the valid tets, the others the crossing edges; CTA c of either
// group serves sub-queue c % kQueues.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
scan_emit_kernel(const FwdBlock* __restrict__ blk, const DevCounters* __restrict__ ctr, const int2* __restrict__ vlist,
                 const int32_t* __restrict__ elist, int filtered, const unsigned* __restrict__ m1_words,
                 const unsigned* __restrict__ m2_words, const uint2* __restrict__ tet_word_prefix,
                 const unsigned* __restrict__ edge_bits, const unsigned* __restrict__ word_prefix,
                 d3h_tet_record* __restrict__ records, float4* __restrict__ w_vert, float4* __restrict__ w_acc,
                 int64_t cap_corners, const unsigned* __restrict__ q_cnt, int64_t cap_qe, int64_t cap_qv, unsigned grid_tets,
                 const __grid_constant__ FrameSet fs, const __grid_constant__ FrameSet topo) {
  pdl_enter();
  {
    // what the frame writes sits in its own workspace, the topology it reads possibly in the first frame's (BatchCtx)
    const int64_t shift = fs.off[blockIdx.y], tshift = topo.off[blockIdx.y];
    // ... and then the records and corner ids are the first frame's business alone (poly_faces_kernel reads them there)
    if (shift != tshift && blockIdx.x < grid_tets) return;
    blk = frame_ptr(blk, shift); ctr = frame_ptr(ctr, shift); records = frame_ptr(records, shift);
    w_vert = frame_ptr(w_vert, shift); w_acc = frame_ptr(w_acc, shift);
    vlist = frame_ptr(vlist, tshift); elist = frame_ptr(elist, tshift); m1_words = frame_ptr(m1_words, tshift);
    m2_words = frame_ptr(m2_words, tshift); tet_word_prefix = frame_ptr(tet_word_prefix, tshift);
    edge_bits = frame_ptr(edge_bits, tshift); word_prefix = frame_ptr(word_prefix, tshift); q_cnt = frame_ptr(q_cnt, tshift);
  }
  const d3h_forward_args& a = blk->a;
  unsigned long long* tr = trace_begin(ctr->trace, ctr->trace_frame, K_EDGE_EMIT);
  if (blockIdx.x < grid_tets) {
    // ---- valid tets -> records (tet order) + polygon corner -> vertex id ----
    const unsigned t1 = ctr->work_tri, t2 = ctr->work_quad;   // 0 / 0 when the record buffer is too small
    const unsigned q = blockIdx.x % kQueues, part = blockIdx.x / kQueues, parts = grid_tets / kQueues;
    const int64_t n = (t1 + t2 == 0u) ? 0 : (int64_t)q_cnt[kQStride * (kQueues + q)];   // (fits: checked by scan_prefix_kernel)
    vlist += (int64_t)q * cap_qv;
    const int4* __restrict__ tets = reinterpret_cast<const int4*>(a.tets);
    const int4* __restrict__ ranks = reinterpret_cast<const int4*>(a.tet_edge_rank);
    int32_t* __restrict__ corners = a.tape_corners;
    for (int64_t j = (int64_t)part * 256 + threadIdx.x; j < n; j += (int64_t)parts * 256) {
      const int2 it = vlist[j];
      const int t = it.x, code = it.y;
      const int4 v4 = __ldg(tets + t);
      const int4 r03 = __ldg(ranks + 2 * (int64_t)t), r45 = __ldg(ranks + 2 * (int64_t)t + 1);
      const unsigned w = (unsigned)t >> 5, below = (1u << (t & 31)) - 1u;
      const uint2 pre = tet_word_prefix[w];
      const unsigned g1 = pre.x + __popc(__ldcg(m1_words + w) & below), g2 = pre.y + __popc(__ldcg(m2_words + w) & below);
      const bool quad = __popc((unsigned)code) == 2;
      const unsigned cr = quad ? g2 : g1, ob = quad ? g1 : g2;
      int4* out = reinterpret_cast<int4*>(records + ((int64_t)g1 + g2));
      out[0] = v4;
      out[1] = make_int4(code, (int)cr, t, (int)ob);
      const int nc = quad ? 4 : 3;
      const int64_t p0 = quad ? (3ll * t1 + 4ll * cr) : 3ll * cr;
      const int rr[6] = {r03.x, r03.y, r03.z, r03.w, r45.x, r45.y};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (k < nc) {
          const int e = c_loop_edge[code][k];
          unsigned r = 0;
#pragma unroll
          for (int q = 0; q < 6; ++q)
            if (q == e) r = (unsigned)rr[q];   // select without dynamic register indexing
          corners[p0 + k] = (int)(__ldcg(word_prefix + (r >> 5)) + __popc(__ldcg(edge_bits + (r >> 5)) & ((1u << (r & 31u)) - 1u)));
        }
      }
    }
  } else {
    // ---- crossing edges -> watertight vertices (zero-crossing interpolation, gshell_tets.py:291-303) ----
    const unsigned c = blockIdx.x - grid_tets, grid_edges = gridDim.x - grid_tets;
    const unsigned q = c % kQueues, part = c / kQueues, parts = grid_edges / kQueues;
    const int64_t nq = (int64_t)q_cnt[kQStride * ((filtered ? 2 : 0) * kQueues + q)];
    const int64_t n = nq < cap_qe ? nq : cap_qe;
    elist += (int64_t)q * cap_qe;
    const int2* __restrict__ edge_ab = reinterpret_cast<const int2*>(a.edge_ab);
    const float* __restrict__ pos = a.pos;
    const float* __restrict__ sdf = a.sdf;
    const float* __restrict__ msdf = a.msdf;
    const int msdf_negate = a.msdf_negate;
    const int64_t cap_verts = a.cap_verts, cap_verts_aug = a.cap_verts_aug;
    float4* __restrict__ vacc = reinterpret_cast<float4*>(a.vacc);
    for (int64_t j = (int64_t)part * 256 + threadIdx.x; j < n; j += (int64_t)parts * 256) {
      const unsigned e = (unsigned)elist[j];
      const int2 ab = __ldg(edge_ab + e);
      const int64_t vid = (int64_t)__ldcg(word_prefix + (e >> 5)) + __popc(__ldcg(edge_bits + (e >> 5)) & ((1u << (e & 31u)) - 1u));
      if (vid >= cap_corners) continue;   // (cannot happen while the records fit: V <= 4 Fv)
      const int ea = ab.x, eb = ab.y;
      float w0, w1, dd;
      crossing_weights(__ldg(sdf + ea), __ldg(sdf + eb), w0, w1, dd);
      float ma = __ldg(msdf + ea), mb = __ldg(msdf + eb);
      if (msdf_negate) { ma = -ma; mb = -mb; }
      const float x = lerp2(__ldg(pos + 3ll * ea + 0), w0, __ldg(pos + 3ll * eb + 0), w1);
      const float y = lerp2(__ldg(pos + 3ll * ea + 1), w0, __ldg(pos + 3ll * eb + 1), w1);
      const float z = lerp2(__ldg(pos + 3ll * ea + 2), w0, __ldg(pos + 3ll * eb + 2), w1);
      const float m = lerp2(ma, w0, mb, w1);
      w_vert[vid] = make_float4(x, y, z, m);
      w_acc[2 * vid] = make_float4(0.f, 0.f, 0.f, 0.f);
      w_acc[2 * vid + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (vid < cap_verts) {
        reinterpret_cast<int2*>(a.tape_edges)[vid] = make_int2(ea, eb);
        a.verts_wt[3 * vid] = x; a.verts_wt[3 * vid + 1] = y; a.verts_wt[3 * vid + 2] = z;
        a.msdf_wt[vid] = m;
        vacc[2 * vid] = make_float4(0.f, 0.f, 0.f, 0.f);
        vacc[2 * vid + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (vid < cap_verts_aug) {
        // rows of verts_aug not referenced by faces_aug are zero (gshell_tets.py:423-427); a watertight vertex is
        // referenced iff its mSDF is positive (every cut case keeps exactly the positive corners)
        const bool used = m > 0.f;
        a.verts_aug[3 * vid] = used ? x : 0.f;
        a.verts_aug[3 * vid + 1] = used ? y : 0.f;
        a.verts_aug[3 * vid + 2] = used ? z : 0.f;
        a.msdf_aug[vid] = m;
      }
    }
  }
  trace_end(tr);
}

static ScanLists scan_lists(const d3h_forward_args& a, const Workspace& ws) {
  ScanLists L;
  L.tile_cnt = ws.tile_cnt;
  L.eblock_cnt = ws.eblock_cnt;
  L.q_cnt = ws.q_cnt;
  L.vlist = ws.vlist;
  L.elist_raw = ws.elist;
  L.elist = a.watertight_template ? ws.elist : ws.elist2;
  L.cap_qe = ws.cap_qe; L.cap_qv = ws.cap_qv;
  return L;
}

static void launch_scan_runs(const d3h_forward_args& a, const Workspace& ws, const ScanLists& L, cudaStream_t stream, bool dep,
                             bool expand) {
  const bool both = a.tet_runs != nullptr && a.watertight_template;
  const unsigned nbe = (unsigned)((a.n_edge_runs + kEScanThreads - 1) / kEScanThreads);
  const unsigned nbt = both ? (unsigned)((a.n_tet_runs + kEScanThreads - 1) / kEScanThreads) : 0u;
  EdgeItem* eitems = reinterpret_cast<EdgeItem*>(ws.elist2);
  TetItem* titems = reinterpret_cast<TetItem*>(ws.records);
  const int64_t cap_e = ws.cap_qe * kQueues * 4 / (int64_t)sizeof(EdgeItem), cap_t = ws.cap_tets;
  {
    ProfScope ps(K_EDGE_SCAN, stream);
    auto go = [&](auto kernel) {
      if (dep) launch_k_dep(kernel, nbe + nbt, (unsigned)kEScanThreads, stream, kLaunchLatency, ws.blk, ws.occ_bits, L, eitems, cap_e, titems, cap_t, nbe, batch_ctx().topo);
      else launch_k(kernel, nbe + nbt, (unsigned)kEScanThreads, stream, kLaunchLatency, ws.blk, ws.occ_bits, L, eitems, cap_e, titems, cap_t, nbe, batch_ctx().topo);
    };
    if (both) go(scan_runs_kernel<true>);
    else go(scan_runs_kernel<false>);
  }
  if (!expand) return;
  // a warp per item; the lists hold a few thousand to a few ten thousand items: one wave of CTAs, a few items per warp
  ProfScope ps(K_EDGE_MARK, stream);
  const unsigned nblk = 148u * 8u;
  const unsigned ctas_edges = both ? (nblk * 2u) / 5u : nblk;
  if (both)
    launch_k_dep(runs_expand_kernel<true>, nblk, 256u, stream, kLaunchLatency, ws.blk, ws.m1_words, ws.m2_words, ws.edge_bits, L,
                 (const EdgeItem*)eitems, cap_e, (const TetItem*)titems, cap_t, ctas_edges, batch_ctx().topo);
  else
    launch_k_dep(runs_expand_kernel<false>, nblk, 256u, stream, kLaunchLatency, ws.blk, ws.m1_words, ws.m2_words, ws.edge_bits, L,
                 (const EdgeItem*)eitems, cap_e, (const TetItem*)titems, cap_t, ctas_edges, batch_ctx().topo);
}

void launch_edge_scan_only(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream) {
  const ScanLists L = scan_lists(a, ws);
  if (a.edge_runs != nullptr) {   // pass A of launch_scan_runs (its counts land in scratch state)
    launch_scan_runs(a, ws, L, stream, /*dep=*/false, /*expand=*/false);
    return;
  }
  if (a.edge_rows != nullptr) {
    launch_scan_rows(a, [&](auto kernel, unsigned nblk) {
      launch_k(kernel, nblk, (unsigned)kEScanThreads, stream, kLaunchStream, ws.blk, ws.occ_bits, L);
    });
    return;
  }
  const int vpt = scan_vpt();
  const int64_t per_cta = (int64_t)kEScanThreads * vpt;
  const unsigned nblk = (unsigned)((a.n_grid + per_cta - 1) / per_cta);
  if (vpt == 1) launch_k(edge_scan_kernel<1>, nblk, (unsigned)kEScanThreads, stream, kLaunchStream, ws.blk, ws.occ_bits, L);
  else if (vpt == 2) launch_k(edge_scan_kernel<2>, nblk, (unsigned)kEScanThreads, stream, kLaunchStream, ws.blk, ws.occ_bits, L);
  else launch_k(edge_scan_kernel<4>, nblk, (unsigned)kEScanThreads, stream, kLaunchStream, ws.blk, ws.occ_bits, L);
}

void launch_edge_scan(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream) {
  ScanLists L;
  L.tile_cnt = ws.tile_cnt;
  L.eblock_cnt = ws.eblock_cnt;
  L.q_cnt = ws.q_cnt;
  L.vlist = ws.vlist;
  L.elist_raw = ws.elist;
  // with the open-mesh prefilter the marking kernel re-queues the edges that survive
  const int filtered = a.watertight_template ? 0 : 1;
  L.elist = filtered ? ws.elist2 : ws.elist;
  L.cap_qe = ws.cap_qe; L.cap_qv = ws.cap_qv;
  const bool runs_both = a.tet_runs != nullptr && a.edge_runs != nullptr && !filtered;
  // the kernels that find the topology run once for frames that share it (BatchCtx); restored before the emit kernel
  BatchCtx& ctx = batch_ctx();
  const int all_frames = ctx.frames;
  ctx.frames = ctx.topo_frames;
  // CTAs per sub-queue of the consumers: enough for one entry per thread at the expected fill (a sub-queue holds
  // 8 / kQueues of the capacity; the expected fill is 1 / kQueues of it)
  auto parts_for = [](int64_t cap_q) {
    int64_t p = (cap_q / 8 + 255) / 256;
    return (unsigned)(p < 1 ? 1 : (p > 16 ? 16 : p));
  };
  if (ctx.reuse_topology && runs_both) {
    // the launch before found this topology in this very workspace: straight to the per-frame kernels
    ctx.frames = all_frames;
    if (ws.cap_corners <= 0) return;
    ProfScope ps(K_EDGE_EMIT, stream);
    const unsigned gt = kQueues * parts_for(ws.cap_qv), ge = kQueues * parts_for(ws.cap_qe);
    launch_k_dep(scan_emit_kernel, gt + ge, 256u, stream, kLaunchLatency, ws.blk, ws.ctr, ws.vlist, L.elist, filtered, ws.m1_words,
                 ws.m2_words, ws.tet_word_prefix, ws.edge_bits, ws.word_prefix, ws.records, ws.vert,
                 reinterpret_cast<float4*>(ws.acc), ws.cap_corners, ws.q_cnt, ws.cap_qe, ws.cap_qv, gt, batch_ctx().fs, batch_ctx().topo);
    return;
  }
  if (a.edge_runs != nullptr) {
    // crossing edges from the compressed edge list and, with the compressed tet array (watertight template), the valid
    // tets as well: pass A tests every entry, pass B expands the few that found something -- no marking kernel
    launch_scan_runs(a, ws, L, stream, /*dep=*/true, /*expand=*/true);
  } else {
    ProfScope ps(K_EDGE_SCAN, stream);
    const int vpt = scan_vpt();
    const int64_t per_cta = (int64_t)kEScanThreads * vpt;
    const unsigned nblk = (unsigned)((a.n_grid + per_cta - 1) / per_cta);
    if (a.edge_rows != nullptr) {
      launch_scan_rows(a, [&](auto kernel, unsigned nb) {
        launch_k_dep(kernel, nb, (unsigned)kEScanThreads, stream, kLaunchStream, ws.blk, ws.occ_bits, L);
      });
    } else if (vpt == 1)
      launch_k_dep(edge_scan_kernel<1>, nblk, (unsigned)kEScanThreads, stream, kLaunchStream, ws.blk, ws.occ_bits, L);
    else if (vpt == 2)
      launch_k_dep(edge_scan_kernel<2>, nblk, (unsigned)kEScanThreads, stream, kLaunchStream, ws.blk, ws.occ_bits, L);
    else
      launch_k_dep(edge_scan_kernel<4>, nblk, (unsigned)kEScanThreads, stream, kLaunchStream, ws.blk, ws.occ_bits, L);
  }
  if (!runs_both) {
    ProfScope ps(K_EDGE_MARK, stream);
    const unsigned nblk = kQueues * parts_for(ws.cap_qe);
    // opt-in (the host passes etets8 only with D3H_MARK_ROWS=1): measured 22.1 us against 23.6 us for the default on the
    // 128^3 capsule frame (r02h) -- not worth the 32 bytes per edge of the table by default
    const bool rows = a.etets8 != nullptr;
    if (!filtered)
      launch_k_dep(rows ? edge_mark_rows_kernel<false> : edge_mark_kernel<false>, nblk, 256u, stream, kLaunchLatency, ws.blk,
               ws.occ_bits, (const unsigned*)nullptr, ws.m1_words, ws.m2_words, ws.edge_bits, L);
    else
      launch_k_dep(rows ? edge_mark_rows_kernel<true> : edge_mark_kernel<true>, nblk, 256u, stream, kLaunchLatency, ws.blk,
               ws.occ_bits, ws.mocc_bits, ws.m1_words, ws.m2_words, ws.edge_bits, L);
  }
  const int64_t maxg = 148 * 4;
  {
    ProfScope ps(K_COMPACT, stream);
    const unsigned gt = (unsigned)(ws.ntiles_compact < maxg ? ws.ntiles_compact : maxg);
    const unsigned ge = (unsigned)(ws.n_eblocks < maxg ? ws.n_eblocks : maxg);
    launch_k_dep(scan_prefix_kernel, gt + ge, 256u, stream, kLaunchLatency, ws.m1_words, ws.m2_words, ws.tile_cnt,
             ws.ntiles_compact, ws.tet_word_prefix, ws.edge_bits, ws.eblock_cnt, ws.n_eblocks, ws.word_prefix, ws.ctr,
             ws.cap_tets, ws.q_cnt, ws.cap_qe, ws.cap_qv, gt, batch_ctx().topo, batch_ctx().fs,
             batch_ctx().topo_frames == 1 ? all_frames : 1);
  }
  ctx.frames = all_frames;
  if (ws.cap_corners <= 0) return;   // counting run: sizes only
  ProfScope ps(K_EDGE_EMIT, stream);
  const unsigned gt = kQueues * parts_for(ws.cap_qv), ge = kQueues * parts_for(ws.cap_qe);
  launch_k_dep(scan_emit_kernel, gt + ge, 256u, stream, kLaunchLatency, ws.blk, ws.ctr, ws.vlist, L.elist, filtered, ws.m1_words,
           ws.m2_words, ws.tet_word_prefix, ws.edge_bits, ws.word_prefix, ws.records, ws.vert,
           reinterpret_cast<float4*>(ws.acc), ws.cap_corners, ws.q_cnt, ws.cap_qe, ws.cap_qv, gt, batch_ctx().fs, batch_ctx().topo);
}

}  // namespace d3h

// The SDF sign-change regulariser reads the same run-length tables with the same sign windows: its kernels and entry
// points are compiled in this translation unit, so the library and its CPU emulation (tests/emu) build them from their
// existing source lists.
#include "d3h_sdf_reg.cu"
