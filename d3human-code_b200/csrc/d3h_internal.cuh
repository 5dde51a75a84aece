// Internal (non-ABI) declarations shared by the translation units of libd3h_tets.so.
#pragma once

#include <cstring>

#include "d3h_common.cuh"

namespace d3h {

// ---- tile shapes ----------------------------------------------------------------------------------
constexpr int kClassifyThreads = 256;
constexpr int kClassifyItems = 8;   // tets per lane: 8 x 16 B loads in flight, one ballot word per item
constexpr int kChunkTets = 32 * kClassifyItems;  // tets one warp classifies per loop trip (256)

constexpr int kCompactThreads = 256;             // one bitmap word (32 tets) per thread
constexpr int kTileTets = 32 * kCompactThreads;  // tets per compaction tile (8192 = 32 warp chunks)

constexpr int kMsdBits = 17;        // MSD radix digit: top bits of the smaller endpoint (<= 131072 buckets)
constexpr int kScanThreads = 1024;  // bucket_scan: one bucket per thread
constexpr int kSortGroup = 256;     // group quantum of the block-local finish
constexpr int kLocalSortCap = 2048; // keys a CTA sorts in shared memory (24 KB); larger groups use global scratch
constexpr int kUniqueThreads = 256;  // threads of the group sort / vertex emission CTAs

constexpr int kPolyThreads = 256;   // one valid tet (= one polygon) per thread

// ---- per-call argument block --------------------------------------------------------------------------
// Everything that changes from call to call (input / output / tape pointers, output capacities, seq) lives in ONE block
// in device memory.  The first kernel of the forward sequence receives it by value and stores it; every later kernel
// reads it through a pointer that is fixed for the workspace.  Launch shapes depend only on (F, N, tet range,
// cap_valid_tets), so the whole forward sequence is a CUDA graph that is captured once per shape and re-launched with
// a single parameter update (3-4 us of host time and a 2.9 us device gap per stream launch on this box versus 1.1 us
// per graph and 0.7 us per kernel node: profiles/bench_launch.cu).
struct FwdBlock {
  d3h_forward_args a;
  d3h_counts* counts_mapped;  // device alias of a.counts_host, or nullptr
  unsigned long long* trace;  // diagnostics: device trace table (d3h_trace_enable) or nullptr
};
unsigned long long* trace_table();  // current device trace table or nullptr

// ---- workspace ------------------------------------------------------------------------------------
// Every region is 256-byte aligned.  Sizes depend on (F, N, cap_valid_tets) only.
struct Workspace {
  DevCounters* ctr;               // 128 B
  FwdBlock* blk;                  // the per-call argument block
  FwdBlock* blk2;                 // argument block of the second extraction of a cloth / body pair
  d3h_counts* counts;             // device copy of the public counts
  d3h_counts* counts2;            // ... of the second extraction of a cloth / body pair
  unsigned* occ_bits;             // ceil(N/32) words: sdf > 0
  unsigned* mocc_bits;            // ceil(N/32) words: (+-)msdf > 0 (open-mesh prefilter only)
  unsigned* m1_words;             // ceil(F/32) words: tet yields one triangle
  unsigned* m2_words;             // ceil(F/32) words: tet yields two triangles
  unsigned* tile_cnt;             // per compaction tile: T1-class count | T2-class count << 16
  d3h_tet_record* records;        // cap_valid_tets
  unsigned long long* keys;       // 4*cap_valid_tets: edge keys in valid-tet order
  unsigned* vals;
  unsigned long long* keys2;      // 4*cap_valid_tets: partitioned by bucket (unsorted inside a bucket)
  unsigned* vals2;
  unsigned long long* keys_scratch;  // 8*cap_valid_tets: padded copies of oversized groups
  unsigned* vals_scratch;
  unsigned* msd_hist;             // msd_bins (+pad): keys per bucket
  unsigned* msd_fill;             // msd_bins: absolute scatter cursors of the partition pass
  unsigned* msd_base;             // msd_bins + 1: exclusive scan of msd_hist
  unsigned long long* st_scan;    // one status word per bucket_scan CTA
  unsigned* group_start;          // cap_corners / kSortGroup + 2: first key of every block-local sort group
  int64_t msd_bins;               // buckets actually used for this grid: ((N-1) >> msd_shift) + 1
  unsigned* group_heads;          // distinct keys of every sort group
  unsigned* gblock_heads;         // distinct keys of every 256 sort groups
  unsigned* poly_cnt;             // ntiles_poly * 8: polygons per faces_aug bucket in each polygon tile
  unsigned* poly_excl;            // ntiles_poly * 8: exclusive prefix of poly_cnt over the tiles
  unsigned* poly_gcnt;            // ntiles_poly * 8 * 8: the same counts per group of 32 polygons
  unsigned char* poly_used;       // cap_valid_tets: per polygon, the boundary vertices its mSDF cut references (bit k: edge k -> k+1)
  float4* vert;                   // (x,y,z,msdf) per watertight vertex, 4*cap_valid_tets
  float* acc;                     // 8 floats per watertight vertex: normal xyz + count, tangent xyz + pad
  int32_t* owner;                 // per watertight vertex: the polygon corner slot that writes its tangent rows
  // static edge table path (n_edges > 0)
  unsigned* edge_bits;            // ceil(n_edges/32) words: edge is crossed by a valid tet of this call
  unsigned* word_prefix;          // per word of edge_bits: number of marked edges before it (= first vertex id of the word)
  unsigned* eblock_cnt;           // marked edges per 8192-edge block (one edge_emit CTA)
  unsigned* corner_rank;          // 4 per valid-tet record: edge rank of every polygon corner
  // edge-scan path: unordered work queues, kQueues sub-queues each (see d3h_scan.cu)
  unsigned* q_cnt;                // [4][kQueues] entries appended per sub-queue: raw edges, valid tets, filtered edges; [3]: items of the run-length scan
  int2* vlist;                    // kQueues x cap_qv: (tet id, occupancy code) of every valid tet
  int32_t* elist;                 // kQueues x cap_qe: rank of every crossing edge
  int32_t* elist2;                // kQueues x cap_qe: ... that survives the open-mesh prefilter
  int64_t cap_qe, cap_qv;         // entries per sub-queue
  uint2* tet_word_prefix;         //                 per word of m1 / m2: (T1-class, T2-class) valid tets before it
  int64_t n_edges, n_eblocks;
  int64_t nwords_tet;             // words of m1_words / m2_words (32 tets each), padded to whole compaction tiles
  int64_t cap_tets, cap_corners;
  int64_t ntiles_compact, nscan_ctas, ngroups, ntiles_poly;
  int64_t total_bytes;
};

// the same workspace of another frame of the launch (see FrameSet below): every region moved by `shift` bytes
__device__ __forceinline__ void shift_workspace(Workspace& w, int64_t shift) {
#define D3H_SHIFT(m) w.m = w.m ? reinterpret_cast<decltype(w.m)>(reinterpret_cast<uintptr_t>(w.m) + shift) : w.m
  D3H_SHIFT(ctr); D3H_SHIFT(blk); D3H_SHIFT(blk2); D3H_SHIFT(counts); D3H_SHIFT(counts2); D3H_SHIFT(occ_bits);
  D3H_SHIFT(mocc_bits); D3H_SHIFT(m1_words); D3H_SHIFT(m2_words); D3H_SHIFT(tile_cnt); D3H_SHIFT(records); D3H_SHIFT(keys);
  D3H_SHIFT(vals); D3H_SHIFT(keys2); D3H_SHIFT(vals2); D3H_SHIFT(keys_scratch); D3H_SHIFT(vals_scratch); D3H_SHIFT(msd_hist);
  D3H_SHIFT(msd_fill); D3H_SHIFT(msd_base); D3H_SHIFT(st_scan); D3H_SHIFT(group_start); D3H_SHIFT(group_heads);
  D3H_SHIFT(gblock_heads); D3H_SHIFT(poly_cnt); D3H_SHIFT(poly_excl); D3H_SHIFT(poly_gcnt); D3H_SHIFT(poly_used);
  D3H_SHIFT(vert); D3H_SHIFT(acc);
  D3H_SHIFT(owner); D3H_SHIFT(edge_bits); D3H_SHIFT(word_prefix); D3H_SHIFT(eblock_cnt); D3H_SHIFT(corner_rank);
  D3H_SHIFT(q_cnt); D3H_SHIFT(vlist); D3H_SHIFT(elist); D3H_SHIFT(elist2); D3H_SHIFT(tet_word_prefix);
#undef D3H_SHIFT
}

// Carves `base` (may be nullptr when only the size is wanted).
Workspace carve_workspace(void* base, int64_t n_tets, int64_t n_grid, int64_t cap_valid_tets, int64_t n_edges = 0);
constexpr int kQueues = 64;        // sub-queues of the edge-scan path's work queues
constexpr int kQStride = 32;       // words between two sub-queue counters (one 128-byte line each)
constexpr int kEdgeBlock = 8192;  // edges per edge_emit CTA (256 threads x one 32-bit word)

int key_bits_for(int64_t n_grid);   // bits per endpoint in the packed edge key
int msd_shift_for(int64_t n_grid);  // endpoint >> shift = MSD bucket

// grid size of a persistent kernel: SM count x resident CTAs per SM (queried once per kernel)
int persistent_grid(const void* kernel, int threads, size_t dyn_smem);

// ---- stage launchers (all asynchronous on `stream`) -------------------------------------------------
void launch_prepare(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream);
void launch_prepare_frames(const d3h_forward_args* a, const Workspace& ws, cudaStream_t stream);
// the forward sequence behind launch_prepare; `a` only supplies the launch shapes, the kernels read the block
// parts of a forward call: the head is the bandwidth-bound part (the O(F) classification stream behind prepare_kernel),
// the tail everything that works on the O(surface) records.  A batch runs the heads of all frames back to back on one
// stream and the tails on the lanes.
enum ForwardParts { kPartHead = 1, kPartTail = 2, kPartAll = 3 };
void launch_forward_sequence(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream, int parts = kPartAll,
                             cudaStream_t side = nullptr, cudaEvent_t fork = nullptr, cudaEvent_t join = nullptr);
void launch_classify(const d3h_forward_args& a, const Workspace& ws, d3h_tet_record* records, int64_t cap_records,
                     bool emit_keys, cudaStream_t stream, int parts = kPartAll);
void launch_edge_sort(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream);
void launch_edge_emit(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream);  // static edge table path
// edge-scan path (d3h_forward_args.etets): replaces the classification stream + compaction by a walk over the static edge
// list, then compacts / numbers only the tiles and edge blocks that were marked
void launch_edge_scan(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream);
inline bool edge_scan_path(const d3h_forward_args& a) { return a.edge_off != nullptr && a.etets != nullptr; }
void launch_edge_scan_only(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream);   // diagnostics: the stream kernel alone
void launch_surface(const d3h_forward_args& a, const Workspace& ws, const d3h_tet_record* records,
                    cudaStream_t stream);
// second extraction of a cloth / body pair: replays the mSDF cut on the shared surface (d3h_forward_args.pair_*)
void launch_pair_replay(const d3h_forward_args& a, const Workspace& ws, const d3h_tet_record* records,
                        cudaStream_t stream);
void launch_rank_records(const d3h_forward_args& a, const Workspace& ws, d3h_tet_record* records, int64_t n_records,
                         cudaStream_t stream);
void launch_zero_grads_from_block(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream);
void launch_backward(const d3h_backward_args& a, cudaStream_t stream);
void launch_backward_batch(const d3h_backward_args* a, int64_t n, cudaStream_t stream);

void set_error(const char* fmt, ...);

// ---- launches with a scheduling priority ------------------------------------------------------------------------
// Frames of a batch run on concurrent lanes (d3h_extract_forward_batch).  The O(surface) kernels are dependency-latency
// bound and use a fraction of the SMs; the O(F) / O(N) streams are bandwidth bound and would occupy every CTA slot for
// their whole duration.  Launching the streams at the lowest priority and everything else at the highest lets the block
// scheduler slip the surface CTAs of one frame in between the retiring CTAs of another frame's stream, so the latency
// chains hide under the HBM traffic.  The priority is a per-launch attribute (also recorded in captured graph nodes).
enum LaunchClass { kLaunchStream = 0, kLaunchLatency = 1 };
int launch_priority(LaunchClass c);

// ---- several frames in ONE launch (d3h_extract_forward_batch on the run-length tables) ---------------------------------
// With one graph per frame on concurrent lanes a 32-frame step is 256 kernel nodes of a few microseconds each, and the
// front end starts one node per ~5 us whatever the lanes (r02ac: the kernels of a frame sum to 60 us, its span on a lane is
// 244 us).  The kernels of the run-length path therefore take the frame from blockIdx.y: every workspace pointer they
// are given belongs to frame 0, FrameSet.off[f] is the byte offset of frame f's workspace (all frames of a launch have
// the same capacities, hence the same layout).  A single call is a launch with one frame and offset 0.
constexpr int kMaxFused = 8;
struct FrameSet {
  int64_t off[kMaxFused];
};
struct FwdBlockSet {   // the argument blocks of the frames of a launch, by value (kernel parameters may take 32 KB)
  FwdBlock f[kMaxFused];
};
struct BatchCtx {
  int frames;     // gridDim.y of every launch made through launch_k / launch_k_dep
  FrameSet fs;
  // Frames that share sdf, msdf and the template have ONE topology (crossing edges, valid tets, their numbering): it is
  // found once, in the workspace of the launch's first frame, and only the kernels that touch positions (vertex
  // interpolation, normals / tangents, the mSDF cut with its boundary vertices) run per frame.  topo.off[f] is where
  // frame f finds the topology: 0 when shared, fs.off[f] otherwise; topo_frames = 1 when shared, frames otherwise.
  int topo_frames;
  FrameSet topo;
  // a later launch of the same call whose frames share the topology of an earlier launch AND whose first frame lives in
  // the workspace that holds it: nothing is searched again, the frames only get their argument blocks and the totals
  bool reuse_topology;
};
BatchCtx& batch_ctx();   // of the calling thread; one frame, zero offsets outside d3h_extract_forward_batch
template <typename T>
__device__ __forceinline__ T* frame_ptr(T* p, int64_t shift) {   // (a null pointer of a multi-frame launch must not be tested afterwards)
  return reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(p) + shift);
}

template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), unsigned grid, unsigned block, cudaStream_t stream, LaunchClass cls,
                     Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid, (unsigned)batch_ctx().frames, 1);
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributePriority;
  at[0].val.priority = launch_priority(cls);
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
// The same for a kernel that starts with pdl_enter(): launched with programmatic stream serialization (D3H_PDL=0 turns
// it off), the launch latency of the kernel overlaps the tail of its predecessor -- the forward chain of one frame is
// seven dependent kernels of a few microseconds each.
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline void launch_k_dep(void (*kernel)(KArgs...), unsigned grid, unsigned block, cudaStream_t stream, LaunchClass cls,
                         Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid, (unsigned)batch_ctx().frames, 1);
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributePriority;
  at[0].val.priority = launch_priority(cls);
  cfg.attrs = at;
  cfg.numAttrs = 1;
#ifndef D3H_CPU_EMU
  if (pdl_enabled()) {
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
  }
#endif
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
d3h_counts* mapped_counts_pointer(d3h_counts* host);
bool profiling_enabled();

// ---- optional per-kernel timing (d3h_profile_*): CUDA events recorded on the launching stream around each launch ----
enum KernelKind {
  K_PREPARE = 0, K_CLASSIFY, K_COMPACT, K_BUCKET_SCAN, K_PARTITION, K_GROUP_SORT, K_VERTEX_EMIT, K_POLY_FACES,
  K_POLY_CUT, K_ZERO, K_ADJOINT, K_RANK_RECORDS, K_EDGE_EMIT, K_ADJOINT_POLY, K_PAIR_REPLAY, K_MESH_EDGES, K_MESH_NORMALS,
  K_MESH_ADJOINT, K_EDGE_SCAN, K_EDGE_MARK, K_COUNT
};
struct ProfScope {
  ProfScope(int kind, cudaStream_t stream);
  ~ProfScope();
  int slot;
  cudaStream_t stream;
};

}  // namespace d3h
