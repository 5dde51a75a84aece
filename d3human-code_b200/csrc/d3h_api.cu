// C-ABI entry points of libd3h_tets.so (declared in include/d3h_tets.h) and the workspace carving.
#include <chrono>
#include <cstdlib>
#include <mutex>
#include <vector>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>

#include "d3h_internal.cuh"

namespace d3h {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

// ---- profiler -------------------------------------------------------------------------------------
static bool g_prof_on = false;
struct ProfRec { int kind; cudaEvent_t a, b; cudaStream_t stream; };
static ProfRec g_prof[4096];
static int g_prof_n = 0;

ProfScope::ProfScope(int kind, cudaStream_t st) : slot(-1), stream(st) {
  if (!g_prof_on || g_prof_n >= 4096) return;
  slot = g_prof_n++;
  ProfRec& r = g_prof[slot];
  r.kind = kind;
  r.stream = st;
  cudaEventCreate(&r.a);
  cudaEventCreate(&r.b);
  cudaEventRecord(r.a, stream);
}
ProfScope::~ProfScope() {
  if (slot >= 0) cudaEventRecord(g_prof[slot].b, stream);
}

bool profiling_enabled() { return g_prof_on; }

// ---- device trace table (diagnostics) ---------------------------------------------------------------
static unsigned long long* g_trace_dev = nullptr;
unsigned long long* trace_table() { return g_trace_dev; }

// ---- launch priorities ------------------------------------------------------------------------------
BatchCtx& batch_ctx() {
  static thread_local BatchCtx ctx = {1, {}, 1, {}, false};
  return ctx;
}

int launch_priority(LaunchClass c) {
  static int lo = 0, hi = 0;
  static bool init = false;
  if (!init) {
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) { lo = hi = 0; cudaGetLastError(); }
    init = true;
  }
  return c == kLaunchStream ? lo : hi;  // numerically lower = scheduled first
}

bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* env = getenv("D3H_PDL");
    v = (env && env[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

// ---- lanes: internal streams the frames of a batch are spread over -----------------------------------------------
constexpr int kMaxLanes = 8;
constexpr int kMaxDevices = 16;
constexpr int kClsEvents = 64;
struct LaneSet {
  bool ready;
  cudaStream_t lane[kMaxLanes];
  cudaStream_t head;                 // the heads (prepare + O(F) stream) of all frames, back to back
  cudaEvent_t fork, join[kMaxLanes], join_head;
  cudaEvent_t done[kMaxLanes];       // tail of the lane's last frame: its workspace may be reused
  bool done_valid[kMaxLanes];
  cudaEvent_t cls[kClsEvents];       // head of a frame finished (ring)
  unsigned cls_next;
  bool busy;                         // frames were put on the lanes since the last join (a fused batch joins them first)
};
static LaneSet g_lanes[kMaxDevices];
static std::mutex g_lane_mu;

static LaneSet* lanes_for_current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return nullptr;
  std::lock_guard<std::mutex> lock(g_lane_mu);
  LaneSet& ls = g_lanes[dev];
  if (!ls.ready) {
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    for (int i = 0; i < kMaxLanes; ++i) {
      if (cudaStreamCreateWithPriority(&ls.lane[i], cudaStreamNonBlocking, hi) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&ls.join[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&ls.done[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
      ls.done_valid[i] = false;
    }
    if (cudaStreamCreateWithPriority(&ls.head, cudaStreamNonBlocking, hi) != cudaSuccess) return nullptr;
    for (int i = 0; i < kClsEvents; ++i)
      if (cudaEventCreateWithFlags(&ls.cls[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    ls.cls_next = 0;
    if (cudaEventCreateWithFlags(&ls.fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&ls.join_head, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    ls.ready = true;
  }
  return &ls;
}

static inline int64_t align256(int64_t x) { return (x + 255) & ~int64_t(255); }

Workspace carve_workspace(void* base, int64_t n_tets, int64_t n_grid, int64_t cap_valid_tets, int64_t n_edges) {
  Workspace ws;
  memset(&ws, 0, sizeof(ws));
  char* p = reinterpret_cast<char*>(base);
  int64_t off = 0;
  auto take = [&](int64_t bytes) -> void* {
    void* r = p ? (p + off) : nullptr;
    off += align256(bytes > 0 ? bytes : 1);
    return r;
  };
  const int64_t cap = cap_valid_tets > 0 ? cap_valid_tets : 0;
  const int64_t capc = 4 * cap;
  ws.cap_tets = cap;
  ws.cap_corners = capc;
  const int64_t nchunks = (n_tets + kChunkTets - 1) / kChunkTets;
  const int64_t nwords_f = nchunks * kClassifyItems;
  ws.ntiles_compact = (n_tets + kTileTets - 1) / kTileTets;
  ws.nwords_tet = nwords_f + kCompactThreads;
  ws.ngroups = capc / kSortGroup + 1;
  ws.ntiles_poly = (cap + kPolyThreads - 1) / kPolyThreads;
  ws.msd_bins = ((n_grid - 1) >> msd_shift_for(n_grid)) + 1;
  ws.nscan_ctas = (ws.msd_bins + kScanThreads - 1) / kScanThreads;
  const int64_t nwords = (n_grid + 31) / 32 + 1;
  ws.ctr = reinterpret_cast<DevCounters*>(take(sizeof(DevCounters)));
  ws.blk = reinterpret_cast<FwdBlock*>(take(sizeof(FwdBlock)));
  ws.blk2 = reinterpret_cast<FwdBlock*>(take(sizeof(FwdBlock)));
  ws.counts = reinterpret_cast<d3h_counts*>(take(sizeof(d3h_counts)));
  ws.counts2 = reinterpret_cast<d3h_counts*>(take(sizeof(d3h_counts)));
  ws.occ_bits = reinterpret_cast<unsigned*>(take(nwords * 4));
  ws.mocc_bits = reinterpret_cast<unsigned*>(take(nwords * 4));
  ws.m1_words = reinterpret_cast<unsigned*>(take((nwords_f + kCompactThreads) * 4));
  ws.m2_words = reinterpret_cast<unsigned*>(take((nwords_f + kCompactThreads) * 4));
  ws.tile_cnt = reinterpret_cast<unsigned*>(take((ws.ntiles_compact + 1) * 4));
  ws.records = reinterpret_cast<d3h_tet_record*>(take(cap * (int64_t)sizeof(d3h_tet_record)));
  ws.keys = reinterpret_cast<unsigned long long*>(take(capc * 8));
  ws.vals = reinterpret_cast<unsigned*>(take(capc * 4));
  ws.keys2 = reinterpret_cast<unsigned long long*>(take(capc * 8));
  ws.vals2 = reinterpret_cast<unsigned*>(take(capc * 4));
  ws.keys_scratch = reinterpret_cast<unsigned long long*>(take(2 * capc * 8));
  ws.vals_scratch = reinterpret_cast<unsigned*>(take(2 * capc * 4));
  ws.msd_hist = reinterpret_cast<unsigned*>(take((ws.msd_bins + 12) * 4));
  ws.msd_fill = reinterpret_cast<unsigned*>(take((ws.msd_bins + 8) * 4));
  ws.msd_base = reinterpret_cast<unsigned*>(take((ws.msd_bins + 8) * 4));
  ws.st_scan = reinterpret_cast<unsigned long long*>(take(ws.nscan_ctas * 8));
  ws.group_start = reinterpret_cast<unsigned*>(take((ws.ngroups + 2) * 4));
  ws.group_heads = reinterpret_cast<unsigned*>(take((ws.ngroups + 1) * 4));
  ws.gblock_heads = reinterpret_cast<unsigned*>(take((ws.ngroups / 256 + 2) * 4));
  ws.poly_cnt = reinterpret_cast<unsigned*>(take((ws.ntiles_poly + 1) * 32));
  ws.poly_excl = reinterpret_cast<unsigned*>(take((ws.ntiles_poly + 1) * 32));
  // ... and per 32-polygon group (one warp of poly_faces_kernel): 8 words per group
  ws.poly_gcnt = reinterpret_cast<unsigned*>(take((ws.ntiles_poly + 1) * (kPolyThreads / 32) * 32));
  ws.poly_used = reinterpret_cast<unsigned char*>(take(cap));
  ws.vert = reinterpret_cast<float4*>(take(capc * 16));
  ws.acc = reinterpret_cast<float*>(take(capc * 32));
  ws.owner = reinterpret_cast<int32_t*>(take(capc * 4));
  ws.n_edges = n_edges > 0 ? n_edges : 0;
  ws.n_eblocks = (ws.n_edges + kEdgeBlock - 1) / kEdgeBlock;
  if (ws.n_edges > 0) {
    const int64_t ewords = ws.n_eblocks * (kEdgeBlock / 32);
    ws.edge_bits = reinterpret_cast<unsigned*>(take(ewords * 4));
    ws.word_prefix = reinterpret_cast<unsigned*>(take(ewords * 4));
    ws.eblock_cnt = reinterpret_cast<unsigned*>(take((ws.n_eblocks + 1) * 4));
    ws.corner_rank = reinterpret_cast<unsigned*>(take(capc * 4));
    // work queues of the edge-scan path: kQueues sub-queues, each 8 / kQueues of the total capacity (8x the expected fill)
    ws.cap_qv = cap > 0 ? (cap * 8 + kQueues - 1) / kQueues : 0;
    ws.cap_qe = capc > 0 ? (capc * 8 + kQueues - 1) / kQueues : 0;
    ws.q_cnt = reinterpret_cast<unsigned*>(take(4 * kQueues * kQStride * 4));
    ws.vlist = reinterpret_cast<int2*>(take(ws.cap_qv * kQueues * 8));
    ws.elist = reinterpret_cast<int32_t*>(take(ws.cap_qe * kQueues * 4));
    ws.elist2 = reinterpret_cast<int32_t*>(take(ws.cap_qe * kQueues * 4));
    ws.tet_word_prefix = reinterpret_cast<uint2*>(take((nwords_f + kCompactThreads) * 8));
  }
  ws.total_bytes = off;
  return ws;
}

// Device-visible alias of the caller's pinned counts buffer, or nullptr when the pointer is not mapped host memory
// (then the counts are copied with cudaMemcpyAsync at the end of the call instead).  One driver query per new pointer.
d3h_counts* mapped_counts_pointer(d3h_counts* host) {
  // cached per 4 KB page of host memory: a page belongs to one pinned allocation, whose device alias is at a constant
  // offset (the count slots of a plan are a 32 KB ring, 8 pages)
  constexpr int kSlots = 64;
  static thread_local uintptr_t page[kSlots] = {0};
  static thread_local intptr_t delta[kSlots] = {0};
  static thread_local bool mapped[kSlots] = {false};
  if (host == nullptr) return nullptr;
  const uintptr_t h = reinterpret_cast<uintptr_t>(host);
  const uintptr_t pg = h >> 12;
  const int slot = (int)(pg % kSlots);
  if (page[slot] != pg) {
    cudaPointerAttributes at;
    bool ok = cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer != nullptr;
    if (!ok) cudaGetLastError();  // plain pageable memory: clear the sticky error of the query
    page[slot] = pg;
    mapped[slot] = ok;
    delta[slot] = ok ? (intptr_t)(reinterpret_cast<uintptr_t>(at.devicePointer) - h) : 0;
  }
  return mapped[slot] ? reinterpret_cast<d3h_counts*>(h + delta[slot]) : nullptr;
}

static int check_forward_args(const d3h_forward_args* a, const char* who) {
  if (!a) { set_error("%s: null argument struct", who); return D3H_E_BADARG; }
  if (a->n_grid <= 0 || a->n_grid >= (1ll << 31) || a->n_tets < 0 || a->n_tets >= (1ll << 31)) {
    set_error("%s: n_grid=%lld / n_tets=%lld outside [1,2^31) / [0,2^31)", who, (long long)a->n_grid, (long long)a->n_tets);
    return D3H_E_BADARG;
  }
  if (!a->pos || !a->sdf || !a->msdf || (!a->tets && a->n_tets > 0) || !a->workspace) {
    set_error("%s: null input / workspace pointer", who);
    return D3H_E_BADARG;
  }
  if (reinterpret_cast<uintptr_t>(a->tets) & 15) { set_error("%s: tets must be 16-byte aligned", who); return D3H_E_BADARG; }
  if (reinterpret_cast<uintptr_t>(a->workspace) & 255) { set_error("%s: workspace must be 256-byte aligned", who); return D3H_E_BADARG; }
  if (a->tet_begin < 0 || a->tet_end < a->tet_begin || a->tet_end > a->n_tets) {
    set_error("%s: tet range [%lld,%lld) outside [0,%lld)", who, (long long)a->tet_begin, (long long)a->tet_end, (long long)a->n_tets);
    return D3H_E_BADARG;
  }
  if (a->cap_valid_tets < 0 || a->cap_valid_tets > (1ll << 27) || a->cap_verts < 0 || a->cap_verts_aug < 0 ||
      a->cap_faces_wt < 0 || a->cap_faces_aug < 0) {
    set_error("%s: capacities must be >= 0 and cap_valid_tets <= 2^27", who);
    return D3H_E_BADARG;
  }
  if (a->edge_off != nullptr &&
      (!a->edge_ab || a->n_edges <= 0 || a->n_edges >= (1ll << 31) || (a->cap_verts > 0 && !a->vacc) ||
       ((reinterpret_cast<uintptr_t>(a->edge_ab) | reinterpret_cast<uintptr_t>(a->vacc)) & 15))) {
    set_error("%s: static edge table needs edge_ab (8-byte pairs, 16-byte aligned), 0 < n_edges < 2^31 and vacc", who);
    return D3H_E_BADARG;
  }
  if (a->tet_edge_rank != nullptr && (a->edge_off == nullptr || (reinterpret_cast<uintptr_t>(a->tet_edge_rank) & 15))) {
    set_error("%s: tet_edge_rank needs the static edge table and 16-byte alignment", who);
    return D3H_E_BADARG;
  }
  if (a->etets != nullptr &&
      (!a->edge_off || (!a->edge_b && !a->edge_rows && !a->edge_runs) || !a->etet_off || !a->tet_edge_rank || a->tet_begin != 0 ||
       a->tet_end != a->n_tets)) {
    set_error("%s: the edge-scan path needs edge_off / edge_b or edge_rows or edge_runs / etet_off / etets / tet_edge_rank and the whole tet range", who);
    return D3H_E_BADARG;
  }
  if ((a->edge_rows != nullptr) != (a->edge_row_off != nullptr) || (a->edge_rows != nullptr && a->etets == nullptr) ||
      (reinterpret_cast<uintptr_t>(a->edge_rows) & 127)) {
    set_error("%s: edge_rows (128-byte aligned) and edge_row_off come together and with the edge-scan tables", who);
    return D3H_E_BADARG;
  }
  if (a->edge_runs != nullptr &&
      (!a->edge_run_chunk || !a->edge_run_ids || a->n_edge_runs <= 0 || a->n_edge_runs >= (1ll << 26) || a->etets == nullptr ||
       (reinterpret_cast<uintptr_t>(a->edge_runs) & 7))) {
    set_error("%s: edge_runs (8-byte aligned) needs edge_run_chunk, edge_run_ids, 0 < n_edge_runs < 2^26 and the edge-scan tables", who);
    return D3H_E_BADARG;
  }
  if (a->tet_runs != nullptr &&
      (!a->tet_run_chunk || !a->tet_run_ids || a->n_tet_runs <= 0 || a->n_tet_runs >= (1ll << 26) || a->edge_runs == nullptr ||
       (reinterpret_cast<uintptr_t>(a->tet_runs) & 15))) {
    set_error("%s: tet_runs (16-byte aligned) needs tet_run_chunk, tet_run_ids, 0 < n_tet_runs < 2^26 and edge_runs", who);
    return D3H_E_BADARG;
  }
  if ((a->etets8 != nullptr && a->etets == nullptr) || (reinterpret_cast<uintptr_t>(a->etets8) & 15) ||
      (a->etets != nullptr && (reinterpret_cast<uintptr_t>(a->edge_b) & 15))) {
    set_error("%s: etets8 needs the edge-scan tables; etets8 and edge_b must be 16-byte aligned", who);
    return D3H_E_BADARG;
  }
  if (a->cap_valid_tets > 0 && (!a->tape_corners || (a->edge_off == nullptr && (!a->tape_slots || !a->tape_runs)))) {
    set_error("%s: tape_corners / tape_slots (4*cap_valid_tets int32) and tape_runs (cap_verts+1 int32) are required", who);
    return D3H_E_BADARG;
  }
  if ((reinterpret_cast<uintptr_t>(a->sdf) | reinterpret_cast<uintptr_t>(a->msdf)) & 15) {
    set_error("%s: sdf / msdf must be 16-byte aligned", who);
    return D3H_E_BADARG;
  }
  if ((reinterpret_cast<uintptr_t>(a->pos) | reinterpret_cast<uintptr_t>(a->zero_g_pos) |
       reinterpret_cast<uintptr_t>(a->zero_g_sdf) | reinterpret_cast<uintptr_t>(a->zero_g_msdf)) & 3) {
    set_error("%s: pos / zero_g_* must be 4-byte aligned", who);
    return D3H_E_BADARG;
  }
  if ((a->cap_verts > 0 && (!a->verts_wt || !a->v_tng_wt || !a->msdf_wt || !a->tape_edges)) ||
      (a->cap_verts_aug > 0 && (!a->verts_aug || !a->v_tng_aug || !a->msdf_aug)) ||
      (a->cap_faces_wt > 0 && !a->faces_wt) || (a->cap_faces_aug > 0 && !a->faces_aug)) {
    set_error("%s: an output pointer is null while its capacity is > 0", who);
    return D3H_E_BADARG;
  }
  const int64_t need = carve_workspace(nullptr, a->n_tets, a->n_grid, a->cap_valid_tets, a->edge_off ? a->n_edges : 0).total_bytes;
  if (a->workspace_bytes < need) {
    set_error("%s: workspace has %lld bytes, %lld needed", who, (long long)a->workspace_bytes, (long long)need);
    return D3H_E_SMALLWS;
  }
  return D3H_OK;
}

static int finish(const char* who, const d3h_forward_args* a, const Workspace& ws, cudaStream_t stream) {
  if (a->counts_host && mapped_counts_pointer(a->counts_host) == nullptr)  // not device-mapped: copy at the end
    cudaMemcpyAsync(a->counts_host, ws.counts, sizeof(d3h_counts), cudaMemcpyDeviceToHost, stream);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("%s: %s", who, cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}

// `side` (graph capture only): a second stream of the same capture.  The zero-fill of the gradient buffers depends on
// nothing but the argument block, so in a captured graph it runs as a parallel branch right behind prepare_kernel: its
// 43 MB of stores hide under the latency-bound kernels of the surface stages instead of extending the chain by ~5 us.
void launch_forward_sequence(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream, int parts,
                             cudaStream_t side, cudaEvent_t fork, cudaEvent_t join) {
  const bool zero = (a.zero_g_pos || a.zero_g_sdf || a.zero_g_msdf) && (parts & kPartTail);
  const bool branch = zero && side != nullptr && (parts & kPartHead);
  if (branch) {
    cudaEventRecord(fork, stream);
    cudaStreamWaitEvent(side, fork, 0);
    launch_zero_grads_from_block(a, ws, side);
    cudaEventRecord(join, side);
  }
  if (edge_scan_path(a)) {
    // no classification stream: the walk over the static edge list marks crossing edges and valid tets
    if (parts & kPartHead) launch_edge_scan(a, ws, stream);
  } else {
    launch_classify(a, ws, ws.records, ws.cap_tets, /*emit_keys=*/true, stream, parts);
    if (parts & kPartTail) {
      if (a.edge_off != nullptr) launch_edge_emit(a, ws, stream);
      else launch_edge_sort(a, ws, stream);
    }
  }
  if (parts & kPartTail) {
    launch_surface(a, ws, ws.records, stream);
    if (zero && !branch) launch_zero_grads_from_block(a, ws, stream);
  }
  if (branch) cudaStreamWaitEvent(stream, join, 0);
}

// ---- graph cache -----------------------------------------------------------------------------------
// One instantiated CUDA graph per launch shape.  Only the parameters of the first node (prepare_kernel, which carries
// the argument block by value) change between launches.
const void* prepare_kernel_address();

struct GraphKey {
  void* workspace;
  int64_t n_tets, n_grid, tet_begin, tet_end, cap_valid_tets;
  int watertight, has_zero, device, is_static, parts;
  int64_t n_edges, n_edge_runs, n_tet_runs;   // (launch grids are captured: everything they are computed from is part of the key)
  bool operator==(const GraphKey& o) const {
    return parts == o.parts && is_static == o.is_static && n_edges == o.n_edges && n_edge_runs == o.n_edge_runs && n_tet_runs == o.n_tet_runs && workspace == o.workspace && n_tets == o.n_tets && n_grid == o.n_grid && tet_begin == o.tet_begin &&
           tet_end == o.tet_end && cap_valid_tets == o.cap_valid_tets && watertight == o.watertight &&
           has_zero == o.has_zero && device == o.device;
  }
};
struct GraphEntry {
  GraphKey key;
  cudaGraph_t graph;
  cudaGraphExec_t exec;
  cudaGraphNode_t prepare_node;
  cudaKernelNodeParams prepare_params;
  uint64_t last_use;
};
static std::mutex g_graph_mu;
static std::vector<GraphEntry> g_graphs;
static uint64_t g_graph_clock = 0;
static int g_graph_state = -1;  // -1 unknown, 0 disabled (D3H_DISABLE_GRAPH=1), 1 enabled
constexpr size_t kMaxGraphs = 128;

static void destroy_entry(GraphEntry& e) {
  cudaGraphExecDestroy(e.exec);
  cudaGraphDestroy(e.graph);
}

static int build_entry(const d3h_forward_args& a, const Workspace& ws, const GraphKey& key, GraphEntry& out) {
  const int parts = key.parts;
  static thread_local cudaStream_t cs = nullptr, cs2 = nullptr;
  static thread_local cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  if (cs == nullptr && cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking) != cudaSuccess) return -1;
  if (cs2 == nullptr && cudaStreamCreateWithFlags(&cs2, cudaStreamNonBlocking) != cudaSuccess) return -1;
  if (ev_fork == nullptr && cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming) != cudaSuccess) return -1;
  if (ev_join == nullptr && cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming) != cudaSuccess) return -1;
  static int zero_branch = -1;
  if (zero_branch < 0) {
    const char* env = getenv("D3H_ZERO_BRANCH");
    zero_branch = (env && env[0] == '0') ? 0 : 1;
  }
  cudaGraph_t graph = nullptr;
  if (cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return -1; }
  if (parts & kPartHead) launch_prepare(a, ws, cs);
  launch_forward_sequence(a, ws, cs, parts, zero_branch ? cs2 : nullptr, ev_fork, ev_join);
  if (cudaStreamEndCapture(cs, &graph) != cudaSuccess || graph == nullptr) { cudaGetLastError(); return -1; }
  size_t nn = 0;
  cudaGraphGetNodes(graph, nullptr, &nn);
  std::vector<cudaGraphNode_t> nodes(nn);
  cudaGraphGetNodes(graph, nodes.data(), &nn);
  bool found = !(parts & kPartHead);  // the tail has no per-call parameters: its kernels read the argument block
  for (size_t i = 0; i < nn && !found; ++i) {
    cudaGraphNodeType ty;
    if (cudaGraphNodeGetType(nodes[i], &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
    cudaKernelNodeParams kp;
    if (cudaGraphKernelNodeGetParams(nodes[i], &kp) != cudaSuccess) continue;
    if (kp.func == prepare_kernel_address()) {
      out.prepare_node = nodes[i];
      out.prepare_params = kp;
      found = true;
    }
  }
  cudaGraphExec_t exec = nullptr;
  // Instantiated WITHOUT cudaGraphInstantiateFlagUseNodePriority: every node runs at the priority of the lane stream.
  // Measured (profiles/graph_trace.py): with per-node priorities the latency-bound kernels of the other lanes take CTA
  // slots from the O(F) stream, which needs the whole register file to reach the HBM rate (64 regs x 4 CTAs / SM) and
  // slows down 2x -- the batch gets 8 % slower.  What the lanes buy is the overlap of one frame's dependency bubbles
  // with another frame's kernels, not free SM time.
  static int node_prio = -1;
  if (node_prio < 0) {
    const char* env = getenv("D3H_NODE_PRIORITY");
    node_prio = (env && env[0] == '1') ? 1 : 0;
  }
  if (!found || cudaGraphInstantiateWithFlags(&exec, graph, node_prio ? cudaGraphInstantiateFlagUseNodePriority : 0) !=
                    cudaSuccess) {
    cudaGetLastError();
    cudaGraphDestroy(graph);
    return -1;
  }
  out.key = key;
  out.graph = graph;
  out.exec = exec;
  return 0;
}

// Returns 0 when the call was enqueued as a graph launch, -1 when the caller must launch the kernels directly.
static int launch_forward_graph(const d3h_forward_args& a, const Workspace& ws, cudaStream_t stream,
                                int parts = kPartAll) {
  if (g_graph_state < 0) {
    const char* env = getenv("D3H_DISABLE_GRAPH");
    g_graph_state = (env && env[0] == '1') ? 0 : 1;
  }
  if (g_graph_state == 0 || profiling_enabled()) return -1;
  {
    // the caller is capturing this stream into its own graph: a graph launch cannot be captured, enqueue the kernels
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cap) != cudaSuccess) { cudaGetLastError(); return -1; }
    if (cap != cudaStreamCaptureStatusNone) return -1;
  }
  if (a.counts_host && mapped_counts_pointer(a.counts_host) == nullptr) return -1;  // needs the trailing memcpy
  GraphKey key;
  memset(&key, 0, sizeof(key));
  key.workspace = a.workspace;
  key.n_tets = a.n_tets; key.n_grid = a.n_grid; key.tet_begin = a.tet_begin; key.tet_end = a.tet_end;
  key.cap_valid_tets = a.cap_valid_tets;
  key.watertight = a.watertight_template ? 1 : 0;
  key.has_zero = (a.zero_g_pos || a.zero_g_sdf || a.zero_g_msdf) ? 1 : 0;
  key.parts = parts;
  key.is_static = a.edge_off != nullptr ? (a.etets != nullptr ? (a.etets8 != nullptr ? 4 : 3) : (a.tet_edge_rank != nullptr ? 2 : 1)) : 0;
  if (a.edge_rows != nullptr) key.is_static += 8;   // another stream kernel
  if (a.edge_runs != nullptr) key.is_static += 16;
  if (a.tet_runs != nullptr) key.is_static += 32;
  key.n_edge_runs = a.edge_runs != nullptr ? a.n_edge_runs : 0;
  key.n_tet_runs = a.tet_runs != nullptr ? a.n_tet_runs : 0;
  key.n_edges = a.edge_off != nullptr ? a.n_edges : 0;
  cudaGetDevice(&key.device);
  std::lock_guard<std::mutex> lock(g_graph_mu);
  GraphEntry* e = nullptr;
  for (auto& g : g_graphs)
    if (g.key == key) { e = &g; break; }
  if (e == nullptr) {
    GraphEntry ne;
    memset(&ne, 0, sizeof(ne));
    if (build_entry(a, ws, key, ne) != 0) { g_graph_state = 0; return -1; }  // capture unsupported here: stay direct
    if (g_graphs.size() >= kMaxGraphs) {
      size_t victim = 0;
      for (size_t i = 1; i < g_graphs.size(); ++i)
        if (g_graphs[i].last_use < g_graphs[victim].last_use) victim = i;
      destroy_entry(g_graphs[victim]);
      g_graphs[victim] = ne;
      e = &g_graphs[victim];
    } else {
      g_graphs.push_back(ne);
      e = &g_graphs.back();
    }
  }
  e->last_use = ++g_graph_clock;
  if (parts & kPartHead) {
    FwdBlock blk;
    blk.a = a;
    blk.counts_mapped = mapped_counts_pointer(a.counts_host);
    blk.trace = trace_table();
    Workspace wcopy = ws;
    void* kargs[2] = {&blk, &wcopy};
    cudaKernelNodeParams kp = e->prepare_params;
    kp.kernelParams = kargs;
    kp.extra = nullptr;
    if (cudaGraphExecKernelNodeSetParams(e->exec, e->prepare_node, &kp) != cudaSuccess) { cudaGetLastError(); return -1; }
  }
  if (cudaGraphLaunch(e->exec, stream) != cudaSuccess) { cudaGetLastError(); return -1; }
  return 0;
}

}  // namespace d3h

using namespace d3h;

// Evicts L2 by READING a buffer larger than the cache (a fill would leave it full of dirty lines whose write-back then
// competes with the kernel under test: measured 26.5 us after a 256 MB memset against 20.4 us under ncu's cache control).
__global__ void __launch_bounds__(256) flush_read_kernel(const uint4* __restrict__ p, int64_t n, unsigned* __restrict__ sink) {
  unsigned acc = 0u;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 v = __ldcg(p + i);
    acc ^= v.x ^ v.y ^ v.z ^ v.w;
  }
  if (acc == 0x9e3779b9u) *sink = acc;      // (practically never: keeps the loads alive)
}

extern "C" int d3h_profile_scan_kernel(const d3h_forward_args* a, int32_t reps, void* flush, int64_t flush_bytes,
                                       float* ms_total, d3h_stream_t s) {
  if (!a || !ms_total || reps <= 0 || reps > 1000 || flush_bytes < 0) { set_error("d3h_profile_scan_kernel: bad argument"); return D3H_E_BADARG; }
  int rc = check_forward_args(a, "d3h_profile_scan_kernel");
  if (rc) return rc;
  if (!edge_scan_path(*a)) { set_error("d3h_profile_scan_kernel: the arguments do not select the edge-scan path"); return D3H_E_BADARG; }
  cudaStream_t stream = (cudaStream_t)s;
  Workspace ws = carve_workspace(a->workspace, a->n_tets, a->n_grid, a->cap_valid_tets, a->n_edges);
  std::vector<cudaEvent_t> ev(2 * (size_t)reps);
  for (auto& e : ev)
    if (cudaEventCreate(&e) != cudaSuccess) { set_error("d3h_profile_scan_kernel: no events"); return D3H_E_CUDA; }
  launch_edge_scan_only(*a, ws, stream);          // warm-up
  for (int i = 0; i < reps; ++i) {
    // reading `flush` evicts L2 (the static edge list would otherwise stay resident between the launches) and keeps the
    // GPU busy up to the launch, so the event pair brackets the kernel and not an idle gap
    if (flush && flush_bytes >= 64)
      launch_k(flush_read_kernel, 148u * 8u, 256u, stream, kLaunchStream, reinterpret_cast<const uint4*>(flush), flush_bytes / 16,
               reinterpret_cast<unsigned*>(flush));
    cudaEventRecord(ev[2 * i], stream);
    launch_edge_scan_only(*a, ws, stream);
    cudaEventRecord(ev[2 * i + 1], stream);
  }
  cudaError_t e = cudaEventSynchronize(ev.back());
  float total = 0.f;
  for (int i = 0; i < reps && e == cudaSuccess; ++i) {
    float ms = 0.f;
    e = cudaEventElapsedTime(&ms, ev[2 * i], ev[2 * i + 1]);
    total += ms;
  }
  for (auto& x : ev) cudaEventDestroy(x);
  if (e != cudaSuccess) { set_error("d3h_profile_scan_kernel: %s", cudaGetErrorString(e)); return D3H_E_CUDA; }
  *ms_total = total;
  return D3H_OK;
}

extern "C" int d3h_version(void) { return D3H_VERSION; }
extern "C" const char* d3h_last_error_string(void) { return g_error; }

extern "C" int64_t d3h_workspace_bytes(int64_t n_tets, int64_t n_grid, int64_t cap_valid_tets) {
  if (n_tets < 0 || n_grid <= 0 || cap_valid_tets < 0) return D3H_E_BADARG;
  return carve_workspace(nullptr, n_tets, n_grid, cap_valid_tets).total_bytes;
}
extern "C" int64_t d3h_workspace_bytes_static(int64_t n_tets, int64_t n_grid, int64_t cap_valid_tets, int64_t n_edges) {
  if (n_tets < 0 || n_grid <= 0 || cap_valid_tets < 0 || n_edges < 0) return D3H_E_BADARG;
  return carve_workspace(nullptr, n_tets, n_grid, cap_valid_tets, n_edges).total_bytes;
}
extern "C" int64_t d3h_backward_workspace_bytes(int64_t n_verts) { (void)n_verts; return 0; }

extern "C" int d3h_wait_counts(const d3h_counts* counts_host, int64_t seq, int64_t timeout_us) {
  if (!counts_host) { set_error("d3h_wait_counts: null pointer"); return D3H_E_BADARG; }
  const volatile int64_t* flag = &counts_host->seq;
  const auto t0 = std::chrono::steady_clock::now();
  for (unsigned spins = 0;; ++spins) {
    if (*flag == seq) {
      __atomic_thread_fence(__ATOMIC_ACQUIRE);
      return D3H_OK;
    }
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
    if (timeout_us > 0 && (spins & 1023u) == 1023u) {
      const auto dt = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
      if (dt > timeout_us) { set_error("d3h_wait_counts: seq %lld not published after %lld us", (long long)seq, (long long)dt); return D3H_E_TIMEOUT; }
    }
  }
}

extern "C" int d3h_extract_forward(const d3h_forward_args* a, d3h_stream_t s) {
  int rc = check_forward_args(a, "d3h_extract_forward");
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)s;
  Workspace ws = carve_workspace(a->workspace, a->n_tets, a->n_grid, a->cap_valid_tets, a->edge_off ? a->n_edges : 0);
  const bool pair = a->pair_counts_host != nullptr;
  if (pair && ((a->cap_verts_aug > 0 && (!a->pair_verts_aug || !a->pair_v_tng_aug || !a->pair_msdf_aug)) ||
               (a->cap_verts > 0 && (!a->pair_verts_wt || !a->pair_v_tng_wt || !a->pair_msdf_wt)) ||
               (a->cap_faces_aug > 0 && !a->pair_faces_aug) || (a->cap_faces_wt > 0 && !a->pair_faces_wt) ||
               (a->edge_off != nullptr && a->cap_verts > 0 && !a->pair_vacc))) {
    set_error("d3h_extract_forward: pair_counts_host is set but a pair_* output is missing");
    return D3H_E_BADARG;
  }
  if (launch_forward_graph(*a, ws, stream) != 0) {
    launch_prepare(*a, ws, stream);
    launch_forward_sequence(*a, ws, stream);
  }
  if (pair) {
    launch_pair_replay(*a, ws, ws.records, stream);
    if (mapped_counts_pointer(a->pair_counts_host) == nullptr)   // not device-mapped: copy at the end
      cudaMemcpyAsync(a->pair_counts_host, ws.counts2, sizeof(d3h_counts), cudaMemcpyDeviceToHost, stream);
  }
  return finish("d3h_extract_forward", a, ws, stream);
}

// The frames of a batch in ONE launch per kernel (grid.y = frame; see FrameSet in d3h_internal.cuh): possible when every
// frame takes the run-length path on the watertight template with the same grid, tables and capacities (so the workspaces
// have one layout), publishes its counts through mapped memory and wants no second extraction.  Frames that share a
// workspace go into consecutive launches.
static bool fusable(const d3h_forward_args* args, int64_t n_frames) {
  static int enabled = -1;
  if (enabled < 0) {
    const char* env = getenv("D3H_FUSE_FRAMES");
    enabled = (env && env[0] == '0') ? 0 : 1;
  }
  if (!enabled || n_frames < 2) return false;
  const d3h_forward_args& r = args[0];
  for (int64_t i = 0; i < n_frames; ++i) {
    const d3h_forward_args& a = args[i];
    if (!a.edge_runs || !a.tet_runs || !a.watertight_template || a.pair_verts_aug || a.cap_valid_tets <= 0 ||
        !a.counts_host || mapped_counts_pointer(a.counts_host) == nullptr)
      return false;
    if (a.n_tets != r.n_tets || a.n_grid != r.n_grid || a.tets != r.tets || a.cap_valid_tets != r.cap_valid_tets ||
        a.n_edges != r.n_edges || a.edge_off != r.edge_off || a.edge_ab != r.edge_ab || a.tet_edge_rank != r.tet_edge_rank ||
        a.etet_off != r.etet_off || a.etets != r.etets || a.edge_runs != r.edge_runs || a.edge_run_chunk != r.edge_run_chunk ||
        a.edge_run_ids != r.edge_run_ids || a.n_edge_runs != r.n_edge_runs || a.tet_runs != r.tet_runs ||
        a.tet_run_chunk != r.tet_run_chunk || a.tet_run_ids != r.tet_run_ids || a.n_tet_runs != r.n_tet_runs ||
        a.tet_begin != r.tet_begin || a.tet_end != r.tet_end || a.workspace_bytes != r.workspace_bytes)
      return false;
  }
  return true;
}

static bool shared_topology_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* env = getenv("D3H_SHARE_TOPOLOGY");
    on = (env && env[0] == '0') ? 0 : 1;
  }
  return on != 0;
}

static int forward_batch_fused(const d3h_forward_args* args, int64_t n_frames, cudaStream_t stream, LaneSet* ls) {
  BatchCtx& ctx = batch_ctx();
  int rc = D3H_OK;
  if (ls->busy) {   // frames of an earlier per-lane batch may still be at work in these workspaces
    for (int l = 0; l < kMaxLanes; ++l) {
      cudaEventRecord(ls->join[l], ls->lane[l]);
      cudaStreamWaitEvent(stream, ls->join[l], 0);
    }
    cudaEventRecord(ls->join_head, ls->head);
    cudaStreamWaitEvent(stream, ls->join_head, 0);
    ls->busy = false;
  }
  int64_t i0 = 0;
  const d3h_forward_args* topo_of = nullptr;   // first frame of the launch whose topology is still standing in its workspace
  while (i0 < n_frames) {
    // the longest run of frames with distinct workspaces, at most kMaxFused
    int64_t i1 = i0 + 1;
    while (i1 < n_frames && i1 - i0 < kMaxFused) {
      bool clash = false;
      for (int64_t j = i0; j < i1; ++j) clash = clash || args[j].workspace == args[i1].workspace;
      if (clash) break;
      ++i1;
    }
    const d3h_forward_args& a = args[i0];
    const Workspace ws = carve_workspace(a.workspace, a.n_tets, a.n_grid, a.cap_valid_tets, a.n_edges);
    ctx.frames = (int)(i1 - i0);
    bool shared = shared_topology_enabled();
    for (int64_t j = i0; j < i1; ++j) {
      ctx.fs.off[j - i0] = (int64_t)(reinterpret_cast<intptr_t>(args[j].workspace) - reinterpret_cast<intptr_t>(a.workspace));
      shared = shared && args[j].sdf == a.sdf && args[j].msdf == a.msdf && args[j].msdf_negate == a.msdf_negate;
    }
    ctx.topo_frames = shared ? 1 : ctx.frames;
    for (int f = 0; f < ctx.frames; ++f) ctx.topo.off[f] = shared ? 0 : ctx.fs.off[f];
    // rounds of one call (frames beyond the number of workspaces): the same field again, found by the round before in the
    // very workspace this round's first frame uses -- keep it
    ctx.reuse_topology = shared && ctx.frames > 1 && topo_of != nullptr && topo_of->workspace == a.workspace &&
                         topo_of->sdf == a.sdf && topo_of->msdf == a.msdf && topo_of->msdf_negate == a.msdf_negate;
    topo_of = (shared && ctx.frames > 1) ? &a : nullptr;
    launch_prepare_frames(args + i0, ws, stream);
    // the zero-fill of the gradient buffers depends on nothing but the argument blocks: a side stream takes it
    bool zero = false;
    for (int64_t j = i0; j < i1; ++j) zero = zero || args[j].zero_g_pos || args[j].zero_g_sdf || args[j].zero_g_msdf;
    if (zero) {
      cudaEventRecord(ls->fork, stream);
      cudaStreamWaitEvent(ls->lane[0], ls->fork, 0);
      launch_zero_grads_from_block(a, ws, ls->lane[0]);
      cudaEventRecord(ls->join[0], ls->lane[0]);
    }
    launch_edge_scan(a, ws, stream);
    launch_surface(a, ws, ws.records, stream);
    if (zero) cudaStreamWaitEvent(stream, ls->join[0], 0);
    ctx.frames = ctx.topo_frames = 1;
    ctx.reuse_topology = false;
    memset(&ctx.fs, 0, sizeof(ctx.fs));
    memset(&ctx.topo, 0, sizeof(ctx.topo));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("d3h_extract_forward_batch: %s", cudaGetErrorString(e)); rc = D3H_E_CUDA; }
    i0 = i1;
  }
  return rc;
}

static int forward_batch(const d3h_forward_args* args, int64_t n_frames, int32_t lanes, d3h_stream_t s, bool join) {
  if (!args || n_frames < 0 || lanes < 1) { set_error("d3h_extract_forward_batch: null args / bad sizes"); return D3H_E_BADARG; }
  if (lanes > kMaxLanes) lanes = kMaxLanes;
  if (lanes > n_frames) lanes = (int32_t)(n_frames > 0 ? n_frames : 1);
  for (int64_t i = 0; i < n_frames; ++i) {
    int rc = check_forward_args(&args[i], "d3h_extract_forward_batch");
    if (rc) return rc;
    for (int64_t j = 0; j < i; ++j)
      if (args[j].workspace == args[i].workspace && (j % lanes) != (i % lanes)) {
        set_error("d3h_extract_forward_batch: frames %lld and %lld share a workspace but run on different lanes",
                  (long long)j, (long long)i);
        return D3H_E_BADARG;
      }
  }
  if (n_frames == 0) return D3H_OK;
  if (n_frames == 1) return d3h_extract_forward(args, s);  // nothing to overlap: stay on the caller's stream
  cudaStream_t stream = (cudaStream_t)s;
  LaneSet* ls = lanes_for_current_device();
  if (ls == nullptr) { set_error("d3h_extract_forward_batch: cannot create the lane streams"); return D3H_E_CUDA; }
  {
    // a capturing caller gets the plain sequence on its own stream (events recorded outside the capture cannot be waited)
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cap) != cudaSuccess) cudaGetLastError();
    if (cap != cudaStreamCaptureStatusNone) {
      int rc = D3H_OK;
      for (int64_t i = 0; i < n_frames; ++i) {
        const int r = d3h_extract_forward(&args[i], s);
        if (r) rc = r;
      }
      return rc;
    }
  }
  if (fusable(args, n_frames)) return forward_batch_fused(args, n_frames, stream, ls);
  // Otherwise: one graph per frame, frame i on lane i % lanes.  The hardware takes equal-priority kernels in submission
  // order, so the O(F) streams of the frames run one after the other at full rate and the latency-bound kernels of the
  // other lanes fill in around them.
  // D3H_SPLIT_HEAD=1 (experiment, profiles/README.md): the heads of all frames (prepare + stream) back to back on ONE
  // stream, the tail of frame i on lane i % lanes once its head is done.  Measured slower: a stream that shares the SMs
  // with tails needs 55-60 us instead of 35, and graph launches on one stream leave ~10 us between graphs.
  static int split_head = -1;
  if (split_head < 0) {
    const char* env = getenv("D3H_SPLIT_HEAD");
    split_head = (env && env[0] == '1') ? 1 : 0;
  }
  ls->busy = true;
  cudaEventRecord(ls->fork, stream);
  if (split_head) cudaStreamWaitEvent(ls->head, ls->fork, 0);
  for (int l = 0; l < lanes; ++l) cudaStreamWaitEvent(ls->lane[l], ls->fork, 0);
  int rc = D3H_OK;
  for (int64_t i = 0; i < n_frames; ++i) {
    const d3h_forward_args* a = &args[i];
    const int l = (int)(i % lanes);
    cudaStream_t lane = ls->lane[l];
    Workspace ws = carve_workspace(a->workspace, a->n_tets, a->n_grid, a->cap_valid_tets, a->edge_off ? a->n_edges : 0);
    if (!split_head) {
      if (launch_forward_graph(*a, ws, lane) != 0) {
        launch_prepare(*a, ws, lane);
        launch_forward_sequence(*a, ws, lane);
      }
    } else {
      // the head overwrites the workspace of the frame that ran on this lane before
      if (ls->done_valid[l]) cudaStreamWaitEvent(ls->head, ls->done[l], 0);
      launch_prepare(*a, ws, ls->head);
      launch_forward_sequence(*a, ws, ls->head, kPartHead);
      cudaEvent_t cls = ls->cls[ls->cls_next++ % kClsEvents];
      cudaEventRecord(cls, ls->head);
      cudaStreamWaitEvent(lane, cls, 0);
      if (launch_forward_graph(*a, ws, lane, kPartTail) != 0) launch_forward_sequence(*a, ws, lane, kPartTail);
      cudaEventRecord(ls->done[l], lane);
      ls->done_valid[l] = true;
    }
    const int r = finish("d3h_extract_forward_batch", a, ws, lane);
    if (r) rc = r;
  }
  if (join || rc != D3H_OK) {  // after an error always join: the caller's stream must not lose the lanes
    for (int l = 0; l < kMaxLanes; ++l) {
      cudaEventRecord(ls->join[l], ls->lane[l]);
      cudaStreamWaitEvent(stream, ls->join[l], 0);
    }
    cudaEventRecord(ls->join_head, ls->head);
    cudaStreamWaitEvent(stream, ls->join_head, 0);
  }
  return rc;
}

// A batch of independent extractions (video frames, or the cloth / body pair of one iteration): frame i runs on
// internal lane i % lanes, the lanes fork from `stream` and join back into it, so for the caller the batch is ordered
// like one call.  Frames that share a lane may share a workspace (they are serialised); frames on different lanes
// must not.  Every frame publishes its own d3h_counts (args[i].counts_host / seq).
extern "C" int d3h_extract_forward_batch(const d3h_forward_args* args, int64_t n_frames, int32_t lanes,
                                         d3h_stream_t s) {
  return forward_batch(args, n_frames, lanes, s, /*join=*/true);
}

// Same without the join: the lanes keep running, `stream` is NOT ordered behind them until d3h_lanes_join(stream) is
// called.  Several batches launched back to back this way queue up per lane, so the O(F) stream of the next batch
// starts on a lane the moment that lane's frame of the previous batch is done -- no drain / refill of the pipeline at
// the batch boundary.  The caller must join before `stream` touches any output (or frees any buffer) of the batches.
extern "C" int d3h_extract_forward_batch_nojoin(const d3h_forward_args* args, int64_t n_frames, int32_t lanes,
                                                d3h_stream_t s) {
  return forward_batch(args, n_frames, lanes, s, /*join=*/false);
}

// Orders `stream` behind everything enqueued on the lanes so far.
extern "C" int d3h_lanes_join(d3h_stream_t s) {
  LaneSet* ls = lanes_for_current_device();
  if (ls == nullptr) { set_error("d3h_lanes_join: cannot create the lane streams"); return D3H_E_CUDA; }
  for (int l = 0; l < kMaxLanes; ++l) {
    cudaEventRecord(ls->join[l], ls->lane[l]);
    cudaStreamWaitEvent((cudaStream_t)s, ls->join[l], 0);
  }
  cudaEventRecord(ls->join_head, ls->head);
  cudaStreamWaitEvent((cudaStream_t)s, ls->join_head, 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("d3h_lanes_join: %s", cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}

static int check_backward_args(const d3h_backward_args* a, const char* who) {
  if (!a) { set_error("%s: null argument struct", who); return D3H_E_BADARG; }
  if (a->n_grid <= 0 || a->n_verts < 0 || a->n_tri_tets < 0 || a->n_quad_tets < 0 || !a->g_pos || !a->g_sdf ||
      !a->pos || !a->sdf || !a->msdf) {
    set_error("%s: null pointer or negative size", who);
    return D3H_E_BADARG;
  }
  if (a->n_verts > 0 && (!a->tape_edges || !a->tape_corners || !a->verts_wt || !a->msdf_wt ||
                         ((!a->tape_slots || !a->tape_runs) && !a->vacc))) {
    set_error("%s: tape / saved outputs missing", who);
    return D3H_E_BADARG;
  }
  if ((reinterpret_cast<uintptr_t>(a->g_pos) | reinterpret_cast<uintptr_t>(a->g_sdf) |
       reinterpret_cast<uintptr_t>(a->g_msdf)) & 3) {
    set_error("%s: gradient buffers must be 4-byte aligned", who);
    return D3H_E_BADARG;
  }
  return D3H_OK;
}

// Adjoints of a batch.  Gradient buffers may be shared between frames (sdf / msdf of a batch of video frames are the
// same tensors): every frame accumulates with atomics, so a shared buffer ends up with the sum over the frames.  With
// grads_prezeroed = 0 the call zeroes such a buffer once, before any frame accumulates into it; with grads_prezeroed = 1
// on every frame that uses it, it must be zero on entry.
extern "C" int d3h_extract_backward_batch(const d3h_backward_args* args, int64_t n_frames, int32_t lanes,
                                          d3h_stream_t s) {
  if (!args || n_frames < 0 || lanes < 1) { set_error("d3h_extract_backward_batch: null args / bad sizes"); return D3H_E_BADARG; }
  for (int64_t i = 0; i < n_frames; ++i) {
    int rc = check_backward_args(&args[i], "d3h_extract_backward_batch");
    if (rc) return rc;
  }
  (void)lanes;
  if (n_frames == 0) return D3H_OK;
  launch_backward_batch(args, n_frames, (cudaStream_t)s);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("d3h_extract_backward_batch: %s", cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}

// stage 1 only: prepare + classify of [tet_begin, tet_end); the compact records land in `records_out`
// (class ranks are local to the range) and the counts so far (n_valid/n_tri/n_quad) in `counts_dev_out`.
__global__ void export_range_counts_kernel(const DevCounters* ctr, d3h_counts* out, int64_t seq) {
  memset(out, 0, sizeof(d3h_counts));
  out->n_valid_tets = ctr->n_valid;
  out->n_tri_tets = ctr->n_tri;
  out->n_quad_tets = ctr->n_quad;
  out->n_corners = 3ll * ctr->n_tri + 4ll * ctr->n_quad;
  out->overflow = (ctr->n_valid != ctr->work_tri + ctr->work_quad) ? 1 : 0;
  out->seq = seq;
}

extern "C" int d3h_classify_range(const d3h_forward_args* a_in, d3h_tet_record* records_out, int64_t cap_records,
                                  d3h_counts* counts_dev_out, d3h_stream_t s) {
  if (!a_in) { set_error("d3h_classify_range: null argument struct"); return D3H_E_BADARG; }
  d3h_forward_args general = *a_in;  // the sharded stages always take the general (sort) path
  general.edge_off = nullptr; general.edge_ab = nullptr; general.n_edges = 0;
  general.tet_edge_rank = nullptr; general.edge_b = nullptr; general.etet_off = nullptr; general.etets = nullptr;
  general.etets8 = nullptr; general.edge_rows = nullptr; general.edge_row_off = nullptr;
  general.edge_runs = nullptr; general.edge_run_chunk = nullptr; general.edge_run_ids = nullptr; general.n_edge_runs = 0;
  general.tet_runs = nullptr; general.tet_run_chunk = nullptr; general.tet_run_ids = nullptr; general.n_tet_runs = 0;
  const d3h_forward_args* a = &general;
  int rc = check_forward_args(a, "d3h_classify_range");
  if (rc) return rc;
  if ((!records_out && cap_records > 0) || cap_records < 0 || !counts_dev_out) {
    set_error("d3h_classify_range: null records / counts pointer");
    return D3H_E_BADARG;
  }
  cudaStream_t stream = (cudaStream_t)s;
  Workspace ws = carve_workspace(a->workspace, a->n_tets, a->n_grid, a->cap_valid_tets, a->edge_off ? a->n_edges : 0);
  launch_prepare(*a, ws, stream);
  launch_classify(*a, ws, records_out, cap_records, /*emit_keys=*/false, stream);
#ifndef D3H_CPU_EMU
  export_range_counts_kernel<<<1, 1, 0, stream>>>(ws.ctr, counts_dev_out, a->seq);
#else   // tests/emu: g++ has no <<< >>>
  launch_k(export_range_counts_kernel, 1u, 1u, stream, kLaunchLatency, ws.ctr, counts_dev_out, a->seq);
#endif
  if (a->counts_host) cudaMemcpyAsync(a->counts_host, counts_dev_out, sizeof(d3h_counts), cudaMemcpyDeviceToHost, stream);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("d3h_classify_range: %s", cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}

// stage 2 only: `records` is the rank-order concatenation of the shards' records (= global tet order);
// n_tri_tets + n_quad_tets records.  Class ranks are recomputed over the concatenation.
extern "C" int d3h_extract_from_records(const d3h_forward_args* a_in, const d3h_tet_record* records, int64_t n_tri_tets,
                                        int64_t n_quad_tets, d3h_stream_t s) {
  if (!a_in) { set_error("d3h_extract_from_records: null argument struct"); return D3H_E_BADARG; }
  d3h_forward_args general = *a_in;
  general.edge_off = nullptr; general.edge_ab = nullptr; general.n_edges = 0;
  general.tet_edge_rank = nullptr; general.edge_b = nullptr; general.etet_off = nullptr; general.etets = nullptr;
  general.etets8 = nullptr; general.edge_rows = nullptr; general.edge_row_off = nullptr;
  general.edge_runs = nullptr; general.edge_run_chunk = nullptr; general.edge_run_ids = nullptr; general.n_edge_runs = 0;
  general.tet_runs = nullptr; general.tet_run_chunk = nullptr; general.tet_run_ids = nullptr; general.n_tet_runs = 0;
  const d3h_forward_args* a = &general;
  int rc = check_forward_args(a, "d3h_extract_from_records");
  if (rc) return rc;
  const int64_t n = n_tri_tets + n_quad_tets;
  if (n < 0 || n_tri_tets < 0 || n_quad_tets < 0 || n > a->cap_valid_tets || (!records && n > 0)) {
    set_error("d3h_extract_from_records: %lld records do not fit cap_valid_tets=%lld", (long long)n, (long long)a->cap_valid_tets);
    return D3H_E_BADARG;
  }
  cudaStream_t stream = (cudaStream_t)s;
  Workspace ws = carve_workspace(a->workspace, a->n_tets, a->n_grid, a->cap_valid_tets, a->edge_off ? a->n_edges : 0);
  d3h_forward_args b = *a;
  b.tet_begin = b.tet_end = 0;  // prepare still resets the scan state; no tets are classified here
  launch_prepare(b, ws, stream);
  if (n > 0) cudaMemcpyAsync(ws.records, records, n * sizeof(d3h_tet_record), cudaMemcpyDeviceToDevice, stream);
  launch_rank_records(*a, ws, ws.records, n, stream);
  launch_edge_sort(*a, ws, stream);
  launch_surface(*a, ws, ws.records, stream);
  if (a->zero_g_pos || a->zero_g_sdf || a->zero_g_msdf) launch_zero_grads_from_block(*a, ws, stream);
  return finish("d3h_extract_from_records", a, ws, stream);
}

extern "C" int d3h_extract_backward(const d3h_backward_args* a, d3h_stream_t s) {
  int rc = check_backward_args(a, "d3h_extract_backward");
  if (rc) return rc;
  launch_backward(*a, (cudaStream_t)s);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("d3h_extract_backward: %s", cudaGetErrorString(e)); return D3H_E_CUDA; }
  return D3H_OK;
}

// ---- diagnostics: per-kernel device time, measured with CUDA events on the launching stream -----------------------
static const char* kKernelNames[K_COUNT] = {"prepare", "classify", "compact", "bucket_scan", "partition", "group_sort",
                                            "vertex_emit", "poly_faces", "poly_cut", "zero", "adjoint", "rank_records",
                                            "edge_emit", "adjoint_poly", "pair_replay", "mesh_edges", "mesh_normals",
                                            "mesh_adjoint", "edge_scan", "edge_mark"};
extern "C" int d3h_profile_enable(int on) {
  g_prof_on = on != 0;
  return D3H_OK;
}
extern "C" int d3h_profile_kinds(void) { return K_COUNT; }
extern "C" const char* d3h_profile_kernel_name(int k) { return (k >= 0 && k < K_COUNT) ? kKernelNames[k] : ""; }
// Synchronises the recorded events, adds their durations (ms) and launch counts per kernel kind, then clears the log.
extern "C" int d3h_profile_read(float* ms_by_kind, int* launches_by_kind) {
  if (!ms_by_kind || !launches_by_kind) { set_error("d3h_profile_read: null output"); return D3H_E_BADARG; }
  for (int k = 0; k < K_COUNT; ++k) { ms_by_kind[k] = 0.f; launches_by_kind[k] = 0; }
  int rc = D3H_OK;
  for (int i = 0; i < g_prof_n; ++i) {
    ProfRec& r = g_prof[i];
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(r.b);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, r.a, r.b);
    if (e != cudaSuccess) { set_error("d3h_profile_read: %s", cudaGetErrorString(e)); rc = D3H_E_CUDA; }
    ms_by_kind[r.kind] += ms;
    launches_by_kind[r.kind] += 1;
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  g_prof_n = 0;
  return rc;
}

// Timeline variant of d3h_profile_read: start / end of every recorded launch in milliseconds since the first one, its
// kernel kind and a small integer naming the stream it ran on (lanes of a batch run concurrently).  Clears the log.
extern "C" int d3h_profile_timeline(float* start_ms, float* end_ms, int* kind, int* stream_id, int cap) {
  if (!start_ms || !end_ms || !kind || !stream_id) { set_error("d3h_profile_timeline: null output"); return D3H_E_BADARG; }
  int n = g_prof_n < cap ? g_prof_n : cap;
  cudaStream_t seen[64];
  int nseen = 0;
  for (int i = 0; i < g_prof_n; ++i) {
    ProfRec& r = g_prof[i];
    cudaEventSynchronize(r.b);
    if (i < n) {
      float a = 0.f, b = 0.f;
      cudaEventElapsedTime(&a, g_prof[0].a, r.a);
      cudaEventElapsedTime(&b, g_prof[0].a, r.b);
      start_ms[i] = a; end_ms[i] = b; kind[i] = r.kind;
      int sid = -1;
      for (int k = 0; k < nseen; ++k) if (seen[k] == r.stream) sid = k;
      if (sid < 0 && nseen < 64) { seen[nseen] = r.stream; sid = nseen++; }
      stream_id[i] = sid;
    }
  }
  for (int i = 0; i < g_prof_n; ++i) { cudaEventDestroy(g_prof[i].a); cudaEventDestroy(g_prof[i].b); }
  g_prof_n = 0;
  cudaGetLastError();
  return n;
}

// Device-side trace (works inside the cached graphs, unlike the event profiler): every forward kernel stamps
// %globaltimer when its block 0 starts and when its last block exits, into row (seq % 64) of a device table.  Enabling
// allocates that 16 KB table with cudaMalloc -- the one allocation this library ever makes, diagnostics only.
extern "C" int d3h_trace_enable(int on) {
  const size_t bytes = (size_t)kTraceFrames * kTraceKinds * 2 * sizeof(unsigned long long);
  if (on) {
    if (g_trace_dev == nullptr && cudaMalloc(&g_trace_dev, bytes) != cudaSuccess) {
      g_trace_dev = nullptr;
      set_error("d3h_trace_enable: cudaMalloc failed");
      cudaGetLastError();
      return D3H_E_CUDA;
    }
    cudaMemset(g_trace_dev, 0, bytes);
  } else if (g_trace_dev != nullptr) {
    cudaDeviceSynchronize();
    cudaFree(g_trace_dev);
    g_trace_dev = nullptr;
  }
  return D3H_OK;
}
// Copies the table out ((64, 24, 2) uint64 nanoseconds: [seq % 64][kernel kind][start, end]; 0 = not run) and clears
// it.  Synchronises the device.
extern "C" int d3h_trace_read(uint64_t* out) {
  if (!out) { set_error("d3h_trace_read: null output"); return D3H_E_BADARG; }
  const size_t bytes = (size_t)kTraceFrames * kTraceKinds * 2 * sizeof(unsigned long long);
  if (g_trace_dev == nullptr) { memset(out, 0, bytes); return D3H_OK; }
  cudaDeviceSynchronize();
  if (cudaMemcpy(out, g_trace_dev, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) {
    set_error("d3h_trace_read: %s", cudaGetErrorString(cudaGetLastError()));
    return D3H_E_CUDA;
  }
  cudaMemset(g_trace_dev, 0, bytes);
  return D3H_OK;
}

// ---- test hook: the case tables, from the same initializer macros the __constant__ copies are built from --------
// which: 0 num_tri[16], 1 loop_edge[16][4], 2 tri_edge[16][6], 3 cut_tri[8][6], 4 num_cut_tri[8],
//        5 cut_quad[16][12], 6 num_cut_quad[16], 7 edge_p[6], 8 edge_q[6].  Returns the element count.  Host only.
extern "C" int d3h_debug_table(int which, int8_t* out, int cap) {
  static const int8_t t0[16] = D3H_T_NUM_TRI;
  static const int8_t t1[16][4] = D3H_T_LOOP_EDGE;
  static const int8_t t2[16][6] = D3H_T_TRI_EDGE;
  static const int8_t t3[8][6] = D3H_T_CUT_TRI;
  static const int8_t t4[8] = D3H_T_NUM_CUT_TRI;
  static const int8_t t5[16][12] = D3H_T_CUT_QUAD;
  static const int8_t t6[16] = D3H_T_NUM_CUT_QUAD;
  static const int8_t t7[6] = D3H_T_EDGE_P;
  static const int8_t t8[6] = D3H_T_EDGE_Q;
  const void* src[9] = {t0, t1, t2, t3, t4, t5, t6, t7, t8};
  const int len[9] = {16, 64, 96, 48, 8, 192, 16, 6, 6};
  if (which < 0 || which > 8) { set_error("d3h_debug_table: unknown table %d", which); return D3H_E_BADARG; }
  if (cap < len[which] || !out) { set_error("d3h_debug_table: buffer too small"); return D3H_E_BADARG; }
  memcpy(out, src[which], len[which]);
  return len[which];
}
