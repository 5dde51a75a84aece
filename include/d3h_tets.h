/*
 * d3h_tets.h -- C ABI of the B200-native G-Shell / mSDF marching-tetrahedra extraction.
 *
 * This is the drop-in boundary for ONE path of D3-Human:
 *     GShell_Tets.__call__   geometry/gshell_tets.py:253-447
 *     hmSDF_Tets.__call__    geometry/hmsdf_tets_split.py:254-454
 * The reference has no native implementation of this path (it is ~200 PyTorch ops); its other
 * plugins bind `at::Tensor` through pybind11 (render/renderutils/c_src/torch_bindings.cpp:14-31,
 * loaded by render/renderutils/ops.py:23-87).  Here the binding is a plain C ABI instead: raw device
 * pointers, sizes and a cudaStream_t, loaded with ctypes.CDLL by the Python host
 * (d3human-code_b200/_cabi.py).  INTEGRATION.md shows the stub a maintainer adds to the reference.
 *
 * Conventions
 *   - every function returns 0 on success, a negative D3H_E_* code otherwise; the message is available
 *     from d3h_last_error_string() (thread-local).  CUDA errors are reported as D3H_E_CUDA.
 *   - the library never allocates device memory: inputs, outputs, tape and scratch are caller-owned
 *     (torch tensors in the Python host).  Outputs are over-allocated to caller-chosen capacities;
 *     the true sizes come back in d3h_counts.  A capacity that is too small is NOT an error: the
 *     kernels drop the out-of-range writes and the caller re-runs with the sizes just reported.
 *   - no host synchronisation inside any call; everything is enqueued on `stream` and is CUDA-graph
 *     capturable.  d3h_counts is written to `counts_host` (pinned, device-mapped host memory) by the
 *     kernel that finalises it, ahead of the output-writing kernels; the caller polls counts_host->seq
 *     (d3h_wait_counts) or synchronises the stream before reading it.  If the pointer is not device
 *     accessible the library falls back to a cudaMemcpyAsync at the end of the call.
 *   - all float data is fp32; index outputs are int64 (the reference returns torch.long faces,
 *     gshell_tets.py:413-420); tet indices are consumed as packed int32x4 (16-byte loads).
 */
#ifndef D3H_TETS_H_
#define D3H_TETS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D3H_VERSION 501 /* 0.5.1: d3h_sdf_reg_* */

enum {
  D3H_OK = 0,
  D3H_E_BADARG = -1,  /* null pointer, negative size, N or F >= 2^31, misaligned tet pointer */
  D3H_E_CUDA = -2,    /* a CUDA runtime call failed; see d3h_last_error_string() */
  D3H_E_SMALLWS = -3, /* workspace_bytes smaller than d3h_workspace_bytes(...) */
  D3H_E_TIMEOUT = -4  /* d3h_wait_counts gave up */
};

/* Opaque to C callers that only pass it around; the layout is fixed so ctypes can mirror it. */
typedef void* d3h_stream_t; /* cudaStream_t */

/* Sizes produced by one forward call (device copy lives in the workspace, host copy in pinned memory).
 * Names follow SURVEY.md section 8(a): Fv valid tets, T1/T2 tets producing 1/2 watertight triangles,
 * P = 3*T1 + 4*T2 polygon corners (= boundary vertices), V crossing edges (= watertight vertices),
 * Va = V + P augmented vertices, Fw = T1 + 2*T2 watertight faces, Fa open-mesh faces in 6 buckets
 * (tri polygons cut into 1,2 triangles; quad polygons cut into 1,2,3,4 triangles; gshell_tets.py:413-420). */
typedef struct d3h_counts {
  int64_t n_valid_tets;   /* Fv */
  int64_t n_tri_tets;     /* T1 */
  int64_t n_quad_tets;    /* T2 */
  int64_t n_corners;      /* P  */
  int64_t n_verts;        /* V  */
  int64_t n_faces_aug;    /* Fa */
  int64_t bucket_polys[6];/* polygons per faces_aug bucket, in bucket order */
  int64_t bad_index;      /* number of tet indices outside [0,N) seen by d3h_pack_tets_* (0 = clean) */
  int64_t overflow;       /* 1: Fv exceeded cap_valid_tets, the surface stages were skipped (re-run with more room) */
  int64_t seq;            /* d3h_forward_args.seq of the call that produced these counts; written LAST */
  int64_t reserved;
} d3h_counts;

/* ---- forward ------------------------------------------------------------------------------------- */
typedef struct d3h_forward_args {
  /* inputs (device) */
  const float* pos;        /* (N,3)  tet-grid vertex positions, `pos_nx3`, gshell_tets.py:253 */
  const float* sdf;        /* (N)    `sdf_n` after .float(), gshell_tets.py:254 */
  const float* msdf;       /* (N)    `msdf_n` */
  const int32_t* tets;     /* (F,4)  packed int32x4 tet indices, 16-byte aligned (d3h_pack_tets_i64) */
  int64_t n_grid;          /* N */
  int64_t n_tets;          /* F  (defines the UV atlas size, gshell_tets.py:319) */
  int64_t tet_begin;       /* classify tets [tet_begin, tet_end) only; whole grid = [0,F) */
  int64_t tet_end;
  int32_t msdf_negate;     /* 1 for hmSDF_Tets(type="body"): msdf is used as -msdf (hmsdf_tets_split.py:261-264) */
  int32_t watertight_template; /* `output_watertight_template` (default 1), gshell_tets.py:272-275 */
  /* capacities, in rows, of the caller's output / tape buffers */
  int64_t cap_valid_tets;  /* also sizes the workspace (see d3h_workspace_bytes) */
  int64_t cap_verts;       /* V  rows available in the *_watertight outputs and tape_edges */
  int64_t cap_verts_aug;   /* Va rows available in verts_aug, v_tng_aug, msdf_aug */
  int64_t cap_faces_wt;    /* Fw rows available in faces_watertight */
  int64_t cap_faces_aug;   /* Fa rows available in faces_aug */
  /* outputs (device); any may be NULL with capacity 0 for a counting-only run */
  float* verts_aug;        /* (Va,3) rows not referenced by faces_aug are zero (gshell_tets.py:423-427) */
  float* v_tng_aug;        /* (Va,3) */
  float* msdf_aug;         /* (Va)   extra['msdf']; [V:] is extra['msdf_boundary'] */
  int64_t* faces_aug;      /* (Fa,3) */
  float* verts_wt;         /* (V,3)  extra['vertices_watertight'] */
  float* v_tng_wt;         /* (V,3)  extra['v_tng_watertight'] */
  float* msdf_wt;          /* (V)    extra['msdf_watertight'] */
  int64_t* faces_wt;       /* (Fw,3) extra['faces_watertight'] */
  /* tape for the backward pass (device) */
  int32_t* tape_edges;     /* (cap_verts,2)   (a,b), a<b: grid vertices of each crossing edge, sorted (interp_v, gshell_tets.py:287) */
  int32_t* tape_corners;   /* (4*cap_valid_tets) polygon corner -> watertight vertex id, layout [3*T1 | 4*T2] */
  int32_t* tape_slots;     /* (4*cap_valid_tets) corner slots grouped by watertight vertex (the sorted inverse map);
                              general path only: not written when edge_off is given */
  int32_t* tape_runs;      /* (cap_verts + 1) start of every vertex's run in tape_slots; [V] = P; general path only */
  /* optional: dense gradient buffers of the coming backward call, zero-filled here next to the latency-bound surface
   * stages (pass them to d3h_extract_backward with grads_prezeroed = 1); NULL = not wanted: the backward call zeroes
   * them instead (grads_prezeroed = 0) */
  float* zero_g_pos;       /* (N,3) */
  float* zero_g_sdf;       /* (N)   */
  float* zero_g_msdf;      /* (N)   */
  /* scratch + counts */
  void* workspace;         /* >= d3h_workspace_bytes(F, N, cap_valid_tets) bytes, 256-byte aligned */
  int64_t workspace_bytes;
  d3h_counts* counts_host; /* pinned host memory, or NULL to skip the copy.  The counts are published as soon as they
                              are final -- before the kernels that only write outputs have run -- and `seq` is the
                              last word written: poll it with d3h_wait_counts() instead of synchronising the stream */
  int64_t seq;             /* caller-chosen non-zero tag of this call, echoed in counts_host->seq */
  /* optional: static edge table of the tet grid (d3h_edge_table_*): the tet indices of a training run never change
   * (hmsdf.py:207-212), so the sorted list of ALL distinct tet edges is built once and every call de-duplicates its
   * crossing edges by marking them in a bitmap over that list -- no per-call sort.  edge_off == NULL selects the general
   * path (radix sort + run-length scan of the crossing-edge keys of this call). */
  const int32_t* edge_off; /* (N+1) edges whose smaller endpoint is a have ranks [edge_off[a], edge_off[a+1]) */
  const int32_t* edge_ab;  /* (n_edges,2) (a,b), a<=b, ascending lexicographically: rank -> endpoints */
  int64_t n_edges;
  float* vacc;             /* (cap_verts,8) per-vertex accumulator of the scatter-form adjoint, zeroed here; required
                              with edge_off (the static path leaves no tape_slots / tape_runs) */
  /* optional (d3h_extract_forward only): the PAIR of extractions of one split-stage iteration, hmSDF_Tets(type="cloth")
   * and hmSDF_Tets(type="body") on the same pos / sdf / msdf (train.py:1040-1047).  The second extraction uses the mSDF
   * with the opposite sign of `msdf_negate`; classification, edge de-duplication, vertex positions, normals and tangents
   * are shared (the interpolated mSDF of the second one is the exact negation), only the mSDF cut is redone.  Same
   * capacities as the first set; the tape (tape_edges / tape_corners / tape_slots / tape_runs) is common to both.
   * pair_verts_aug == NULL: no second extraction. */
  float* pair_verts_aug;
  float* pair_v_tng_aug;
  float* pair_msdf_aug;
  int64_t* pair_faces_aug;
  float* pair_verts_wt;
  float* pair_v_tng_wt;
  float* pair_msdf_wt;
  int64_t* pair_faces_wt;
  float* pair_vacc;        /* (cap_verts,8) accumulator of the second extraction's scatter-form adjoint (with edge_off) */
  d3h_counts* pair_counts_host; /* sizes of the second extraction (n_faces_aug, bucket_polys differ), pinned like counts_host */
  int64_t pair_seq;
  /* optional companion of the static edge table (EXPERIMENTAL, opt-in): rank in edge_ab of the 6 edges of every tet,
   * (F,8) int32 rows (edges in the order of gshell_tets.py:187, 2 words of padding), 16-byte aligned.  With it the
   * compaction kernel reads the ranks of a valid tet's edges instead of bisecting the neighbour lists (32 B per valid
   * tet instead of ~5 dependent loads per corner); costs 32 B per tet of device memory.  NULL: bisect. */
  const int32_t* tet_edge_rank;
  /* optional: the EDGE-SCAN path (needs edge_off / edge_ab / tet_edge_rank as well).  With the incidence lists of the
   * static edge table the call never streams the tet array: one kernel walks the edge list (4 bytes per edge instead of
   * 16 per tet), marks the edges whose endpoints differ in sign -- exactly the crossing edges torch.unique would keep,
   * gshell_tets.py:279-287 -- and, through the edge -> tet incidence, the tets around them (exactly the valid tets,
   * :261-275).  Everything downstream is unchanged.  NULL: classify the tets (classify_kernel). */
  const int32_t* edge_b;   /* (n_edges)   larger endpoint of every edge: edge_ab[:,1], contiguous */
  const int32_t* etet_off; /* (n_edges+1) tets around edge r: etets[etet_off[r] .. etet_off[r+1]) */
  const int32_t* etets;    /* (<= 6F)     tet ids, ascending and distinct per edge */
  /* optional companion of the edge-scan path: the same incidence in fixed-width rows, one 32-byte row per edge --
   * the first 8 tets around edge r, padded with -1; [7] == -2 marks an edge with more than 8 tets (the kernel then walks
   * etet_off / etets for it).  One dependent load per crossing edge instead of two.  16-byte aligned.  NULL: CSR only. */
  const int32_t* etets8;   /* (n_edges,8) */
  /* optional companion of the edge-scan path: the larger end points once more, TRANSPOSED per chunk of 32 consecutive
   * grid vertices, so that the walk over the edge list is made of fully coalesced 128-byte rows (lane l of a warp owns
   * vertex 32c + l).  Chunk c owns rows [edge_row_off[c], edge_row_off[c+1]) -- as many as its vertex of highest
   * degree has larger neighbours; entry (row r, lane l) = edge_rows[32 r + l] = the (r - edge_row_off[c])-th larger
   * neighbour of vertex 32c + l in ascending order, i.e. end point b of edge edge_off[32c + l] + r - edge_row_off[c],
   * or the vertex ITSELF where it has fewer (an edge to itself never crosses), 0 for the lanes beyond n_grid in the
   * last chunk.  EIGHT SPARE ROWS of zeros follow the last row (the kernel reads 8 rows from a chunk's first row
   * whatever the chunk's row count and masks the surplus).  128-byte aligned.  With it edge_b may be NULL.
   * NULL: walk edge_b through edge_off. */
  const int32_t* edge_rows;    /* (32 * (edge_row_off[ceil(N/32)] + 8)) */
  const int32_t* edge_row_off; /* (ceil(N/32) + 1) */
  /* optional companion of the edge-scan path, preferred over edge_rows / edge_b when given: the edge list RUN-LENGTH
   * compressed by end-point difference per chunk of 32 consecutive vertices.  Entry k = (d, mask) = edge_runs[2k], [2k+1]
   * of chunk c = edge_run_chunk[k], entries ascending in (c, d), d >= 0: bit l of mask is set iff (32c + l, 32c + l + d) is
   * an edge of the grid, and edge_run_ids[32k + l] is its rank in the sorted edge list (edge_ab; -1 where the bit is
   * clear).  On a lattice numbered along its axes every vertex has the same few differences, so a chunk needs ~7 entries
   * instead of ~224 end points, and the signs of all 32 far end points of an entry are ONE 32-bit window of the sign
   * bitmap: 32 edges are tested with a funnel shift and an xor.  Worth it when entries are shared by several lanes (the
   * host builds it when the grid averages >= 4 edges per entry); exact for any grid. */
  const int32_t* edge_runs;      /* (n_edge_runs, 2) int32, 8-byte aligned */
  const int32_t* edge_run_chunk; /* (n_edge_runs) */
  const int32_t* edge_run_ids;   /* (n_edge_runs, 32) */
  int64_t n_edge_runs;
  /* optional companion of edge_runs: the TET array compressed the same way, so that the valid tets (mixed signs,
   * gshell_tets.py:261-275) are found from the sign bitmap without walking the tets around every crossing edge.  A tet
   * (v0, v1, v2, v3) is filed under the chunk of its FIRST vertex, lane v0 & 31, and its shape (v1 - v0, v2 - v0, v3 - v0):
   * entry k = (d1, d2, d3, mask) = tet_runs[4k .. 4k+3] of chunk tet_run_chunk[k] -- bit l of mask is set iff the grid
   * holds the tet (32c + l, 32c + l + d1, 32c + l + d2, 32c + l + d3), whose index is tet_run_ids[32k + l] (-1 elsewhere).
   * The occupancy codes of the 32 tets of an entry are four 32-bit windows of the sign bitmap.  Needs edge_runs; used on
   * the watertight template only (output_watertight_template = 1).  The host builds it when the grid averages >= 4 tets
   * per entry and no two tets list the same vertices in the same order. */
  const int32_t* tet_runs;       /* (n_tet_runs, 4) int32, 16-byte aligned */
  const int32_t* tet_run_chunk;  /* (n_tet_runs) */
  const int32_t* tet_run_ids;    /* (n_tet_runs, 32) */
  int64_t n_tet_runs;
} d3h_forward_args;

/* ---- backward ------------------------------------------------------------------------------------ */
typedef struct d3h_backward_args {
  /* forward inputs again */
  const float* pos;
  const float* sdf;
  const float* msdf;
  int64_t n_grid;
  int32_t msdf_negate;
  int32_t grads_prezeroed; /* 1: g_pos / g_sdf / g_msdf are zero on entry (the forward call filled them, zero_g_*);
                              0: the backward call zeroes them before it accumulates */
  /* saved by forward */
  const int32_t* tape_edges;
  const int32_t* tape_corners;
  const int32_t* tape_slots;
  const int32_t* tape_runs;
  const float* verts_wt;   /* (V,3) */
  const float* msdf_wt;    /* (V)   */
  int64_t n_verts;         /* V  */
  int64_t n_tri_tets;      /* T1 */
  int64_t n_quad_tets;     /* T2 */
  /* upstream gradients (device); NULL = zero */
  const float* g_verts_aug;   /* (Va,3) */
  const float* g_msdf_aug;    /* (Va)   */
  const float* g_verts_wt;    /* (V,3)  */
  const float* g_msdf_wt;     /* (V)    */
  /* outputs (device); fully written (zero where nothing flows) */
  float* g_pos;            /* (N,3) */
  float* g_sdf;            /* (N)   */
  float* g_msdf;           /* (N) or NULL (type="body" has no msdf gradient) */
  /* scratch (unused since the adjoint became a gather over tape_slots; kept for ABI stability, may be NULL) */
  void* workspace;
  int64_t workspace_bytes;
  /* optional second upstream gradient of the augmented mSDF, for its boundary slice only: extra['msdf_boundary'] is
   * msdf[V:] (gshell_tets.py:397), (Va - V) rows; added to g_msdf_aug[V:] by the kernel.  NULL = none */
  const float* g_msdf_boundary;
  /* static-edge-table calls: tape_slots / tape_runs are NULL and the adjoint runs in scatter form through this
   * (n_verts,8) accumulator (zero on entry -- the forward call zeroes it -- and zero again on return) */
  float* vacc;
  /* optional: what arrives through the TANGENT branch (d3h_tangent_backward, SURVEY A.5 "optional branch"): gradient
   * w.r.t. the watertight vertex positions (V,3) and w.r.t. the interpolated mSDF through the boundary coefficients (V);
   * added to the per-vertex gradients before the crossing-edge step.  NULL = none. */
  const float* g_verts_tng;
  const float* g_mvert_tng;
} d3h_backward_args;

/* ---- tangent branch of the backward pass (optional) ---------------------------------------------------------------
 * Adjoint of auto_normals (gshell_tets.py:9-34), compute_tangents (:40-78: per-face tangents from the vertex-id UVs,
 * scatter-mean, normalise, Gram-Schmidt against the normal, normalise) and of the boundary interpolation of the tangents
 * (:380-385), for upstream gradients on v_tng_aug (Va,3) and / or extra['v_tng_watertight'] (V,3).  D3-Human never
 * back-propagates through the tangents (hmsdf.py:454,548 drop them); provided for API completeness.  Writes g_verts
 * (V,3) and g_mvert (V) -- pass them to d3h_extract_backward as g_verts_tng / g_mvert_tng.  `workspace`: 16 floats per
 * watertight vertex, 16-byte aligned.  A watertight mesh of exactly three faces (the torch.cross quirk, :19) is refused
 * with D3H_E_BADARG. */
typedef struct d3h_tangent_backward_args {
  const float* verts_wt;        /* (V,3)  extra['vertices_watertight'] of the forward call */
  const float* msdf_wt;         /* (V)    */
  const float* v_tng_wt;        /* (V,3)  extra['v_tng_watertight'] */
  const int64_t* faces_wt;      /* (Fw,3) */
  const int32_t* tape_corners;  /* polygon corner -> watertight vertex id, [3*T1 | 4*T2] */
  int64_t n_verts, n_tri_tets, n_quad_tets;
  int64_t n_tets;               /* F of the grid (defines the UV atlas, gshell_tets.py:319) */
  const float* g_tng_aug;       /* (Va,3) or NULL */
  const float* g_tng_wt;        /* (V,3)  or NULL */
  float* g_verts;               /* (V,3) out */
  float* g_mvert;               /* (V)   out */
  void* workspace;
  int64_t workspace_bytes;      /* >= 64 * V */
} d3h_tangent_backward_args;
int d3h_tangent_backward(const d3h_tangent_backward_args* args, d3h_stream_t stream);

int d3h_version(void);
const char* d3h_last_error_string(void);

/* Scratch sizes.  Replaces nothing in the reference (torch allocates every temporary there). */
int64_t d3h_workspace_bytes(int64_t n_tets, int64_t n_grid, int64_t cap_valid_tets);
/* ... when the calls carry a static edge table of n_edges entries (adds the edge bitmap and its prefix words) */
int64_t d3h_workspace_bytes_static(int64_t n_tets, int64_t n_grid, int64_t cap_valid_tets, int64_t n_edges);
int64_t d3h_backward_workspace_bytes(int64_t n_verts);

/* One-time conversion of the static `tet_fx4` (int64 in the reference, hmsdf.py:207-212) to packed int32x4,
 * with a range check against N; the number of out-of-range indices is added to *bad_count_dev (device int64,
 * caller-zeroed).  d3h_check_tets_i32 validates an int32 grid in place. */
int d3h_pack_tets_i64(const int64_t* tets, int64_t n_tets, int64_t n_grid, int32_t* out_tets,
                      int64_t* bad_count_dev, d3h_stream_t stream);
int d3h_check_tets_i32(const int32_t* tets, int64_t n_tets, int64_t n_grid, int64_t* bad_count_dev,
                       d3h_stream_t stream);

/* The whole forward extraction (replaces GShell_Tets.__call__ / hmSDF_Tets.__call__ up to the return
 * statement, gshell_tets.py:254-445). */
int d3h_extract_forward(const d3h_forward_args* args, d3h_stream_t stream);

/* Host-side wait for the counts of call `seq`: spins on counts_host->seq (the reference blocks the host ~40 times per
 * call on boolean-mask sizes; this is the single size read of this implementation).  Returns 0, or D3H_E_TIMEOUT after
 * timeout_us microseconds (<= 0: wait forever). */
int d3h_wait_counts(const d3h_counts* counts_host, int64_t seq, int64_t timeout_us);

/* Adjoint of the float pipeline (replaces autograd through gshell_tets.py:291-303, 342-397, 427). */
int d3h_extract_backward(const d3h_backward_args* args, d3h_stream_t stream);

/* Batches of independent extractions: the video frames of one training step (BASELINE.json configs[3]) or the
 * cloth / body pair the reference extracts every iteration (train.py:1040-1047).  No counterpart in the reference, which
 * runs them one after the other.  Frame i runs on internal lane (i % lanes), lanes <= 8; the lanes fork from `stream`
 * and join back into it, so the batch is ordered on `stream` like a single call.  The bandwidth-bound kernels of one
 * frame overlap the latency-bound surface kernels of the others (per-kernel launch priorities).
 *   forward : args[i] as for d3h_extract_forward; frames on different lanes need distinct workspaces (frames of the same
 *             lane may share one); every frame publishes its own counts (args[i].counts_host, args[i].seq).
 *   backward: gradient buffers may be shared between frames (sdf / msdf common to all frames): all frames accumulate
 *             with atomics.  The buffers of the frames with grads_prezeroed = 0 are zeroed first, in one launch, a
 *             shared buffer once; with grads_prezeroed = 1 on every frame that uses it, a buffer must be zero on entry.
 *             Frames without a surface or without upstream gradients are zeroed too and otherwise skipped.  The
 *             adjoints of up to 16 consecutive frames are one kernel launch (grid.y = frame); `lanes` is ignored. */
int d3h_extract_forward_batch(const d3h_forward_args* args, int64_t n_frames, int32_t lanes, d3h_stream_t stream);
/* The same without the final join: `stream` is not ordered behind the lanes until d3h_lanes_join(stream).  Batches
 * launched back to back this way queue up per lane (no drain / refill of the lanes at the batch boundary); the caller
 * joins before `stream` touches an output, or frees a buffer, of those batches. */
int d3h_extract_forward_batch_nojoin(const d3h_forward_args* args, int64_t n_frames, int32_t lanes, d3h_stream_t stream);
int d3h_lanes_join(d3h_stream_t stream);
int d3h_extract_backward_batch(const d3h_backward_args* args, int64_t n_frames, int32_t lanes, d3h_stream_t stream);

/* Compact gradient return.  The rows of a dense (N, width) gradient that one extraction can have touched are the end
 * points of its crossing edges: `ids` = the frame's tape_edges read as a flat list of 2V vertex ids (the crossing edges
 * of gshell_tets.py:281-287).  out[i][:] = src[ids[i]][:] (ids outside [0, n_rows) give zero rows); an id that occurs
 * several times yields the same row every time, so a consumer ASSIGNS dense[ids] = out.  Lets a host-side caller fetch
 * ~2V rows instead of N (the dense gradient is > 99 % zeros). */
int d3h_gather_rows(const int32_t* ids, int64_t n_ids, const float* src, int64_t n_rows, int32_t width, float* out,
                    d3h_stream_t stream);

/* Tet-range sharding (multi-GPU, SURVEY.md section 8e): stage 1 classifies tets [tet_begin, tet_end) and leaves
 * compact valid-tet records in the caller's buffers; the ranks all-gather those (NCCL) and stage 2 runs the
 * surface stages on the concatenated records.  d3h_extract_forward == stage 1 on [0,F) + stage 2. */
typedef struct d3h_tet_record { /* 32 bytes */
  int32_t v[4];            /* tet vertex ids */
  int32_t code;            /* 4-bit occupancy code, gshell_tets.py:307-308 */
  int32_t class_rank;      /* rank among the shard's valid tets with the same triangle count (T1 or T2 class) */
  int32_t tet_id;          /* global tet index */
  int32_t other_before;    /* number of the shard's valid tets of the OTHER class that precede this one */
} d3h_tet_record;

int d3h_classify_range(const d3h_forward_args* args, d3h_tet_record* records_out, int64_t cap_records,
                       d3h_counts* counts_dev_out, d3h_stream_t stream);
int d3h_extract_from_records(const d3h_forward_args* args, const d3h_tet_record* records, int64_t n_tri_tets,
                             int64_t n_quad_tets, d3h_stream_t stream);

/* ---- SDF sign-change regulariser (compute_sdf_reg_loss, hmsdf.py:162-170) --------------------------------------------
 * Over the distinct edges (a, b) of a grid, given as ONE of the two static tables of the edge scan above (edge_runs +
 * edge_run_chunk, or edge_rows + edge_row_off, same layouts as in d3h_forward_args; the other pair NULL), an edge is
 * selected when sign(sdf[a]) != sign(sdf[b]) with the three-valued sign (0 differs from both signs; +0.0 and -0.0 do
 * not differ; an edge to itself is never selected).  With M selected edges:
 *     loss = mean_e BCE(sdf[a], [sdf[b] > 0]) + mean_e BCE(sdf[b], [sdf[a] > 0]),  BCE(x, t) = (1 - t) x - log_sigmoid(x)
 * NaN when M == 0 (the mean of an empty selection) or when sdf holds a NaN anywhere.  ±inf is not handled specially.
 * The loss is summed in float64 in a fixed order: the same inputs give the same bits on every run.
 * workspace: d3h_sdf_reg_workspace_bytes(N, n_edge_runs) bytes (n_edge_runs = 0 with the rows form), 16-byte aligned;
 * the forward call leaves the sign bitmaps and M there for the backward call, which must use the same workspace, sdf
 * and tables.  Both calls are asynchronous on `stream` and never wait for the device. */
int64_t d3h_sdf_reg_workspace_bytes(int64_t n_grid, int64_t n_entries);
/* *loss (one float, device memory) */
int d3h_sdf_reg_forward(const float* sdf, int64_t n_grid, const int32_t* edge_runs, const int32_t* edge_run_chunk,
                        int64_t n_edge_runs, const int32_t* edge_rows, const int32_t* edge_row_off, void* workspace,
                        int64_t workspace_bytes, float* loss, d3h_stream_t stream);
/* g_sdf[a] += g (sigmoid(sdf[a]) - [sdf[b] > 0]) / M and g_sdf[b] += g (sigmoid(sdf[b]) - [sdf[a] > 0]) / M over the
 * selected edges; g = *g_loss (device memory), M from the workspace.  g_sdf (N) ACCUMULATES (zero it first). */
int d3h_sdf_reg_backward(const float* sdf, int64_t n_grid, const int32_t* edge_runs, const int32_t* edge_run_chunk,
                         int64_t n_edge_runs, const int32_t* edge_rows, const int32_t* edge_row_off, const float* g_loss,
                         void* workspace, int64_t workspace_bytes, float* g_sdf, d3h_stream_t stream);

/* ---- diagnostics (no counterpart in the reference) ------------------------------------------------------------- */
/* Per-kernel device time: when enabled, every kernel launch of this library is bracketed by cudaEventRecord on the
 * launching stream.  d3h_profile_read synchronises those events, returns the summed milliseconds and launch counts
 * per kernel kind (arrays of d3h_profile_kinds() entries, names from d3h_profile_kernel_name) and clears the log. */
int d3h_profile_enable(int on);
int d3h_profile_kinds(void);
const char* d3h_profile_kernel_name(int kind);
int d3h_profile_read(float* ms_by_kind, int* launches_by_kind);
/* Timeline form: start / end (ms since the first recorded launch), kernel kind and a stream ordinal per launch, in launch
 * order; returns the number of entries written (<= cap) and clears the log. */
int d3h_profile_timeline(float* start_ms, float* end_ms, int* kind, int* stream_id, int cap);

/* Diagnostics: the dominant kernel of the edge-scan path timed ALONE -- `reps` launches of edge_scan_kernel on the state
 * the last forward call with these arguments left in its workspace (argument block, sign bitmap), each between its own
 * pair of CUDA events on `stream`; before every launch `flush` (caller-owned, > L2 size, 16-byte aligned; NULL = no flush)
 * is READ through so that the static edge list comes from HBM, not from L2 (a fill would leave dirty lines behind).  *ms_total = sum of the per-launch times (synchronises the
 * stream).  The work queues of the workspace overflow harmlessly (writes are capacity-checked); the next forward call
 * resets them.  bench.py divides the kernel's algorithmic bytes by ms_total / reps for `roofline`. */
int d3h_profile_scan_kernel(const d3h_forward_args* args, int32_t reps, void* flush, int64_t flush_bytes, float* ms_total,
                            d3h_stream_t stream);
/* Device-side trace, usable inside the cached CUDA graphs: every forward kernel stamps %globaltimer when its first block
 * starts and when its last block exits.  d3h_trace_read fills out[64][24][2] (uint64 ns; row = seq % 64, column = kernel
 * kind as in d3h_profile_kernel_name) and clears the table.  enabling allocates a 24 KB device table (diagnostics only). */
int d3h_trace_enable(int on);
int d3h_trace_read(uint64_t* out);
/* Host copies of the case tables the kernels index (same initialisers as the __constant__ copies; no GPU needed).
 * which: 0 num_triangles[16], 1 polygon loop edges[16][4], 2 triangle_table[16][6], 3 triangle_table_tri[8][6],
 * 4 num_triangles_tri[8], 5 triangle_table_quad[16][12], 6 num_triangles_quad[16], 7/8 tet-edge endpoints[6].
 * Returns the element count written to `out`. */
int d3h_debug_table(int which, int8_t* out, int cap);

#ifdef __cplusplus
}
#endif
#endif /* D3H_TETS_H_ */
