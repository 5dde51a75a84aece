"""Host side of the extraction: capacity planning, workspace / tet-index caches and the autograd.Function.

Mirrors the contract of the reference's `GShell_Tets.__call__` (geometry/gshell_tets.py:253-447) and
`hmSDF_Tets.__call__` (geometry/hmsdf_tets_split.py:254-454): same inputs, same 6-tuple, same `extra` keys, gradients
to `pos_nx3`, `sdf_n`, `msdf_n`.  All arithmetic happens in libd3h_tets.so (hand-written sm_100a kernels); torch is used
for device memory, the current stream and autograd bookkeeping only.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Tuple

import numpy as np
import torch

from . import _cabi

ctypes_array = Any

_SLACK_NUM, _SLACK_DEN, _SLACK_ABS = 9, 8, 1024  # capacity = need * 9/8 + 1024 rows


def _grow(n: int) -> int:
    return n * _SLACK_NUM // _SLACK_DEN + _SLACK_ABS


# --------------------------------------------------------------------------------------------------
# static tet indices: converted once to packed int32x4 and range-checked (tet_fx4 is static for a whole
# training run, hmsdf.py:207-212; the reference re-reads the int64 array every call)
# --------------------------------------------------------------------------------------------------
_packed_cache: Dict[Tuple, Tuple[torch.Tensor, "weakref.ref"]] = {}


def packed_tets(tet_fx4: torch.Tensor, n_grid: int) -> torch.Tensor:
    """(F,4) integer tensor on a CUDA device -> contiguous int32 (F,4), 16-byte aligned, validated against N.
    Cached on (data_ptr, version, shape, dtype, device, N)."""
    if tet_fx4.dim() != 2 or tet_fx4.shape[1] != 4:
        raise ValueError(f"tet_fx4 must have shape (F,4), got {tuple(tet_fx4.shape)}")
    if not tet_fx4.is_cuda:
        raise RuntimeError("d3human-code_b200 has no CPU path: tet_fx4 must live on a CUDA device")
    key = (tet_fx4.data_ptr(), tet_fx4._version, tuple(tet_fx4.shape), tet_fx4.dtype, tet_fx4.device, int(n_grid))
    hit = _packed_cache.get(key)
    if hit is not None and hit[1]() is not None:
        return hit[0]
    L = _cabi.lib()
    n_tets = tet_fx4.shape[0]
    stream = torch.cuda.current_stream(tet_fx4.device).cuda_stream
    bad = torch.zeros(1, dtype=torch.int64, device=tet_fx4.device)
    with torch.cuda.device(tet_fx4.device):
        if tet_fx4.dtype == torch.int32 and tet_fx4.is_contiguous() and tet_fx4.data_ptr() % 16 == 0:
            out = tet_fx4
            _cabi.check(L.d3h_check_tets_i32(out.data_ptr(), n_tets, n_grid, bad.data_ptr(), stream), "d3h_check_tets_i32")
        else:
            src = tet_fx4.contiguous().to(torch.int64)
            out = torch.empty((n_tets, 4), dtype=torch.int32, device=tet_fx4.device)
            _cabi.check(L.d3h_pack_tets_i64(src.data_ptr(), n_tets, n_grid, out.data_ptr(), bad.data_ptr(), stream),
                        "d3h_pack_tets_i64")
    nbad = int(bad.item())  # one-time sync per grid
    if nbad:
        raise IndexError(f"tet_fx4 holds {nbad} vertex indices outside [0, {n_grid})")
    if len(_packed_cache) > 16:
        for k in [k for k, v in _packed_cache.items() if v[1]() is None]:
            del _packed_cache[k]
    try:
        ref = weakref.ref(tet_fx4)
    except TypeError:  # pragma: no cover
        ref = lambda: tet_fx4  # noqa: E731
    _packed_cache[key] = (out, ref)
    return out


# --------------------------------------------------------------------------------------------------
# static edge table: the sorted list of ALL distinct tet edges of a grid, built once per tet array.  With it a call
# de-duplicates its crossing edges by marking a bitmap over the list (rank among the marked edges = vertex id, the order
# of torch.unique(dim=0) at gshell_tets.py:279) instead of sorting their keys.
# --------------------------------------------------------------------------------------------------
_TET_EDGES = ((0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3))   # gshell_tets.py:187
_static_cache: Dict[Tuple, list] = {}
_static_mode = os.environ.get("D3H_STATIC_EDGES", "auto")       # "auto": from the 2nd call on the same tets, "1", "0"
_tet_edge_ranks = os.environ.get("D3H_TET_EDGE_RANKS", "0") == "1"   # per-tet edge-rank table for compact_kernel<3> (+32 B / tet)
#: edge-scan path (csrc/d3h_scan.cu): with the static tables a call walks the edge list (4 B / edge) instead of streaming
#: the tet array (16 B / tet); needs the edge -> tet incidence and the per-tet edge ranks (+56 B / tet of static tables)
_edge_scan = os.environ.get("D3H_EDGE_SCAN", "1") == "1"
#: transposed copy of the edge list for the stream kernel (edge_scan_rows_kernel: coalesced 128-byte rows per chunk of 32
#: vertices); replaces edge_b.  D3H_SCAN_ROWS=0 keeps the CSR walk (edge_scan_kernel)
_scan_rows = os.environ.get("D3H_SCAN_ROWS", "1") == "1"
#: run-length compressed edge list for the stream kernel (edge_scan_runs_kernel: one (difference, lane mask) entry stands
#: for up to 32 edges); built instead of the rows when the grid averages >= _RUNS_MIN_EDGES edges per entry (lattices
#: numbered along their axes: 32).  D3H_SCAN_RUNS=0 never builds it
_scan_runs = os.environ.get("D3H_SCAN_RUNS", "1") == "1"
_RUNS_MIN_EDGES = 4
#: opt-in: fixed-width incidence rows (etets8, +32 B / edge) for the rule-based marking kernel (edge_mark_rows_kernel)
_mark_rows = os.environ.get("D3H_MARK_ROWS", "0") == "1"


def set_edge_scan(on: bool) -> None:
    """Tables already built keep their form (reset_plans() drops them)."""
    global _edge_scan
    _edge_scan = bool(on)


def set_scan_rows(on: bool) -> None:
    """Build the transposed edge rows with the next edge table (tables already built keep their form)."""
    global _scan_rows
    _scan_rows = bool(on)


def set_scan_runs(on: bool) -> None:
    """Allow the run-length compressed edge list with the next edge table (tables already built keep their form)."""
    global _scan_runs
    _scan_runs = bool(on)


def set_mark_rows(on: bool) -> None:
    """Build the fixed-width incidence rows with the next edge table (the library uses them when D3H_MARK_ROWS=1)."""
    global _mark_rows
    _mark_rows = bool(on)



def set_tet_edge_ranks(on: bool) -> None:
    """EXPERIMENTAL: also build the per-tet edge-rank table with the static edge table (tables already built keep their form)."""
    global _tet_edge_ranks
    _tet_edge_ranks = bool(on)


def set_static_edges(mode: str) -> None:
    """'auto' (default): build the static edge table when a tet array is used a second time (a training run reuses
    it every iteration); '1': build it on first use; '0': always take the general per-call sort path."""
    global _static_mode
    if mode not in ("auto", "0", "1"):
        raise ValueError(mode)
    _static_mode = mode


def build_edge_table(tets_i32: torch.Tensor, n_grid: int):
    """One-time setup on the device (torch sort of the 6F edge keys; not on the per-call path).
    Returns (edge_off (N+1,) int32, edge_ab (U,2) int32, U, tet_rank, edge_b, etet_off, etets, etets8, edge_rows,
    edge_row_off, (edge_runs, edge_run_chunk, edge_run_ids), (tet_runs, tet_run_chunk, tet_run_ids)): edges ascending in
    (min,max), CSR offsets per min vertex.  Entries 3 .. 9 and the members of the two triples are None unless asked for:
      edge_rows, edge_row_off : the larger end points transposed per chunk of 32 vertices (layout: include/d3h_tets.h);
                                edge_b is None then
      edge_runs, edge_run_chunk, edge_run_ids : the edge list run-length compressed by end-point difference per chunk
                                (include/d3h_tets.h); edge_rows and edge_b are None then
      tet_runs, tet_run_chunk, tet_run_ids : the tet array compressed by shape per chunk (build_tet_runs), with edge_runs
      tet_rank (F,8) int32 : rank in the edge list of the six edges of every tet (order of gshell_tets.py:187, 2 pad words)
      edge_b   (U,)  int32 : the larger endpoints, contiguous (the 4-byte-per-edge stream of the edge-scan path)
      etet_off (U+1,), etets (<=6F,) int32 : the tets around every edge, ascending and distinct tet ids
      etets8 (U,8) int32 : the first 8 of them per edge in fixed-width rows (-1 padding, [7] = -2: more than 8)."""
    t = tets_i32.long()
    n_tets = t.shape[0]
    key6 = torch.stack([torch.minimum(t[:, i], t[:, j]) * n_grid + torch.maximum(t[:, i], t[:, j]) for i, j in _TET_EDGES], 1)
    del t
    uk = torch.unique(key6.reshape(-1))          # ascending
    ea = torch.div(uk, n_grid, rounding_mode="floor")
    edge_ab = torch.stack([ea, uk - ea * n_grid], 1).to(torch.int32).contiguous()
    counts = torch.bincount(ea, minlength=n_grid)
    edge_off = torch.zeros(n_grid + 1, dtype=torch.int64, device=tets_i32.device)
    edge_off[1:] = torch.cumsum(counts, 0)
    del ea, counts
    n_edges = int(uk.shape[0])
    if n_edges >= 2 ** 31:
        raise ValueError("tet grid has more than 2^31 distinct edges")
    tet_rank = edge_b = etet_off = etets = etets8 = edge_rows = edge_row_off = None
    edge_runs = edge_run_chunk = edge_run_ids = tet_runs = tet_run_chunk = tet_run_ids = None
    if _tet_edge_ranks or _edge_scan:
        rank6 = torch.searchsorted(uk, key6.reshape(-1)).reshape(n_tets, 6)
        del key6
        tet_rank = torch.zeros((n_tets, 8), dtype=torch.int32, device=tets_i32.device)
        tet_rank[:, :6] = rank6.to(torch.int32)
        if _edge_scan:
            flat = rank6.reshape(-1)             # entry t*6 + e
            order = torch.argsort(flat, stable=True)
            eid = flat[order]                    # edge of every (edge, tet) incidence, ascending; tets ascending per edge
            tid = torch.div(order, 6, rounding_mode="floor")
            del order
            # a tet that lists a vertex twice meets one of its edges twice: keep every (edge, tet) pair once
            keep = torch.ones_like(eid, dtype=torch.bool)
            keep[1:] = (eid[1:] != eid[:-1]) | (tid[1:] != tid[:-1])
            if not bool(keep.all()):
                eid, tid = eid[keep], tid[keep]
            del keep
            etets = tid.to(torch.int32).contiguous()
            off64 = torch.zeros(n_edges + 1, dtype=torch.int64, device=tets_i32.device)
            off64[1:] = torch.cumsum(torch.bincount(eid, minlength=n_edges), 0)
            etet_off = off64.to(torch.int32).contiguous()
            if _scan_runs:
                edge_runs, edge_run_chunk, edge_run_ids = build_edge_runs(edge_off, edge_ab, n_grid)
            if edge_runs is not None:
                tet_runs, tet_run_chunk, tet_run_ids = build_tet_runs(tets_i32, n_grid)
            elif _scan_rows:
                edge_rows, edge_row_off = build_edge_rows(edge_off, edge_ab, n_grid)
            else:
                edge_b = edge_ab[:, 1].contiguous()
            if _mark_rows:
                # fixed-width rows: the first 8 tets of every edge (one 32-byte load per crossing edge), -2 in the last
                # slot of an edge with more than 8
                within = torch.arange(eid.shape[0], device=eid.device) - off64[eid]
                sel = within < 8
                etets8 = torch.full((n_edges, 8), -1, dtype=torch.int32, device=tets_i32.device)
                etets8[eid[sel], within[sel]] = etets[sel]
                etets8[(off64[1:] - off64[:-1]) > 8, 7] = -2
                del within, sel
            del eid, tid, off64
        del rank6
    return (edge_off.to(torch.int32).contiguous(), edge_ab, n_edges, tet_rank, edge_b, etet_off, etets, etets8, edge_rows,
            edge_row_off, (edge_runs, edge_run_chunk, edge_run_ids), (tet_runs, tet_run_chunk, tet_run_ids))


def build_tet_runs(tets_i32: torch.Tensor, n_grid: int, min_tets_per_entry: Optional[float] = None):
    """The tet array compressed by shape per chunk of 32 consecutive FIRST vertices (one-time setup; companion of
    build_edge_runs): -> (tet_runs (K,4) int32 rows (d1, d2, d3, mask), tet_run_chunk (K,) int32, tet_run_ids (K,32)
    int32) as d3h_forward_args.tet_runs describes, or (None, None, None) when the grid averages fewer than
    `min_tets_per_entry` tets per entry or two tets list the same vertices in the same order."""
    if min_tets_per_entry is None:
        min_tets_per_entry = _RUNS_MIN_EDGES
    dev = tets_i32.device
    n_tets = tets_i32.shape[0]
    t = tets_i32.long()
    v0 = t[:, 0]
    span = 2 * n_grid                                     # differences lie in (-N, N)
    k12 = (t[:, 1] - v0 + n_grid) * span + (t[:, 2] - v0 + n_grid)
    u12, i12 = torch.unique(k12, return_inverse=True)
    k123 = i12 * span + (t[:, 3] - v0 + n_grid)
    del k12, i12
    upat, pid = torch.unique(k123, return_inverse=True)   # the distinct shapes (6 on a Kuhn lattice)
    del k123, t
    n_pat = int(upat.shape[0])
    uk, inv = torch.unique((v0 >> 5) * n_pat + pid, return_inverse=True)   # entries ascending in (chunk, shape)
    del pid
    n_runs = int(uk.shape[0])
    if n_runs == 0 or n_tets < min_tets_per_entry * n_runs or n_runs >= 2 ** 26:
        return None, None, None
    slot = inv * 32 + (v0 & 31)
    ids = torch.full((n_runs * 32,), -1, dtype=torch.int32, device=dev)
    ids[slot] = torch.arange(n_tets, dtype=torch.int32, device=dev)
    if int((ids >= 0).sum()) != n_tets:                   # two tets in one slot: identical vertex lists
        return None, None, None
    mask = torch.zeros(n_runs, dtype=torch.int64, device=dev)
    mask.scatter_add_(0, inv, torch.ones_like(v0) << (v0 & 31))
    mask = torch.where(mask >= 2 ** 31, mask - 2 ** 32, mask)
    chunk = torch.div(uk, n_pat, rounding_mode="floor")
    k123 = upat[uk - chunk * n_pat]
    q12 = torch.div(k123, span, rounding_mode="floor")
    d3 = k123 - q12 * span - n_grid
    k12 = u12[q12]
    d1 = torch.div(k12, span, rounding_mode="floor")
    d2 = k12 - d1 * span - n_grid
    runs = torch.stack([d1 - n_grid, d2, d3, mask], 1).to(torch.int32).contiguous()
    return runs, chunk.to(torch.int32).contiguous(), ids.view(n_runs, 32)


def build_edge_runs(edge_off: torch.Tensor, edge_ab: torch.Tensor, n_grid: int, min_edges_per_entry: Optional[float] = None):
    """The sorted edge list run-length compressed by end-point difference per chunk of 32 consecutive vertices (one-time
    setup): -> (edge_runs (K,2) int32 rows (d, mask), edge_run_chunk (K,) int32, edge_run_ids (K,32) int32), entries
    ascending in (chunk, d), bit l of mask set iff (32c + l, 32c + l + d) is an edge, whose rank in the sorted list is
    ids[k, l] (d3h_forward_args.edge_runs) -- or (None, None, None) when the grid averages fewer than
    `min_edges_per_entry` edges per entry (vertex numbering without structure: the transposed rows are the better
    table).  Self edges (d = 0, tets that repeat a vertex) never cross (the window is the chunk's own word); they are kept
    for simplicity."""
    if min_edges_per_entry is None:
        min_edges_per_entry = _RUNS_MIN_EDGES
    dev = edge_ab.device
    n_edges = edge_ab.shape[0]
    a, b = edge_ab[:, 0].long(), edge_ab[:, 1].long()
    key = (a >> 5) * n_grid + (b - a)                     # (chunk, difference): ascending = the order of the entries
    uk, inv = torch.unique(key, return_inverse=True)
    n_runs = int(uk.shape[0])
    if n_runs == 0 or n_edges < min_edges_per_entry * n_runs or n_runs >= 2 ** 26:
        return None, None, None
    lane = a & 31
    mask = torch.zeros(n_runs, dtype=torch.int64, device=dev)
    mask.scatter_add_(0, inv, torch.ones_like(a) << lane)           # distinct edges: every (entry, lane) is added once
    mask = torch.where(mask >= 2 ** 31, mask - 2 ** 32, mask)       # as int32 bit patterns
    ids = torch.full((n_runs * 32,), -1, dtype=torch.int32, device=dev)
    ids[inv * 32 + lane] = torch.arange(n_edges, dtype=torch.int32, device=dev)
    chunk = torch.div(uk, n_grid, rounding_mode="floor")
    runs = torch.stack([uk - chunk * n_grid, mask], 1).to(torch.int32).contiguous()
    return runs, chunk.to(torch.int32).contiguous(), ids.view(n_runs, 32)


def build_edge_rows(edge_off: torch.Tensor, edge_ab: torch.Tensor, n_grid: int):
    """The larger end points of the sorted edge list, transposed per chunk of 32 consecutive vertices (one-time setup).
    -> (edge_rows (32 (R + 8),) int32, edge_row_off (ceil(N/32)+1,) int32); chunk c owns rows [off[c], off[c+1]), as many as
    its vertex of highest degree has larger neighbours; entry 32 r + l = neighbour r - off[c] of vertex 32 c + l, or the
    vertex itself where it has fewer, or 0 beyond the grid (d3h_forward_args.edge_rows)."""
    dev = edge_ab.device
    off = edge_off.long()
    n_chunks = (n_grid + 31) // 32
    deg = torch.zeros(n_chunks * 32, dtype=torch.int64, device=dev)
    deg[:n_grid] = off[1:] - off[:-1]
    width = deg.view(n_chunks, 32).max(1).values
    row_off = torch.zeros(n_chunks + 1, dtype=torch.int64, device=dev)
    row_off[1:] = torch.cumsum(width, 0)
    n_rows = int(row_off[-1])
    if n_rows >= 2 ** 31 // 32:
        raise ValueError("tet grid too large for the transposed edge rows")
    # every slot starts as its own vertex ...
    chunk_of_row = torch.repeat_interleave(torch.arange(n_chunks, device=dev), width)
    rows = chunk_of_row[:, None] * 32 + torch.arange(32, device=dev)[None, :]
    rows[rows >= n_grid] = 0
    # 8 spare rows close the table: the stream kernel always reads 8 rows from a chunk's first one
    flat = rows.to(torch.int32).reshape(-1)
    store = torch.zeros(flat.shape[0] + 8 * 32 + 32, dtype=torch.int32, device=dev)
    lead = (-store.data_ptr() % 128) // 4          # (CUDA allocations are 512-byte aligned; CPU tensors of the tests are not)
    rows = store[lead:lead + flat.shape[0] + 8 * 32]
    rows[:flat.shape[0]] = flat
    del flat
    # ... and edge e = edge_off[a] + j goes to row off[a >> 5] + j, lane a & 31
    a = edge_ab[:, 0].long()
    j = torch.arange(edge_ab.shape[0], device=dev) - off[a]
    rows[(row_off[a >> 5] + j) * 32 + (a & 31)] = edge_ab[:, 1]
    assert rows.data_ptr() % 128 == 0 and rows.is_contiguous()
    return rows, row_off.to(torch.int32).contiguous()


def static_edges_for(tets_i32: torch.Tensor, n_grid: int):
    """-> (edge_off, edge_ab, n_edges) or None, according to the static-edge policy."""
    if _static_mode == "0" or tets_i32.shape[0] == 0:
        return None
    # the version counter is part of the key: an int32 tet_fx4 is used in place (packed_tets returns the caller's tensor),
    # an in-place edit must not find the edge table of the old contents
    key = (tets_i32.data_ptr(), tets_i32._version, tets_i32.shape[0], int(n_grid), tets_i32.device.index, _edge_scan,
           _tet_edge_ranks, _mark_rows, _scan_rows, _scan_runs)
    ent = _static_cache.get(key)
    if ent is None:
        if len(_static_cache) > 8:
            _static_cache.clear()
        ent = _static_cache[key] = [0, None, tets_i32]   # the packed tensor is kept alive: its address is the key
    ent[0] += 1
    if ent[1] is None and (_static_mode == "1" or ent[0] >= 2):
        with torch.cuda.device(tets_i32.device):
            ent[1] = build_edge_table(tets_i32, n_grid)
    return ent[1]


# --------------------------------------------------------------------------------------------------
# argument blocks as int64 matrices: d3h_forward_args / d3h_backward_args are arrays of 8-byte words (the two int32
# flags share one word), so the blocks of a whole batch are filled with a handful of vectorised numpy assignments
# (pointers of frame i are affine in i) instead of ~35 ctypes attribute writes per frame
# --------------------------------------------------------------------------------------------------
def _columns(struct):
    cols = {}
    for name, _typ in struct._fields_:
        off = getattr(struct, name).offset
        cols[name] = off // 8
    return cols, C.sizeof(struct) // 8


_FC, _FW = _columns(_cabi.ForwardArgs)
_BC, _BW = _columns(_cabi.BackwardArgs)
assert _FC["watertight_template"] == _FC["msdf_negate"] and _BC["grads_prezeroed"] == _BC["msdf_negate"]
_CC, _CW = _columns(_cabi.Counts)

MAX_LANES = 8
DEFAULT_LANES = 4


# --------------------------------------------------------------------------------------------------
# per-(device, F, N) plan: workspaces (one per lane) + capacities predicted from the previous call
# --------------------------------------------------------------------------------------------------
@dataclass
class _Plan:
    device: torch.device
    n_tets: int
    n_grid: int
    cap_tets: int = 0
    cap_v: int = 0
    cap_va: int = 0
    cap_fw: int = 0
    cap_fa: int = 0
    seq: int = 0
    slot: int = 0                                                   # next free slot of the count ring
    inflight: int = 0                                               # frames launched whose sizes have not been read yet
    last_stream: Any = None                                         # torch stream of the most recent launch on this plan
    workspaces: List[torch.Tensor] = field(default_factory=list)   # one per lane
    workspace_ptrs: List[int] = field(default_factory=list)
    workspace_bytes: int = 0
    workspace_cap_tets: Any = None                                  # (cap_tets, n_edges) the workspaces were sized for
    counts_host: Optional[torch.Tensor] = None                     # pinned, one 128-byte slot per frame of a batch
    counts_np: Optional[np.ndarray] = None                         # (slots, 16) int64 view of counts_host
    counts_ptr: int = 0
    layouts: Dict[Tuple, Any] = field(default_factory=dict)        # (B, lanes, flags) -> _Layout

    def ensure(self, lanes: int, n_edges: int = 0):
        if self.workspace_cap_tets != (self.cap_tets, n_edges):
            need = _cabi.lib().d3h_workspace_bytes_static(self.n_tets, self.n_grid, self.cap_tets, n_edges)
            if need > self.workspace_bytes:
                self.workspaces, self.workspace_ptrs = [], []
                self.workspace_bytes = need
            self.workspace_cap_tets = (self.cap_tets, n_edges)
        while len(self.workspaces) < lanes:
            w = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
            self.workspaces.append(w)
            self.workspace_ptrs.append(w.data_ptr())
        if self.counts_np is None:
            # pinned host memory is device-mapped (UVA): the kernel that finalises the sizes writes them here directly
            self.counts_host = torch.zeros(_COUNT_RING * _CW, dtype=torch.int64).pin_memory()
            self.counts_np = self.counts_host.numpy().reshape(_COUNT_RING, _CW)
            self.counts_ptr = self.counts_host.data_ptr()


_plans: Dict[Tuple, _Plan] = {}


def _plan_for(device: torch.device, n_tets: int, n_grid: int) -> _Plan:
    key = (device.index, n_tets, n_grid)
    p = _plans.get(key)
    if p is None:
        p = _plans[key] = _Plan(device=device, n_tets=n_tets, n_grid=n_grid)
    return p


def reset_plans() -> None:
    """Drop cached workspaces / capacity predictions (tests)."""
    _plans.clear()
    _packed_cache.clear()
    _static_cache.clear()
    from . import single
    single.reset()


@dataclass
class ForwardResult:
    verts_aug: torch.Tensor
    v_tng_aug: torch.Tensor
    msdf_aug: torch.Tensor
    faces_aug: torch.Tensor
    verts_wt: torch.Tensor
    v_tng_wt: torch.Tensor
    msdf_wt: torch.Tensor
    faces_wt: torch.Tensor
    msdf_bnd: torch.Tensor      # extra['msdf_boundary'] = msdf[V:] (gshell_tets.py:397): a second view of the same rows
    n_verts: int
    n_tri: int
    n_quad: int
    counts: Dict[str, int]


@dataclass
class BatchResult:
    frames: List[ForwardResult]
    fslab: torch.Tensor          # float slab of the batch (every float output is a view of it)
    islab: torch.Tensor          # int64 slab (faces)
    tape: torch.Tensor           # int32 slab; frame i: edges (V,2) | corners (P) | slots (P) | runs (V+1)
    tape_off: Tuple[int, int, int, int, int]   # element offsets inside a frame's tape slice + slice length
    launches: int
    bmat: Optional[np.ndarray]   # (B, words) int64 d3h_backward_args[] prefilled for the coming backward pass

    def tape_edges(self, i=0):
        f = self.frames[i]
        o = i * self.tape_off[4]
        return self.tape[o:o + 2 * f.n_verts].view(-1, 2)

    def tape_corners(self, i=0):
        f = self.frames[i]
        o = i * self.tape_off[4] + self.tape_off[1]
        return self.tape[o:o + 3 * f.n_tri + 4 * f.n_quad]


def _r4(n: int) -> int:
    """round a row count up so that the next region of a slab stays 16-byte aligned"""
    return (n + 3) & ~3


_WAIT_TIMEOUT_US = 60_000_000

#: kernels one forward extraction enqueues: prepare, classify, compact, bucket_scan, partition, group_sort, vertex_emit,
#: poly_faces, poly_cut (+ zero_block_kernel with D3H_ZERO_IN_FORWARD=1); backward: the zero-fill (a batch, unless the
#: forward call did it) + adjoint_kernel
LAUNCHES_FORWARD = 9
#: static edge table path: prepare, classify, compact, edge_emit, poly_faces, poly_cut; backward: adjoint_poly + adjoint
LAUNCHES_FORWARD_STATIC = 6
#: edge-scan path: prepare, edge_scan, edge_mark, scan_prefix, scan_emit, poly_faces, poly_cut
LAUNCHES_FORWARD_SCAN = 7


def forward_launches(static, cap_tets: int) -> int:
    """Kernels one forward extraction enqueues on the given path (without the zero-fill of the gradient buffers)."""
    scan = static is not None and len(static) > 6 and static[6] is not None
    if cap_tets <= 0:          # counting run: the surface stages are replaced by publish_counts_kernel
        return 5 if scan else 4
    return LAUNCHES_FORWARD_SCAN if scan else (LAUNCHES_FORWARD_STATIC if static is not None else LAUNCHES_FORWARD)
LAUNCHES_BACKWARD = 1


class _Layout:
    """Everything about a batch that only depends on (B, lanes, capacities, flags): slab geometry, the static words of
    the argument blocks and the per-frame byte offsets of every output / tape pointer (frame i owns slice i of the three
    slabs, so its pointers are slab base + i * stride + constant)."""

    def __init__(self, plan: _Plan, B: int, lanes: int, wt: int, static=None):
        self.key = (B, lanes, wt, plan.cap_v, plan.cap_va, plan.cap_fw, plan.cap_fa, plan.cap_tets, plan.workspace_bytes,
                    plan.counts_ptr, tuple(plan.workspace_ptrs[:lanes]))
        cv, cva, cfw, cfa, ct = plan.cap_v, plan.cap_va, plan.cap_fw, plan.cap_fa, plan.cap_tets
        self.caps = (cv, cva, cfw, cfa, ct)
        o_vaug, o_tng, o_maug = 0, 3 * _r4(cva), 6 * _r4(cva)
        o_vwt = o_maug + _r4(cva)
        o_twt, o_mwt = o_vwt + 3 * _r4(cv), o_vwt + 6 * _r4(cv)
        self.f_off = (o_vaug, o_tng, o_maug, o_vwt, o_twt, o_mwt)
        self.f_len = o_mwt + _r4(cv)
        self.o_vacc = self.f_len                   # static edge table calls: (cap_v, 8) accumulator of the adjoint
        if static is not None:
            self.f_len += 8 * _r4(cv)
        self.i_len = 3 * (cfa + cfw) + (3 * (cfa + cfw)) % 2      # keep every frame's int64 slice 16-byte aligned
        t_corn, t_slot = 2 * _r4(cv), 2 * _r4(cv) + 4 * ct
        t_runs = t_slot + 4 * ct
        self.t_len = _r4(t_runs + cv + 1)
        self.tape_off = (0, t_corn, t_slot, t_runs, self.t_len)
        ar = np.arange(B, dtype=np.int64)
        c = _FC
        A = np.zeros((B, _FW), dtype=np.int64)
        A[:, c["n_grid"]], A[:, c["n_tets"]], A[:, c["tet_begin"]], A[:, c["tet_end"]] = plan.n_grid, plan.n_tets, 0, plan.n_tets
        A[:, c["cap_valid_tets"]], A[:, c["cap_verts"]], A[:, c["cap_verts_aug"]] = ct, cv, cva
        A[:, c["cap_faces_wt"]], A[:, c["cap_faces_aug"]] = cfw, cfa
        A[:, c["workspace"]] = [plan.workspace_ptrs[i % lanes] for i in range(B)]
        A[:, c["workspace_bytes"]] = plan.workspace_bytes
        if static is not None:
            A[:, c["edge_off"]], A[:, c["edge_ab"]], A[:, c["n_edges"]] = static[0].data_ptr(), static[1].data_ptr(), static[2]
            if len(static) > 3 and static[3] is not None:
                A[:, c["tet_edge_rank"]] = static[3].data_ptr()
            if len(static) > 6 and static[6] is not None:
                A[:, c["etet_off"]], A[:, c["etets"]] = static[5].data_ptr(), static[6].data_ptr()
                if static[4] is not None:
                    A[:, c["edge_b"]] = static[4].data_ptr()
                if len(static) > 7 and static[7] is not None:
                    A[:, c["etets8"]] = static[7].data_ptr()
                if len(static) > 9 and static[8] is not None:
                    A[:, c["edge_rows"]], A[:, c["edge_row_off"]] = static[8].data_ptr(), static[9].data_ptr()
                if len(static) > 11 and static[10][0] is not None:
                    er = static[10]
                    A[:, c["edge_runs"]], A[:, c["edge_run_chunk"]], A[:, c["edge_run_ids"]] = (
                        er[0].data_ptr(), er[1].data_ptr(), er[2].data_ptr())
                    A[:, c["n_edge_runs"]] = er[0].shape[0]
                    tr = static[11]
                    if tr[0] is not None:
                        A[:, c["tet_runs"]], A[:, c["tet_run_chunk"]], A[:, c["tet_run_ids"]] = (
                            tr[0].data_ptr(), tr[1].data_ptr(), tr[2].data_ptr())
                        A[:, c["n_tet_runs"]] = tr[0].shape[0]
            self.vacc_off = ar * (4 * self.f_len) + 4 * self.o_vacc
        self.static = static
        self.A = A
        self.ar = ar
        # columns verts_aug .. tape_runs are adjacent: value = base[which slab] + OFF
        self.c0, self.c1 = c["verts_aug"], c["tape_runs"] + 1
        assert self.c1 - self.c0 == 12
        which = {"verts_aug": (0, 4 * o_vaug), "v_tng_aug": (0, 4 * o_tng), "msdf_aug": (0, 4 * o_maug),
                 "faces_aug": (1, 0), "verts_wt": (0, 4 * o_vwt), "v_tng_wt": (0, 4 * o_twt), "msdf_wt": (0, 4 * o_mwt),
                 "faces_wt": (1, 24 * cfa), "tape_edges": (2, 0), "tape_corners": (2, 4 * t_corn),
                 "tape_slots": (2, 4 * t_slot), "tape_runs": (2, 4 * t_runs)}
        stride = (4 * self.f_len, 8 * self.i_len, 4 * self.t_len)
        self.OFF = np.zeros((B, 12), dtype=np.int64)
        self.slab_of = [0] * 12
        for name, (slab, off) in which.items():
            k = c[name] - self.c0
            self.OFF[:, k] = ar * stride[slab] + off
            self.slab_of[k] = slab
        # backward blocks: template with the static words (n_grid; grads_prezeroed = 1 is OR-ed into the flags)
        self.Bt = np.zeros((B, _BW), dtype=np.int64)
        self.Bt[:, _BC["n_grid"]] = plan.n_grid
        bc = _BC
        assert (bc["pos"], bc["sdf"], bc["msdf"]) == (0, 1, 2) and (c["pos"], c["sdf"], c["msdf"]) == (0, 1, 2)
        assert bc["tape_runs"] - bc["tape_edges"] == 3 and bc["n_quad_tets"] - bc["n_verts"] == 2
        assert bc["g_msdf"] - bc["g_pos"] == 2 and c["zero_g_msdf"] - c["zero_g_pos"] == 2
        assert bc["g_msdf_wt"] - bc["g_verts_aug"] == 3


class _Pending:
    """A batch whose forward kernels have been enqueued but whose sizes have not been read yet."""
    __slots__ = ("inputs", "plan", "lay", "fslab", "islab", "tape", "seq0", "slot0", "bmat", "zero_bwd", "launches", "dev",
                 "B")


_unjoined: Dict[Any, bool] = {}   # device index -> a batch was launched without joining the lanes yet

_COUNT_RING = 256   # pinned 128-byte count slots per plan: batches in flight take consecutive slots of the ring


def _launch_frames(ptrs, negate, dev, n_grid: int, tets_i32: torch.Tensor, watertight_template: bool,
                   lanes: int = DEFAULT_LANES, zero=None, grad_ptrs=None, launcher=None, static=None,
                   fused_pair: bool = False) -> _Pending:
    """Enqueue the forward extraction of a batch of frames: ONE library call (d3h_extract_forward_batch), no host wait.

    ptrs   : (B,3) int64 array (or nested list): per frame the device pointers of pos / sdf / msdf -- contiguous fp32
             data, sdf / msdf 16-byte aligned (the caller keeps the tensors alive); negate: per-frame msdf_negate flags
    zero   : (B,3) pointers (0 = none) of the dense gradient buffers to zero-fill for the coming backward pass, each
             buffer under one frame.  With D3H_ZERO_IN_FORWARD=1 this call fills them, otherwise the backward pass
             does (_zero_backward)
    grad_ptrs : (B,3) pointers of the gradient buffers (pos, sdf, msdf); when given, the d3h_backward_args of the batch
             are prefilled here (everything but the upstream gradients and the sizes is known already)
    launcher : replaces the library call (tet-range sharding, sharding.py): launcher(A, plan, stream) enqueues the work
             described by the argument blocks A and may return a Fv to regrow the record capacity to (retry).
    static : (edge_off, edge_ab, n_edges) of build_edge_table, or None for the general per-call sort path.
    fused_pair : the two frames are the cloth / body pair of one iteration (same pos / sdf / msdf, opposite msdf_negate):
             ONE library call classifies and de-duplicates once and replays only the mSDF cut for the second frame
             (d3h_forward_args.pair_*).
    Frames run on `lanes` concurrent lanes inside the library."""
    L = _cabi.lib()
    ptrs = np.asarray(ptrs, dtype=np.int64)
    B = ptrs.shape[0]
    if B > _COUNT_RING // 2:
        raise ValueError(f"at most {_COUNT_RING // 2} frames per batch")
    n_tets = tets_i32.shape[0]
    plan = _plan_for(dev, n_tets, n_grid)
    lanes = max(1, min(int(lanes), MAX_LANES, B))
    cur_stream = torch.cuda.current_stream(dev)
    stream = cur_stream.cuda_stream
    if plan.inflight + B > _COUNT_RING:
        # the pinned count ring has one slot per frame in flight: wrapping it would overwrite sizes nobody has read yet
        raise RuntimeError(f"{plan.inflight} frames are in flight on this grid and {B} more do not fit the count ring of "
                           f"{_COUNT_RING}: call result() / packed() on the earlier futures first")
    if plan.last_stream is not None and plan.last_stream.cuda_stream != stream:
        # workspaces, lanes and the count ring are per grid, not per stream: a launch from another stream is ordered
        # behind the previous user of the plan
        cur_stream.wait_stream(plan.last_stream)
    plan.last_stream = cur_stream
    wt = int(bool(watertight_template))
    flags = np.asarray(negate, dtype=np.int64) | (wt << 32)
    c = _FC
    pend = _Pending()
    if launcher is not None:
        static = None       # the sharded stages exchange records and always sort
    n_edges = static[2] if static is not None else 0
    if fused_pair:
        if B != 2 or launcher is not None or not np.array_equal(ptrs[0], ptrs[1]) or int(negate[0]) == int(negate[1]):
            raise ValueError("a fused pair is two frames on the same pos / sdf / msdf with opposite msdf_negate")
        lanes = 1
    pend.inputs = (ptrs, negate, dev, n_grid, tets_i32, watertight_template, lanes, zero, grad_ptrs, launcher, static,
                   fused_pair)
    pend.plan, pend.dev, pend.B = plan, dev, B
    with torch.cuda.device(dev):
        for attempt in range(6):
            plan.ensure(lanes, n_edges)
            lkey = (B, lanes, wt, static[0].data_ptr() if static is not None else 0)
            lay = plan.layouts.get(lkey)
            if lay is None or lay.key[3:] != (plan.cap_v, plan.cap_va, plan.cap_fw, plan.cap_fa, plan.cap_tets,
                                              plan.workspace_bytes, plan.counts_ptr, tuple(plan.workspace_ptrs[:lanes])):
                if len(plan.layouts) > 32:
                    plan.layouts.clear()
                lay = plan.layouts[lkey] = _Layout(plan, B, lanes, wt, static)
            A = lay.A
            cv, cva, cfw, cfa, ct = lay.caps
            # three slabs for the whole batch: float outputs, int64 faces, int32 tape; frame i owns slice i of each
            fslab = torch.empty(B * lay.f_len, dtype=torch.float32, device=dev)
            islab = torch.empty(B * lay.i_len, dtype=torch.int64, device=dev)
            tape = torch.empty(B * lay.t_len, dtype=torch.int32, device=dev)
            bases = (fslab.data_ptr(), islab.data_ptr(), tape.data_ptr())
            seq0, slot0 = plan.seq, plan.slot
            plan.seq += B
            plan.slot = (plan.slot + B) % _COUNT_RING
            plan.inflight += B
            A[:, 0:3] = ptrs
            A[:, c["tets"]] = tets_ptr = tets_i32.data_ptr()
            A[:, c["msdf_negate"]] = flags
            np.add(lay.OFF, np.array([bases[k] for k in lay.slab_of], dtype=np.int64), out=A[:, lay.c0:lay.c1])
            if static is not None:
                A[:, c["vacc"]] = lay.vacc_off + bases[0]
            launches = B * forward_launches(static, ct)
            if zero is not None and _zero_in_forward():
                A[:, c["zero_g_pos"]:c["zero_g_msdf"] + 1] = zero
                launches += int(np.count_nonzero(np.asarray(zero).any(axis=1)))
            else:
                A[:, c["zero_g_pos"]:c["zero_g_msdf"] + 1] = 0
            A[:, c["counts_host"]] = plan.counts_ptr + ((slot0 + lay.ar) % _COUNT_RING) * 128
            A[:, c["seq"]] = lay.ar + (seq0 + 1)
            A[:, c["pair_verts_aug"]:c["pair_seq"] + 1] = 0
            if fused_pair:
                # frame 1 is produced by the call of frame 0: its outputs, accumulator, count slot and tag ride along
                for dst, src in (("pair_verts_aug", "verts_aug"), ("pair_v_tng_aug", "v_tng_aug"), ("pair_msdf_aug", "msdf_aug"),
                                 ("pair_faces_aug", "faces_aug"), ("pair_verts_wt", "verts_wt"), ("pair_v_tng_wt", "v_tng_wt"),
                                 ("pair_msdf_wt", "msdf_wt"), ("pair_faces_wt", "faces_wt"), ("pair_vacc", "vacc"),
                                 ("pair_counts_host", "counts_host"), ("pair_seq", "seq")):
                    A[0, c[dst]] = A[1, c[src]]
                if zero is not None and _zero_in_forward():   # one call: every zero-fill duty moves to frame 0
                    z = np.asarray(zero, dtype=np.int64)
                    A[0, c["zero_g_pos"]:c["zero_g_msdf"] + 1] = z[0] | z[1]
                    A[1, c["zero_g_pos"]:c["zero_g_msdf"] + 1] = 0
            if (B == 1 or fused_pair) and _unjoined.get(dev.index):
                # this call runs on the caller's stream and shares workspace 0 with the lanes of an un-joined batch
                _cabi.check(L.d3h_lanes_join(stream), "d3h_lanes_join")
                _unjoined[dev.index] = False
            if fused_pair:
                _cabi.check(L.d3h_extract_forward_batch(A.ctypes.data, 1, 1, stream), "d3h_extract_forward (pair)")
                launches += 3         # pair_vertex + replayed poly_faces / poly_cut; frame 1 launches nothing else
                launches -= forward_launches(static, ct)
            elif launcher is None:
                # no join here: the lanes keep running and the next batch may queue up behind this one lane by lane;
                # _collect_frames orders the caller's stream behind the lanes before any output is handed out
                _cabi.check(L.d3h_extract_forward_batch_nojoin(A.ctypes.data, B, lanes, stream),
                            "d3h_extract_forward_batch")
                if B > 1:
                    _unjoined[dev.index] = True
            else:
                need_tets = launcher(A, plan, stream)
                if need_tets is not None:   # the gathered records do not fit: grow like an overflowed single call
                    plan.inflight -= B
                    plan.cap_tets = _grow(int(need_tets))
                    p4 = 4 * plan.cap_tets
                    plan.cap_v, plan.cap_va = max(cv, p4), max(cva, 2 * p4)
                    plan.cap_fw, plan.cap_fa = max(cfw, 2 * plan.cap_tets), max(cfa, 4 * plan.cap_tets)
                    continue
            break
        else:  # pragma: no cover
            raise RuntimeError("tet-range sharding: record capacity did not converge")
        # the GPU is busy now: prefill the backward blocks of the batch
        bmat = None
        if grad_ptrs is not None:
            b = _BC
            bmat = lay.Bt.copy()
            bmat[:, 0:3] = ptrs
            bmat[:, b["msdf_negate"]] = np.asarray(negate, dtype=np.int64) | (1 << 32)    # grads_prezeroed = 1
            bmat[:, b["tape_edges"]:b["tape_runs"] + 1] = A[:, c["tape_edges"]:c["tape_runs"] + 1]
            bmat[:, b["verts_wt"]], bmat[:, b["msdf_wt"]] = A[:, c["verts_wt"]], A[:, c["msdf_wt"]]
            bmat[:, b["g_pos"]:b["g_msdf"] + 1] = grad_ptrs
            if fused_pair:           # one tape for both frames: the one frame 0's call writes
                bmat[1, b["tape_edges"]:b["tape_runs"] + 1] = bmat[0, b["tape_edges"]:b["tape_runs"] + 1]
            if static is not None:   # scatter-form adjoint: no per-vertex corner lists on the tape
                bmat[:, b["tape_slots"]] = bmat[:, b["tape_runs"]] = 0
                bmat[:, b["vacc"]] = A[:, c["vacc"]]
    pend.lay, pend.fslab, pend.islab, pend.tape = lay, fslab, islab, tape
    pend.seq0, pend.slot0, pend.bmat, pend.launches = seq0, slot0, bmat, launches
    pend.zero_bwd = zero is not None and bmat is not None and not _zero_in_forward()
    return pend


def _collect_frames(pend: _Pending) -> BatchResult:
    """Host side of a launched batch: blocks once per frame on that frame's sizes (written to pinned host memory by the
    kernel that finalises them; the reference blocks ~40 times per frame) and builds the frame's output views while the
    GPU is still working on the later frames.  A capacity overflow re-launches the batch with the sizes just learnt."""
    L = _cabi.lib()
    wait = L.d3h_wait_counts
    ast = torch.as_strided
    launches = 0
    for attempt in range(6):
        plan, lay, B = pend.plan, pend.lay, pend.B
        fslab, islab = pend.fslab, pend.islab
        cv, cva, cfw, cfa, ct = lay.caps
        o_vaug, o_tng, o_maug, o_vwt, o_twt, o_mwt = lay.f_off
        f_len, i_len = lay.f_len, lay.i_len
        counts_base, seq0, slot0 = plan.counts_ptr, pend.seq0, pend.slot0
        launches += pend.launches
        sizes = np.empty((B, 6), dtype=np.int64)   # fv, t1, t2, p, v, fa
        frames: List[ForwardResult] = []
        grow_tets = grow_out = False
        cn = plan.counts_np
        for i in range(B):
            slot = (slot0 + i) % _COUNT_RING
            rc = wait(counts_base + slot * 128, seq0 + 1 + i, _WAIT_TIMEOUT_US)
            if rc:
                _cabi.check(rc, "d3h_wait_counts")
            row = cn[slot].tolist()
            fv, t1, t2, p, v, nfa = row[0:6]
            sizes[i] = row[0:6]
            if fv > ct:
                grow_tets = True
            elif v > cv or v + p > cva or t1 + 2 * t2 > cfw or nfa > cfa:
                grow_out = True
            if grow_tets or grow_out:
                continue  # this attempt is void; keep reading the sizes of the other frames for the regrowth
            # views of frame i, built while the GPU works on the later frames
            va, fw = v + p, t1 + 2 * t2
            fo, io = i * f_len, i * i_len
            frames.append(ForwardResult(
                ast(fslab, (va, 3), (3, 1), fo + o_vaug), ast(fslab, (va, 3), (3, 1), fo + o_tng),
                ast(fslab, (va,), (1,), fo + o_maug), ast(islab, (nfa, 3), (3, 1), io),
                ast(fslab, (v, 3), (3, 1), fo + o_vwt), ast(fslab, (v, 3), (3, 1), fo + o_twt),
                ast(fslab, (v,), (1,), fo + o_mwt), ast(islab, (fw, 3), (3, 1), io + 3 * cfa),
                ast(fslab, (p,), (1,), fo + o_maug + v), v, t1, t2,
                dict(n_valid_tets=fv, n_tri_tets=t1, n_quad_tets=t2, n_corners=p, n_verts=v, n_verts_aug=va,
                     n_faces_watertight=fw, n_faces_aug=nfa, bucket_polys=tuple(row[6:12]))))
        plan.inflight -= B        # every size of this attempt has been read
        if B == 1:
            fw_, va_ = t1 + 2 * t2, v + p
        else:
            mx = sizes.max(axis=0).tolist()
            fv, t1, t2, v, nfa = mx[0], mx[1], mx[2], mx[4], mx[5]
            va_ = int((sizes[:, 4] + sizes[:, 3]).max())
            fw_ = int((sizes[:, 1] + 2 * sizes[:, 2]).max())
        if B > 1 and not pend.inputs[11]:     # (a fused pair runs on the caller's stream: nothing to join)
            _cabi.check(L.d3h_lanes_join(torch.cuda.current_stream(pend.dev).cuda_stream), "d3h_lanes_join")
            _unjoined[pend.dev.index] = False
        if grow_tets or grow_out:
            if grow_tets:  # record buffer too small: surface stages were skipped for some frame, its sizes are unknown
                p = 3 * t1 + 4 * t2
                plan.cap_tets = max(plan.cap_tets, _grow(fv))
                # upper bounds that cannot overflow, so the next attempt is final
                plan.cap_v, plan.cap_va = max(plan.cap_v, p), max(plan.cap_va, 2 * p)
                plan.cap_fw, plan.cap_fa = max(plan.cap_fw, t1 + 2 * t2), max(plan.cap_fa, 2 * t1 + 4 * t2)
            else:
                plan.cap_v, plan.cap_va = max(plan.cap_v, _grow(v)), max(plan.cap_va, _grow(va_))
                plan.cap_fw, plan.cap_fa = max(plan.cap_fw, _grow(fw_)), max(plan.cap_fa, _grow(nfa))
            pend = _launch_frames(*pend.inputs)
            continue
        break
    else:  # pragma: no cover
        raise RuntimeError("d3h_extract_forward_batch: capacities did not converge")
    # next call: predict from this call's sizes (the surface moves slowly between training iterations)
    plan.cap_tets = max(_grow(fv), min(plan.cap_tets, 2 * _grow(fv)))
    plan.cap_v, plan.cap_va = _shrink(plan.cap_v, v), _shrink(plan.cap_va, va_)
    plan.cap_fw, plan.cap_fa = _shrink(plan.cap_fw, fw_), _shrink(plan.cap_fa, nfa)
    bmat = pend.bmat
    if bmat is not None:
        bmat[:, _BC["n_verts"]:_BC["n_quad_tets"] + 1] = sizes[:, (4, 1, 2)]
    res = BatchResult(frames, fslab, islab, pend.tape, lay.tape_off, launches, bmat)
    res.zero_bwd = pend.zero_bwd
    res.geom = (cv, cfa, i_len)      # cap_v, cap_fa, int64 words per frame of the index slab (tangent branch of the backward)
    return res


def _collect_packed(pend: _Pending):
    """_collect_frames without the per-frame views: waits for the sizes of every frame (one library call each), checks
    the capacities of the whole batch with a few numpy operations, regrows and re-launches on overflow.
    -> (pend, sizes (B,6) int64 [fv, t1, t2, p, v, fa], launches)"""
    L = _cabi.lib()
    wait = L.d3h_wait_counts
    launches = 0
    for attempt in range(6):
        plan, lay, B = pend.plan, pend.lay, pend.B
        cv, cva, cfw, cfa, ct = lay.caps
        launches += pend.launches
        base, seq0, slot0 = plan.counts_ptr, pend.seq0, pend.slot0
        for i in range(B):
            rc = wait(base + ((slot0 + i) % _COUNT_RING) * 128, seq0 + 1 + i, _WAIT_TIMEOUT_US)
            if rc:
                _cabi.check(rc, "d3h_wait_counts")
        sizes = plan.counts_np[(slot0 + lay.ar) % _COUNT_RING, 0:6].copy()
        plan.inflight -= B
        if B > 1 and not pend.inputs[11]:
            _cabi.check(L.d3h_lanes_join(torch.cuda.current_stream(pend.dev).cuda_stream), "d3h_lanes_join")
            _unjoined[pend.dev.index] = False
        fv, t1, t2, p, v, nfa = (int(x) for x in sizes.max(axis=0))
        va_ = int((sizes[:, 4] + sizes[:, 3]).max())
        fw_ = int((sizes[:, 1] + 2 * sizes[:, 2]).max())
        if fv > ct:   # record buffer too small: surface stages were skipped for some frame, its sizes are unknown
            pc = 3 * t1 + 4 * t2
            plan.cap_tets = max(plan.cap_tets, _grow(fv))
            plan.cap_v, plan.cap_va = max(plan.cap_v, pc), max(plan.cap_va, 2 * pc)
            plan.cap_fw, plan.cap_fa = max(plan.cap_fw, t1 + 2 * t2), max(plan.cap_fa, 2 * t1 + 4 * t2)
        elif v > cv or va_ > cva or fw_ > cfw or nfa > cfa:
            plan.cap_v, plan.cap_va = max(plan.cap_v, _grow(v)), max(plan.cap_va, _grow(va_))
            plan.cap_fw, plan.cap_fa = max(plan.cap_fw, _grow(fw_)), max(plan.cap_fa, _grow(nfa))
        else:
            break
        pend = _launch_frames(*pend.inputs)
    else:  # pragma: no cover
        raise RuntimeError("d3h_extract_forward_batch: capacities did not converge")
    plan.cap_tets = max(_grow(fv), min(plan.cap_tets, 2 * _grow(fv)))
    plan.cap_v, plan.cap_va = _shrink(plan.cap_v, v), _shrink(plan.cap_va, va_)
    plan.cap_fw, plan.cap_fa = _shrink(plan.cap_fw, fw_), _shrink(plan.cap_fa, nfa)
    if pend.bmat is not None:
        pend.bmat[:, _BC["n_verts"]:_BC["n_quad_tets"] + 1] = sizes[:, (4, 1, 2)]
    return pend, sizes, launches


def forward_frames_raw(ptrs, negate, dev, n_grid: int, tets_i32: torch.Tensor, watertight_template: bool,
                       lanes: int = DEFAULT_LANES, zero=None, grad_ptrs=None, launcher=None, static=None,
                       fused_pair: bool = False) -> BatchResult:
    """Launch + collect (see _launch_frames / _collect_frames)."""
    return _collect_frames(_launch_frames(ptrs, negate, dev, n_grid, tets_i32, watertight_template, lanes, zero,
                                          grad_ptrs, launcher, static, fused_pair))


def forward_raw(pos, sdf, msdf, tets_i32, msdf_negate, watertight_template, static=None) -> BatchResult:
    """One forward extraction without autograd (tests, profiling scripts)."""
    return forward_frames_raw([[pos.data_ptr(), sdf.data_ptr(), msdf.data_ptr()]], [int(bool(msdf_negate))],
                              pos.device, pos.shape[0], tets_i32, watertight_template, lanes=1, static=static)


def _shrink(cap: int, need: int) -> int:
    g = _grow(need)
    return g if (cap < g or cap > 2 * g) else cap


# --------------------------------------------------------------------------------------------------
# autograd
# --------------------------------------------------------------------------------------------------
_OUTS_PER_FRAME = 9   # verts_aug, v_tng_aug, msdf_aug, verts_wt, v_tng_wt, msdf_wt, msdf_boundary, faces_aug, faces_wt


_ref_cache: Dict[Tuple, Tuple] = {}


def _ref_arrays(refs, need):
    """Index pattern of a batch as numpy arrays, cached on (refs, need): the same calling pattern repeats every step.
    -> IDX (B,3) tensor index of pos / sdf / msdf per frame, ROW (B,3) row inside a stacked tensor (0: whole tensor),
       NEG (B,) msdf_negate flags, GMASK (B,3) the frame accumulates into the gradient of that tensor, ZMASK (B,3) ... and
       is the one that zero-fills it, USED (n_tensors,) tensors that need a gradient buffer."""
    key = (refs, need)
    hit = _ref_cache.get(key)
    if hit is not None:
        return hit
    B = len(refs)
    idx = np.array([[r[k][0] for k in range(3)] for r in refs], dtype=np.int64).reshape(B, 3)
    row = np.array([[max(r[k][1], 0) for k in range(3)] for r in refs], dtype=np.int64).reshape(B, 3)
    neg = np.array([int(r[3]) for r in refs], dtype=np.int64)
    gmask = np.zeros((B, 3), dtype=bool)
    zmask = np.zeros((B, 3), dtype=bool)
    used = np.zeros(len(need), dtype=bool)
    if any(need):
        zeroed = set()
        for i, r in enumerate(refs):
            for k in range(3):
                t, rw = r[k]
                if k == 2 and not (need[t] and not r[3]):   # "body" frames do not reach msdf (hmsdf_tets_split.py:256-264)
                    continue
                gmask[i, k] = True
                used[t] = True
                if (t, rw) not in zeroed:
                    zeroed.add((t, rw))
                    zmask[i, k] = True
    if len(_ref_cache) > 64:
        _ref_cache.clear()
    out = _ref_cache[key] = (idx, row, neg, gmask, zmask, used)
    return out


def _zero_in_forward() -> bool:
    """D3H_ZERO_IN_FORWARD=1: the forward call zero-fills the dense gradient buffers (next to its surface kernels)
    instead of the backward call.  The default is the backward call: the forward rounds of a training step are its
    critical path, while the GPU waits for the host around the backward call; the switch keeps both placements
    measurable."""
    return os.environ.get("D3H_ZERO_IN_FORWARD") == "1"


def _zero_backward(bmat, stream) -> None:
    """Zero-fills the gradient buffers of a batch ahead of its adjoints: ONE d3h_extract_backward_batch call with the
    batch's blocks, grads_prezeroed = 0 and no upstream gradients -- the library launches its zero-fill (every buffer
    once, however many frames share it) and no adjoint.  The adjoint call that follows passes grads_prezeroed = 1, so a
    buffer the frames share is never zeroed between two frames' contributions."""
    z = bmat.copy()
    b = _BC
    z[:, b["g_verts_aug"]:b["g_msdf_wt"] + 1] = 0
    z[:, b["g_msdf_boundary"]] = z[:, b["g_verts_tng"]] = z[:, b["g_mvert_tng"]] = 0
    z[:, b["grads_prezeroed"]] &= 0xFFFFFFFF          # grads_prezeroed = 0 (the high half of the word)
    _cabi.check(_cabi.lib().d3h_extract_backward_batch(z.ctypes.data, z.shape[0], 1, stream), "d3h_extract_backward_batch")
    _ExtractFn.total_launches += 1


def _prelaunch(refs, tensors, need, tets_i32, watertight_template, lanes, launcher=None, static=None, fused_pair=False):
    """Everything of a forward call that precedes the size read: pointer tables of the frames, dense gradient buffers
    (allocated here, uninitialised: the backward call zero-fills them before its adjoints -- or, with
    D3H_ZERO_IN_FORWARD=1, the forward call of the frame that owns them), and the launch.
    Returns (pending batch, gradient buffers or None, N)."""
    need = tuple(bool(x) for x in need)
    idx, row, neg, gmask, zmask, used = _ref_arrays(refs, need)
    n_grid = tensors[refs[0][0][0]].shape[-2]
    row_bytes = np.array([12 * n_grid, 4 * n_grid, 4 * n_grid], dtype=np.int64)
    off = row * row_bytes
    base = np.array([t.data_ptr() for t in tensors], dtype=np.int64)
    ptrs = base[idx] + off
    zero = grad_ptrs = gbufs = None
    if used.any():
        gbufs = [torch.empty_like(t) if u else None for t, u in zip(tensors, used)]
        gbase = np.array([g.data_ptr() if g is not None else 0 for g in gbufs], dtype=np.int64)
        grad_ptrs = np.where(gmask, gbase[idx] + off, 0)
        zero = np.where(zmask, grad_ptrs, 0)
    pend = _launch_frames(ptrs, neg, tensors[0].device, n_grid, tets_i32, watertight_template, lanes, zero, grad_ptrs,
                          launcher, static, fused_pair)
    return pend, gbufs, n_grid


class _ExtractFn(torch.autograd.Function):
    """A batch of frames as ONE autograd node.

    forward : (spec, tets_i32, *input tensors) -> 8 tensors per frame (6 float + 2 index outputs)
    backward: dense gradients for every input tensor that needs one; a tensor shared by several frames (sdf / msdf of a
              batch of video frames, everything but msdf for the cloth / body pair) receives the sum over the frames.

    spec = (frame refs, watertight_template, lanes); a frame ref is (pos, sdf, msdf, negate) where each of pos / sdf /
    msdf is (input index, row): row >= 0 selects one row of a stacked (B,N,3) / (B,N) input, row < 0 the whole tensor.

    Differentiable outputs: verts_aug, msdf (augmented, stop-grad coefficients), vertices_watertight, msdf_watertight, and
    -- through the optional tangent branch (tangent_branch / d3h_tangent_backward; the reference's own training never
    consumes them, hmsdf.py:454,548) -- v_tng_aug and v_tng_watertight.
    """

    @staticmethod
    def forward(ctx, spec, tets_i32, *tensors):
        refs, watertight_template, lanes = spec[:3]
        launcher = spec[3] if len(spec) > 3 else None     # tet-range sharding (sharding.py)
        started = spec[4] if len(spec) > 4 else None      # extract_frames_async: the batch is already in flight
        if started is None:
            static = None if launcher is not None else static_edges_for(tets_i32, tensors[refs[0][0][0]].shape[-2])
            started = _prelaunch(refs, tensors, ctx.needs_input_grad[2:], tets_i32, watertight_template, lanes, launcher,
                                 static)
        pend, gbufs, n_grid = started
        res = _collect_frames(pend)
        ctx.save_for_backward(*tensors, res.tape, res.fslab)   # the slabs hold the tape and verts_wt / msdf_wt of all frames
        ctx.islab = res.islab                                  # faces_watertight: only read by the tangent branch of the backward pass
        ctx.bmat, ctx.zero_bwd = res.bmat, res.zero_bwd
        ctx.meta = (refs, tets_i32.shape[0], n_grid, [(f.n_verts, f.n_tri, f.n_quad) for f in res.frames], lanes)
        ctx.caps = res.geom
        ctx.gbufs = gbufs
        ctx.set_materialize_grads(False)
        flat = []
        nondiff = []
        for r in res.frames:
            flat += [r.verts_aug, r.v_tng_aug, r.msdf_aug, r.verts_wt, r.v_tng_wt, r.msdf_wt, r.msdf_bnd, r.faces_aug,
                     r.faces_wt]
            nondiff += [r.faces_aug, r.faces_wt]
        ctx.mark_non_differentiable(*nondiff)
        _ExtractFn.last_counts = [r.counts for r in res.frames]
        _ExtractFn.last_launches = res.launches
        _ExtractFn.last_tape = (res.tape, res.tape_off[4], [f.n_verts for f in res.frames])
        _ExtractFn.total_launches += res.launches
        return tuple(flat)

    @staticmethod
    def backward(ctx, *grads):
        refs, n_tets, n_grid, sizes, lanes = ctx.meta
        tensors = ctx.saved_tensors[:-2]
        need = ctx.needs_input_grad[2:]
        gbufs, ctx.gbufs = ctx.gbufs, None       # the forward call's buffers serve ONE backward pass
        bmat = ctx.bmat
        if bmat is None:
            raise RuntimeError("backward through an extraction whose inputs did not require gradients")
        L = _cabi.lib()
        dev = tensors[0].device
        with torch.cuda.device(dev):
            if gbufs is None:  # second backward through the same node (retain_graph): fresh zero-filled buffers
                gbufs = [None] * len(tensors)
                bmat = bmat.copy()
                row_bytes = (12 * n_grid, 4 * n_grid, 4 * n_grid)
                names = ("g_pos", "g_sdf", "g_msdf")
                for i, r in enumerate(refs):
                    for k in range(3):
                        idx, row = r[k]
                        if bmat[i, _BC[names[k]]] == 0:
                            continue
                        if gbufs[idx] is None:
                            gbufs[idx] = torch.zeros_like(tensors[idx])
                        bmat[i, _BC[names[k]]] = gbufs[idx].data_ptr() + (row * row_bytes[k] if row > 0 else 0)
            elif ctx.zero_bwd:
                _zero_backward(bmat, torch.cuda.current_stream(dev).cuda_stream)
            keep = []
            live = []
            tng = []  # frames with upstream tangent gradients: (frame, g_verts, g_mvert, kept tensors)
            cap_v, cap_fa, i_len = ctx.caps
            gp = []   # per live frame: pointers of g_verts_aug, g_msdf_aug, g_verts_wt, g_msdf_wt (adjacent columns)
            gb = []   # ... and of the gradient of the msdf_boundary view
            f32 = torch.float32
            for i in range(len(refs)):
                o = _OUTS_PER_FRAME * i
                g0, g1, g2, g3, g4, g5, g6 = grads[o:o + 7]
                if g0 is None and g1 is None and g2 is None and g3 is None and g4 is None and g5 is None and g6 is None:
                    continue  # nothing flows into this frame
                n_verts, n_tri, n_quad = sizes[i]
                if g1 is not None or g4 is not None:
                    # optional branch (SURVEY A.5): through the tangents -> extra per-vertex gradients for the adjoint
                    tng.append((i,) + tangent_branch(
                        dev, n_tets, int(bmat[i, _BC["verts_wt"]]), int(bmat[i, _BC["msdf_wt"]]),
                        int(bmat[i, _BC["verts_wt"]]) + 12 * _r4(cap_v), ctx.islab.data_ptr() + 8 * (i * i_len + 3 * cap_fa),
                        int(bmat[i, _BC["tape_corners"]]), n_verts, n_tri, n_quad, g1, g4))
                va = n_verts + 3 * n_tri + 4 * n_quad
                row = []
                for t, rows in ((g0, va), (g2, va), (g3, n_verts), (g5, n_verts), (g6, va - n_verts)):
                    if t is None:
                        row.append(0)
                        continue
                    if t.dtype is not f32 or not t.is_contiguous():
                        t = t.contiguous().float()
                        keep.append(t)
                    assert t.shape[0] == rows, (tuple(t.shape), rows)
                    row.append(t.data_ptr())
                gb.append(row.pop())
                gp.append(row)
                live.append(i)
            if live:
                bmat[:, _BC["g_verts_tng"]] = 0
                bmat[:, _BC["g_mvert_tng"]] = 0
                for i, gvt, gmt, _k in tng:
                    bmat[i, _BC["g_verts_tng"]], bmat[i, _BC["g_mvert_tng"]] = gvt.data_ptr(), gmt.data_ptr()
                m = bmat if len(live) == len(refs) else np.ascontiguousarray(bmat[live])
                m[:, _BC["g_verts_aug"]:_BC["g_msdf_wt"] + 1] = gp
                m[:, _BC["g_msdf_boundary"]] = gb
                # adjoint_kernel (+ adjoint_poly_kernel on the static edge table path) per 16 frames
                per16 = 2 if int(m[0, _BC["tape_slots"]]) == 0 else 1
                _ExtractFn.total_launches += per16 * ((len(live) + 15) // 16)
                _cabi.check(L.d3h_extract_backward_batch(m.ctypes.data, len(live), max(1, min(lanes, len(live))),
                                                         torch.cuda.current_stream(dev).cuda_stream),
                            "d3h_extract_backward_batch")
        return (None, None) + tuple(gbufs[i] if need[i] else None for i in range(len(tensors)))


_ExtractFn.last_counts = None
_ExtractFn.last_launches = 0
_ExtractFn.last_tape = None       # (tape slab, slice length, V per frame) of the most recent batch
_ExtractFn.total_launches = 0      # kernels enqueued by this module since import (forward + backward)


def launch_counter() -> int:
    """Number of library kernels enqueued so far by this process (bench.py reports the difference over its timed region)."""
    return _ExtractFn.total_launches


def _counts_list():
    c = _ExtractFn.last_counts
    if isinstance(c, tuple):     # the single-call path leaves the raw sizes: (Fv, T1, T2, P, V, Va, Fw, Fa, buckets)
        fv, t1, t2, p, v, va, fw, nfa, buckets = c
        c = _ExtractFn.last_counts = [dict(n_valid_tets=fv, n_tri_tets=t1, n_quad_tets=t2, n_corners=p, n_verts=v,
                                           n_verts_aug=va, n_faces_watertight=fw, n_faces_aug=nfa, bucket_polys=buckets)]
    return c


def last_counts() -> Optional[Dict[str, int]]:
    """Sizes of the most recent extraction (Fv, T1, T2, P, V, Va, Fw, Fa, bucket sizes); frame 0 of a batch."""
    c = _counts_list()
    return c[0] if c else None


def last_counts_frames() -> Optional[List[Dict[str, int]]]:
    return _counts_list()


def _aligned(t: torch.Tensor) -> torch.Tensor:
    """Contiguous and 16-byte aligned (the kernels use 16-byte vector loads); a view at an odd offset is cloned."""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _check_cuda(t):
    if not t.is_cuda:
        raise RuntimeError("d3human-code_b200 has no CPU path: inputs must live on a CUDA device "
                           "(the reference hard-codes device='cuda' as well, gshell_tets.py:108)")


def _prep_pos(pos_nx3):
    _check_cuda(pos_nx3)
    if pos_nx3.dim() != 2 or pos_nx3.shape[1] != 3:
        raise ValueError(f"pos_nx3 must have shape (N,3), got {tuple(pos_nx3.shape)}")
    return _aligned(pos_nx3.float())


def _prep_field(f, n_grid):
    f = f.float().reshape(-1)       # gshell_tets.py:254 (.float()); (N,1) from the SDF MLP or (N,)
    if f.shape[0] != n_grid:
        raise ValueError("sdf_n / msdf_n must have one value per grid vertex")
    return _aligned(f)


def _pack_result(r8, output_watertight_template):
    verts_aug, v_tng_aug, msdf_aug, verts_wt, v_tng_wt, msdf_wt, msdf_bnd, faces_aug, faces_wt = r8
    n_wt = verts_wt.shape[0]
    if output_watertight_template:  # gshell_tets.py:430-439
        extra = {
            "n_verts_watertight": n_wt,
            "vertices_watertight": verts_wt,
            "faces_watertight": faces_wt,
            "v_tng_watertight": v_tng_wt,
            "msdf": msdf_aug,
            "msdf_watertight": msdf_wt,
            "msdf_boundary": msdf_bnd,
        }
    else:  # gshell_tets.py:440-445
        extra = {"msdf": msdf_aug, "msdf_watertight": msdf_wt, "msdf_boundary": msdf_bnd}
    return verts_aug, faces_aug, None, None, v_tng_aug, extra


def extract(pos_nx3, sdf_n, msdf_n, tet_fx4, msdf_negate: bool = False, output_watertight_template: bool = True):
    """Shared body of GShell_Tets.__call__ / hmSDF_Tets.__call__: returns the reference's 6-tuple.  One frame: the lean
    host path of single.py (same kernels, same plan)."""
    from . import single
    return single.extract(pos_nx3, sdf_n, msdf_n, tet_fx4, msdf_negate, output_watertight_template)


def extract_generic(pos_nx3, sdf_n, msdf_n, tet_fx4, msdf_negate: bool = False, output_watertight_template: bool = True):
    """The same through the batch machinery with B = 1 (kept for A/B timing and as a cross-check in the tests)."""
    pos = _prep_pos(pos_nx3)
    n_grid = pos.shape[0]
    sdf, msdf = _prep_field(sdf_n, n_grid), _prep_field(msdf_n, n_grid)
    tets = packed_tets(tet_fx4, n_grid)
    spec = ((((0, -1), (1, -1), (2, -1), bool(msdf_negate)),), bool(output_watertight_template), 1)
    return _pack_result(_ExtractFn.apply(spec, tets, pos, sdf, msdf), output_watertight_template)


def tangent_branch(dev, n_tets, verts_wt_ptr, msdf_wt_ptr, v_tng_wt_ptr, faces_wt_ptr, corners_ptr, v, t1, t2, g_aug, g_wt):
    """Backward pass through the tangents (d3h_tangent_backward; SURVEY A.5 optional branch): upstream gradients of
    v_tng_aug (Va,3) / extra['v_tng_watertight'] (V,3) -> (g_verts (V,3), g_mvert (V)) for d3h_backward_args.g_*_tng."""
    f32 = torch.float32
    keep = []

    def ptr(t, rows):
        if t is None:
            return 0
        if t.dtype is not f32 or not t.is_contiguous():
            t = t.contiguous().float()
        keep.append(t)
        assert t.shape[0] == rows, (tuple(t.shape), rows)
        return t.data_ptr()

    g_verts = torch.empty((v, 3), dtype=f32, device=dev)
    g_mvert = torch.empty((v,), dtype=f32, device=dev)
    ws = torch.empty(16 * max(v, 1), dtype=f32, device=dev)
    a = _cabi.TangentBackwardArgs()
    a.verts_wt, a.msdf_wt, a.v_tng_wt, a.faces_wt, a.tape_corners = verts_wt_ptr, msdf_wt_ptr, v_tng_wt_ptr, faces_wt_ptr, corners_ptr
    a.n_verts, a.n_tri_tets, a.n_quad_tets, a.n_tets = v, t1, t2, n_tets
    a.g_tng_aug, a.g_tng_wt = ptr(g_aug, v + 3 * t1 + 4 * t2), ptr(g_wt, v)
    a.g_verts, a.g_mvert = g_verts.data_ptr(), g_mvert.data_ptr()
    a.workspace, a.workspace_bytes = ws.data_ptr(), 64 * v
    with torch.cuda.device(dev):
        rc = _cabi.lib().d3h_tangent_backward(C.addressof(a), torch.cuda.current_stream(dev).cuda_stream)
    if rc:
        msg = _cabi.lib().d3h_last_error_string().decode("utf-8", "replace")
        if "three faces" in msg:
            raise NotImplementedError(msg)
        _cabi.check(rc, "d3h_tangent_backward")
    _ExtractFn.total_launches += 4
    return g_verts, g_mvert, (keep, ws)


def _tape_edges(tape3, i: int) -> torch.Tensor:
    tape, t_len, nv = tape3
    o = i * t_len
    return tape[o:o + 2 * int(nv[i])].view(-1, 2)


class _MappedAlias:
    """__cuda_array_interface__ of a pinned host tensor (its device alias under unified addressing)."""

    def __init__(self, t: torch.Tensor):
        self.__cuda_array_interface__ = {"shape": tuple(t.shape), "typestr": "<f4", "version": 2, "strides": None,
                                         "data": (t.data_ptr(), False)}
        self.keep = t


def mapped_view(host: torch.Tensor, device=None) -> torch.Tensor:
    """A CUDA tensor that ALIASES a pinned host tensor (float32, contiguous): pinned allocations are device-mapped at the
    same address, so kernels can read them in place over PCIe.  Meant for the per-frame grid positions `pos` of a caller
    that keeps them in host memory: an extraction reads only the rows of crossing-edge end points (~2 V of N rows, forward
    and backward), so handing the mapped view to GShell_Tets / extract_frames moves ~1 MB per frame instead of copying the
    26 MB of (N,3) positions first.  The view shares the host tensor's memory: keep it alive and do not write to it
    while a call is in flight.  Gradients w.r.t. such a `pos` are ordinary device tensors."""
    if host.is_cuda:
        return host
    if host.dtype is not torch.float32 or not host.is_contiguous() or not host.is_pinned():
        raise ValueError("mapped_view: needs a pinned, contiguous float32 host tensor")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    out = torch.as_tensor(_MappedAlias(host), device=dev)
    _mapped_keepalive[out.data_ptr()] = host          # (the alias does not own the memory)
    if len(_mapped_keepalive) > 64:
        for k in list(_mapped_keepalive)[:-32]:
            del _mapped_keepalive[k]
    return out


_mapped_keepalive: Dict[int, torch.Tensor] = {}


def gather_touched(grad: torch.Tensor, edges: torch.Tensor) -> torch.Tensor:
    """Compact form of a dense per-grid-vertex gradient of ONE frame: the rows an extraction can have touched are the end
    points of its crossing edges (`edges` = FramesFuture.tape_edges(i), (V,2) int32).  Returns grad[edges.reshape(-1)] as a
    (2V, width) tensor (library kernel d3h_gather_rows); dense[edges.reshape(-1)] = rows restores the dense gradient
    (every other row is zero; repeated ids carry identical rows).  ~2V rows instead of N: what a host-side consumer copies
    back instead of a (N,3) buffer that is > 99 % zeros."""
    g = grad.reshape(grad.shape[0], -1) if grad.dim() > 1 else grad.reshape(-1, 1)
    if g.dtype is not torch.float32 or not g.is_contiguous():
        g = g.float().contiguous()
    ids = edges.reshape(-1)
    out = torch.empty((ids.shape[0], g.shape[1]), dtype=torch.float32, device=g.device)
    with torch.cuda.device(g.device):
        _cabi.check(_cabi.lib().d3h_gather_rows(ids.data_ptr(), ids.shape[0], g.data_ptr(), g.shape[0], g.shape[1],
                                                out.data_ptr(), torch.cuda.current_stream(g.device).cuda_stream),
                    "d3h_gather_rows")
    _ExtractFn.total_launches += 1 if ids.shape[0] else 0
    return out


class PackedFrames:
    """The B frames of a batch as PADDED tensors: frame i owns slice i, rows [0, n_i) of it are valid, the rest is
    uninitialised.  What a batched consumer wants anyway (nvdiffrast's range mode takes exactly this: one vertex /
    triangle buffer per batch plus per-frame ranges), and it keeps the host work per batch O(1): six strided views and
    one autograd node instead of nine views per frame.

    verts_aug, v_tng_aug (B, cap_va, 3); msdf (B, cap_va); faces_aug (B, cap_fa, 3) int64;
    vertices_watertight, v_tng_watertight (B, cap_v, 3); msdf_watertight (B, cap_v); faces_watertight (B, cap_fw, 3)
    n_verts_aug, n_faces_aug, n_verts_watertight, n_faces_watertight: int64 numpy arrays (B,)
    Differentiable: verts_aug, msdf, vertices_watertight, msdf_watertight (upstream gradients in the same padded
    shapes; rows beyond n_i are never read).  `frame(i)` narrows to the reference's 6-tuple of frame i."""

    def __init__(self, outs, sizes, wt):
        (self.verts_aug, self.v_tng_aug, self.msdf, self.vertices_watertight, self.v_tng_watertight,
         self.msdf_watertight, self.faces_aug, self.faces_watertight) = outs
        self.sizes = sizes
        self.n_verts_watertight = sizes[:, 4]
        self.n_verts_aug = sizes[:, 4] + sizes[:, 3]
        self.n_faces_aug = sizes[:, 5]
        self.n_faces_watertight = sizes[:, 1] + 2 * sizes[:, 2]
        self._wt = wt
        self._tape = None

    def __len__(self):
        return self.sizes.shape[0]

    def tape_edges(self, i: int) -> torch.Tensor:
        """(V_i, 2) int32: the crossing edges of frame i, row k = the grid vertices vertex k was interpolated between."""
        return _tape_edges(self._tape, i)

    def frame(self, i: int):
        v, va = int(self.n_verts_watertight[i]), int(self.n_verts_aug[i])
        fa, fw = int(self.n_faces_aug[i]), int(self.n_faces_watertight[i])
        msdf = self.msdf[i, :va]
        r8 = (self.verts_aug[i, :va], self.v_tng_aug[i, :va], msdf, self.vertices_watertight[i, :v],
              self.v_tng_watertight[i, :v], self.msdf_watertight[i, :v], msdf[v:], self.faces_aug[i, :fa],
              self.faces_watertight[i, :fw])
        return _pack_result(r8, self._wt)


class _PackedFn(torch.autograd.Function):
    """A batch of frames as one autograd node with PADDED batched outputs (see PackedFrames)."""

    @staticmethod
    def forward(ctx, spec, tets_i32, *tensors):
        refs, watertight_template, lanes, _launcher, started = spec
        pend, gbufs, n_grid = started
        pend, sizes, launches = _collect_packed(pend)
        lay, B = pend.lay, pend.B
        fslab, islab = pend.fslab, pend.islab
        cv, cva, cfw, cfa, ct = lay.caps
        o_vaug, o_tng, o_maug, o_vwt, o_twt, o_mwt = lay.f_off
        fl, il = lay.f_len, lay.i_len
        ast = torch.as_strided
        outs = (ast(fslab, (B, cva, 3), (fl, 3, 1), o_vaug), ast(fslab, (B, cva, 3), (fl, 3, 1), o_tng),
                ast(fslab, (B, cva), (fl, 1), o_maug), ast(fslab, (B, cv, 3), (fl, 3, 1), o_vwt),
                ast(fslab, (B, cv, 3), (fl, 3, 1), o_twt), ast(fslab, (B, cv), (fl, 1), o_mwt),
                ast(islab, (B, cfa, 3), (il, 3, 1), 0), ast(islab, (B, cfw, 3), (il, 3, 1), 3 * cfa))
        ctx.save_for_backward(*tensors, pend.tape, fslab)
        ctx.bmat, ctx.gbufs, ctx.sizes, ctx.lanes, ctx.nref = pend.bmat, gbufs, sizes, lanes, len(refs)
        ctx.zero_bwd = pend.zero_bwd
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(outs[6], outs[7])
        _ExtractFn.last_counts = None
        _PackedFn.last_sizes = sizes
        _ExtractFn.last_tape = (pend.tape, lay.tape_off[4], sizes[:, 4].tolist())
        _ExtractFn.last_launches = launches
        _ExtractFn.total_launches += launches
        return outs

    @staticmethod
    def backward(ctx, g0, g1, g2, g3, g4, g5, _g6, _g7):
        if g1 is not None or g4 is not None:
            raise NotImplementedError("gradients through v_tng (vertex tangents) are not implemented (see _ExtractFn)")
        tensors = ctx.saved_tensors[:-2]
        need = ctx.needs_input_grad[2:]
        gbufs, ctx.gbufs = ctx.gbufs, None
        bmat = ctx.bmat
        if bmat is None or gbufs is None:
            raise RuntimeError("backward through a packed batch needs inputs that require gradients, and runs once "
                               "(use extract_frames for retain_graph)")
        B = ctx.nref
        dev = tensors[0].device
        if ctx.zero_bwd:
            with torch.cuda.device(dev):
                _zero_backward(bmat, torch.cuda.current_stream(dev).cuda_stream)
        if g0 is None and g2 is None and g3 is None and g5 is None:
            return (None, None) + tuple(gbufs[i] if need[i] else None for i in range(len(tensors)))
        keep = []
        ar = np.arange(B, dtype=np.int64)

        def ptrs(t, inner):
            """per-frame pointers of a padded (B, cap, ...) gradient: rows must be dense, frames may be strided"""
            if t is None:
                return 0
            if t.dtype is not torch.float32 or t.stride()[1:] != inner:
                t = t.float().contiguous()
                keep.append(t)
            return t.data_ptr() + ar * (4 * t.stride(0))

        b = _BC
        bmat[:, b["g_verts_aug"]] = ptrs(g0, (3, 1))
        bmat[:, b["g_msdf_aug"]] = ptrs(g2, (1,))
        bmat[:, b["g_verts_wt"]] = ptrs(g3, (3, 1))
        bmat[:, b["g_msdf_wt"]] = ptrs(g5, (1,))
        bmat[:, b["g_msdf_boundary"]] = 0
        per16 = 2 if int(bmat[0, b["tape_slots"]]) == 0 else 1
        _ExtractFn.total_launches += per16 * ((B + 15) // 16)
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib().d3h_extract_backward_batch(bmat.ctypes.data, B, max(1, min(ctx.lanes, B)),
                                                               torch.cuda.current_stream(dev).cuda_stream),
                        "d3h_extract_backward_batch")
        return (None, None) + tuple(gbufs[i] if need[i] else None for i in range(len(tensors)))


_PackedFn.last_sizes = None


class FramesFuture:
    """A batch whose forward kernels are already running on the GPU (extract_frames_async).  `result()` blocks on the
    sizes, wraps the outputs in the autograd node and returns the list of reference 6-tuples; everything the host does
    between the launch and `result()` -- the `result()` / backward of an earlier batch, a renderer -- overlaps the GPU."""

    def __init__(self, spec, tets, tensors, n_frames, watertight):
        self._args = (spec, tets, tensors)
        self._n, self._wt = n_frames, watertight
        self._out = None
        self._tape = None

    def __del__(self):
        # dropped without result(): the lanes may still be writing this batch's buffers, which are about to be freed
        if self._out is None and self._n and self._args is not None:
            try:
                pend = self._args[0][4][0]
                pend.plan.inflight = max(0, pend.plan.inflight - pend.B)   # its count slots are free again
            except Exception:  # pragma: no cover
                pass
        if self._out is None and self._n > 1 and self._args is not None:
            try:
                dev = self._args[2][0].device
                with torch.cuda.device(dev):
                    _cabi.lib().d3h_lanes_join(torch.cuda.current_stream(dev).cuda_stream)
            except Exception:  # pragma: no cover  (interpreter shutdown)
                pass

    def tape_edges(self, i: int) -> torch.Tensor:
        """(V_i, 2) int32 crossing edges of frame i (after result() / packed()): the grid vertices the frame's gradients
        can touch -- see gather_touched."""
        if self._tape is None:
            raise RuntimeError("tape_edges: call result() or packed() first")
        return _tape_edges(self._tape, i)

    def packed(self) -> "PackedFrames":
        """The batch as padded tensors (PackedFrames) instead of a list of per-frame tuples: O(1) host work per batch."""
        if self._out is None:
            spec, tets, tensors = self._args
            if not self._n:
                raise ValueError("an empty batch has no packed form")
            outs = _PackedFn.apply(spec, tets, *tensors)
            self._out = PackedFrames(outs, _PackedFn.last_sizes, self._wt)
            self._out._tape = self._tape = _ExtractFn.last_tape
            self._args = None
        return self._out

    def result(self):
        if self._out is None:
            spec, tets, tensors = self._args
            flat = _ExtractFn.apply(spec, tets, *tensors) if self._n else ()
            self._out = [_pack_result(flat[_OUTS_PER_FRAME * i:_OUTS_PER_FRAME * (i + 1)], self._wt)
                         for i in range(self._n)]
            self._tape = _ExtractFn.last_tape if self._n else None
            self._args = None
        return self._out


def extract_frames(pos_frames, sdf_n, msdf_n, tet_fx4, types=None, output_watertight_template: bool = True,
                   lanes: int = DEFAULT_LANES, fused_pair: bool = False):
    """extract_frames_async(...).result(): launch, then block on the sizes."""
    return extract_frames_async(pos_frames, sdf_n, msdf_n, tet_fx4, types, output_watertight_template, lanes,
                                fused_pair).result()


def extract_frames_async(pos_frames, sdf_n, msdf_n, tet_fx4, types=None, output_watertight_template: bool = True,
                         lanes: int = DEFAULT_LANES, fused_pair: bool = False) -> FramesFuture:
    """A batch of extractions on the same tet grid in one autograd node and one library call per direction.

    No counterpart in the reference, which would loop over the frames (BASELINE.json configs[3]: a batch of video frames
    per step with per-frame tet-vertex offsets; also the cloth / body pair of train.py:1040-1047).

    pos_frames : (B,N,3) tensor (one autograd leaf for the whole batch) or a sequence of (N,3) tensors
    sdf_n, msdf_n : one tensor shared by all frames ((N,) or (N,1)), a stacked (B,N) tensor, or a sequence per frame
    types : None (GShell_Tets semantics), one of "cloth" / "body" for all frames, or a sequence per frame
            (hmSDF_Tets semantics: "body" uses -msdf and, like the reference, does not back-propagate into msdf_n)
    fused_pair : EXPERIMENTAL (validated on the CPU emulation of the kernels only, tests/test_emu_parity.py): the two
            frames are the cloth / body pair of one iteration (same tensors, types cloth and body); one library call
            classifies and de-duplicates once and only replays the mSDF cut for the second frame.
    Returns a FramesFuture; `.result()` is a list with the reference's 6-tuple `(verts, faces, None, None, v_tng, extra)`
    for every frame.  Gradients of shared tensors are summed over the frames.  The forward kernels are enqueued before
    this function returns; the host only blocks (once per frame, on the output sizes) inside `.result()`.
    """
    tensors: List[torch.Tensor] = []
    index: Dict[int, int] = {}

    def intern(src, prep):
        k = id(src)
        if k not in index:
            index[k] = len(tensors)
            tensors.append(prep(src))
        return index[k]

    if torch.is_tensor(pos_frames):
        if pos_frames.dim() != 3 or pos_frames.shape[2] != 3:
            raise ValueError(f"pos_frames must be (B,N,3), got {tuple(pos_frames.shape)}")
        _check_cuda(pos_frames)
        B, n_grid = pos_frames.shape[0], pos_frames.shape[1]
        if B == 0:
            return FramesFuture(None, None, None, 0, output_watertight_template)
        tensors.append(_aligned(pos_frames.float()))
        pos_refs = [(0, i) for i in range(B)]
    else:
        pos_list = list(pos_frames)
        B = len(pos_list)
        if B == 0:
            return FramesFuture(None, None, None, 0, output_watertight_template)
        pos_refs = [(intern(p, _prep_pos), -1) for p in pos_list]
        n_grid = tensors[pos_refs[0][0]].shape[0]

    def field_refs(f):
        if torch.is_tensor(f):
            if f.dim() == 2 and f.shape[0] == B and f.shape[1] == n_grid and n_grid > 1:   # stacked (B,N)
                if (4 * n_grid) % 16:
                    raise ValueError("a stacked (B,N) field needs N % 4 == 0 (16-byte aligned rows); pass a list instead")
                _check_cuda(f)
                k = intern(f, lambda t: _aligned(t.float()))
                return [(k, i) for i in range(B)]
            k = intern(f, lambda t: _prep_field(t, n_grid))
            return [(k, -1)] * B
        fl = list(f)
        if len(fl) != B:
            raise ValueError("sdf_n / msdf_n / types must be shared or have one entry per frame")
        return [(intern(t, lambda u: _prep_field(u, n_grid)), -1) for t in fl]

    sdf_refs, msdf_refs = field_refs(sdf_n), field_refs(msdf_n)
    type_list = [types] * B if (types is None or isinstance(types, str)) else list(types)
    if len(type_list) != B:
        raise ValueError("sdf_n / msdf_n / types must be shared or have one entry per frame")
    for r in pos_refs:
        if tensors[r[0]].shape[-2] != n_grid:
            raise ValueError("all frames must live on the same tet grid (same N)")
    refs = tuple((pos_refs[i], sdf_refs[i], msdf_refs[i], type_list[i] == "body") for i in range(B))
    tets = packed_tets(tet_fx4, n_grid)
    wt = bool(output_watertight_template)
    grad_on = torch.is_grad_enabled()
    need = tuple(grad_on and t.requires_grad for t in tensors)
    if fused_pair and not (B == 2 and refs[0][:3] == refs[1][:3] and refs[0][3] != refs[1][3]):
        raise ValueError("fused_pair needs exactly two frames on the same pos / sdf / msdf tensors, types cloth and body")
    if fused_pair and not wt:
        # output_watertight_template=False keeps only tets with a positive mSDF vertex (gshell_tets.py:275): the set of
        # valid tets depends on the mSDF sign, cloth and body do not share their classification
        raise ValueError("fused_pair needs output_watertight_template=True")
    started = _prelaunch(refs, tensors, need, tets, wt, int(lanes), None, static_edges_for(tets, n_grid), fused_pair)
    return FramesFuture((refs, wt, int(lanes), None, started), tets, tensors, B, wt)
