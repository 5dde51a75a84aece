"""`compute_sdf_reg_loss`: drop-in for the reference's SDF sign-change regulariser (geometry/hmsdf.py:162-170, called at
:882 with `self.all_edges` from `generate_edges`, :381-388), on the kernels of csrc/d3h_sdf_reg.cu (include/d3h_tets.h).

    loss = mean_e BCE(sdf[a], [sdf[b] > 0]) + mean_e BCE(sdf[b], [sdf[a] > 0])

over the edges (a, b) of `all_edges` whose end points differ in `torch.sign` (three-valued: an edge from 0 to either sign
is selected, (+0.0, -0.0) and self edges are not).  As in the reference the loss is NaN when no edge is selected; it is
also NaN when `sdf` holds a NaN (the reference selects every edge at a NaN vertex, and every vertex of a tet grid lies on
an edge).  ±inf values are not treated specially.

The reference gathers both end points of every edge, compacts the selection with a boolean mask (a device -> host sync)
and runs two BCE kernels.  Here `all_edges` is turned ONCE per tensor into one of the static edge tables of the
extraction's edge scan (extract.build_edge_runs: a (d, mask) entry per chunk of 32 vertices and end-point difference on
grids numbered along their axes; extract.build_edge_rows otherwise), and a call reads that table and two sign bitmaps.
Neither the forward nor the backward pass waits for the device.  CUDA tensors only.
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch
from torch.autograd.function import once_differentiable

from .. import _cabi
from .. import extract as _E

_cache: Dict[Tuple, "EdgeTables"] = {}


class EdgeTables:
    """The static table of one `all_edges` tensor: `form` is "runs" (edge_runs, edge_run_chunk) or "rows" (edge_rows,
    edge_row_off); `nbytes` is what a call reads of it."""

    def __init__(self, n_grid: int, n_edges: int, runs, rows, source: torch.Tensor):
        self.n_grid, self.n_edges = n_grid, n_edges
        self.edge_runs, self.edge_run_chunk = runs
        self.edge_rows, self.edge_row_off = rows
        self.form = "runs" if self.edge_runs is not None else "rows"
        self.n_runs = int(self.edge_runs.shape[0]) if self.form == "runs" else 0
        parts = (self.edge_runs, self.edge_run_chunk) if self.form == "runs" else (self.edge_rows, self.edge_row_off)
        self.nbytes = sum(t.numel() * t.element_size() for t in parts)
        self._source = source            # kept alive: its address is part of the cache key

    def pointers(self):
        p = lambda t: t.data_ptr() if t is not None else None   # noqa: E731
        return p(self.edge_runs), p(self.edge_run_chunk), self.n_runs, p(self.edge_rows), p(self.edge_row_off)


def _build(all_edges: torch.Tensor, n_grid: int) -> EdgeTables:
    if all_edges.dtype.is_floating_point or all_edges.dtype.is_complex or all_edges.dtype == torch.bool:
        raise ValueError(f"all_edges must be an integer tensor, got {all_edges.dtype}")
    if all_edges.dim() != 2 or all_edges.shape[1] != 2:
        raise ValueError(f"all_edges must have shape (E,2), got {tuple(all_edges.shape)}")
    n_edges = int(all_edges.shape[0])
    if n_edges >= 2 ** 31:
        raise ValueError("all_edges has 2^31 edges or more")
    dev = all_edges.device
    e = all_edges.long()
    if n_edges and (int(e.min()) < 0 or int(e.max()) >= n_grid):
        raise ValueError(f"all_edges holds vertex ids outside [0, {n_grid}) (sdf has {n_grid} rows)")
    a, b = torch.minimum(e[:, 0], e[:, 1]), torch.maximum(e[:, 0], e[:, 1])
    key = torch.sort(a * n_grid + b).values                # rows as (min, max), ascending
    if n_edges > 1 and bool((key[1:] == key[:-1]).any()):
        raise ValueError("all_edges lists an edge twice (as (a, b) or (b, a)); generate_edges() yields distinct edges")
    a = torch.div(key, n_grid, rounding_mode="floor") if n_grid else key
    edge_ab = torch.stack([a, key - a * n_grid], 1).to(torch.int32).contiguous()
    edge_off = torch.zeros(n_grid + 1, dtype=torch.int64, device=dev)
    edge_off[1:] = torch.cumsum(torch.bincount(a, minlength=n_grid), 0)
    runs, chunk, _ids = _E.build_edge_runs(edge_off, edge_ab, n_grid)
    rows = (None, None)
    if runs is None:
        rows = _E.build_edge_rows(edge_off, edge_ab, n_grid)
    return EdgeTables(n_grid, n_edges, (runs, chunk), rows, all_edges)


def tables_for(all_edges: torch.Tensor, n_grid: int) -> EdgeTables:
    """The static table of `all_edges` for a field of `n_grid` values, built on first use.  The key holds the tensor's
    version counter: an in-place edit of `all_edges` builds a new table."""
    key = (all_edges.data_ptr(), all_edges._version, tuple(all_edges.shape), str(all_edges.device), int(n_grid))
    ent = _cache.get(key)
    if ent is None:
        if len(_cache) > 8:
            _cache.clear()
        ent = _cache[key] = _build(all_edges, int(n_grid))
    return ent


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _workspace(dev, nbytes: int) -> torch.Tensor:
    """`nbytes` bytes, 16-byte aligned (CUDA allocations are; CPU tensors of the emulated tests need not be)"""
    w = torch.empty(nbytes + 16, dtype=torch.uint8, device=dev)
    off = -w.data_ptr() % 16
    return w[off:off + nbytes]


class _SdfRegFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sdf, tables: EdgeTables):
        L = _cabi.lib()
        dev = sdf.device
        n = sdf.shape[0]
        nbytes = int(L.d3h_sdf_reg_workspace_bytes(n, tables.n_runs))
        ws = _workspace(dev, nbytes)
        loss = torch.empty(1, dtype=torch.float32, device=dev).reshape(())
        with torch.cuda.device(dev):
            _cabi.check(L.d3h_sdf_reg_forward(sdf.data_ptr(), n, *tables.pointers(), ws.data_ptr(), nbytes, loss.data_ptr(),
                                              _stream(dev)), "d3h_sdf_reg_forward")
        ctx.save_for_backward(sdf)
        ctx.tables, ctx.ws, ctx.nbytes = tables, ws, nbytes   # the sign bitmaps and M of this call
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (sdf,) = ctx.saved_tensors
        L = _cabi.lib()
        dev = sdf.device
        g = g.float().contiguous()
        g_sdf = torch.zeros(sdf.shape[0], dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _cabi.check(L.d3h_sdf_reg_backward(sdf.data_ptr(), sdf.shape[0], *ctx.tables.pointers(), g.data_ptr(), ctx.ws.data_ptr(),
                                               ctx.nbytes, g_sdf.data_ptr(), _stream(dev)), "d3h_sdf_reg_backward")
        return g_sdf, None


def compute_sdf_reg_loss(sdf: torch.Tensor, all_edges: torch.Tensor) -> torch.Tensor:
    """sdf (N,1) or (N,) (other float dtypes are computed in float32; the gradient comes back in sdf's shape and dtype),
    all_edges (E,2) integer, distinct edges with ids in [0, N), either row order -> 0-dim float32 loss."""
    _E._check_cuda(sdf)
    _E._check_cuda(all_edges)
    if not (sdf.dim() == 1 or (sdf.dim() == 2 and sdf.shape[1] == 1)):
        raise ValueError(f"sdf must have shape (N,) or (N,1), got {tuple(sdf.shape)}")
    flat = sdf.float().reshape(-1).contiguous()
    return _SdfRegFn.apply(flat, tables_for(all_edges, flat.shape[0]))
