"""Inputs of the SDF regulariser tests: `generate_edges` of the reference (geometry/hmsdf.py:381-388) and grids with a
chosen vertex or entry count.  Test infrastructure only."""
import numpy as np
import torch

from d3human_code_b200 import grids

TET_EDGES = [0, 1, 0, 2, 0, 3, 1, 2, 1, 3, 2, 3]


def generate_edges_reference(indices: torch.Tensor) -> torch.Tensor:
    """The reference's construction, literally: the six edges of every tet, sorted within the row, torch.unique(dim=0)."""
    edges = torch.tensor(TET_EDGES, dtype=torch.long, device=indices.device)
    all_edges = indices[:, edges].reshape(-1, 2)
    return torch.unique(torch.sort(all_edges, dim=1)[0], dim=0)


def generate_edges(indices: torch.Tensor, n_grid: int) -> torch.Tensor:
    """The same (E,2) int64 tensor through a 1-D unique of the keys min * N + max (ascending keys = ascending rows), which
    is far cheaper than unique(dim=0) at 128^3."""
    edges = torch.tensor(TET_EDGES, dtype=torch.long, device=indices.device)
    e = indices.long()[:, edges].reshape(-1, 2)
    key = torch.unique(torch.minimum(e[:, 0], e[:, 1]) * n_grid + torch.maximum(e[:, 0], e[:, 1]))
    a = torch.div(key, n_grid, rounding_mode="floor")
    return torch.stack([a, key - a * n_grid], 1)


def kuhn_edges(res: int, n=None):
    """(pos (n,3), all_edges (E,2) int64 numpy) of the res^3 Kuhn lattice, keeping the first n vertices and the edges
    between them (n = None: all (res+1)^3)"""
    pos, tets = grids.kuhn_grid(res)
    n_all = pos.shape[0]
    e = generate_edges(torch.from_numpy(tets), n_all).numpy()
    if n is not None:
        e = e[(e < n).all(1)]
        pos = pos[:n]
    return pos, e


def chain_edges(n_chunks: int, diffs=(1,)):
    """N = 32 n_chunks vertices and the edges (v, v + d) for every d in diffs: n_chunks entries per d in the run-length
    table (every entry holds >= 32 - d edges)"""
    n = 32 * n_chunks
    v = np.arange(n)
    e = np.concatenate([np.stack([v[v + d < n], v[v + d < n] + d], 1) for d in diffs])
    return n, e


def capsule_field(pos, zeros_every: int = 0):
    """the capsule-union body SDF (grids.capsule_garment_field) in float32; every `zeros_every`-th value an exact zero"""
    s = grids.capsule_garment_field(pos)[0].copy()
    if zeros_every:
        s[::zeros_every] = 0.0
    return s


def random_field(n: int, seed: int = 0, zeros_every: int = 7):
    rng = np.random.default_rng(seed)
    s = rng.standard_normal(n).astype(np.float32)
    if zeros_every:
        s[::zeros_every] = 0.0
    return s
