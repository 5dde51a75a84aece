"""Float64 numpy oracle of the SDF sign-change regulariser (the reference's `compute_sdf_reg_loss`, geometry/hmsdf.py:162-170;
the product: geometry/sdf_reg.py).  Test infrastructure only.

An edge (a, b) is selected when np.sign(s_a) != np.sign(s_b) (three-valued; NaN selects); with M selected edges
    loss     = mean_e BCE(s_a, [s_b > 0]) + mean_e BCE(s_b, [s_a > 0]),  BCE(x, t) = (1 - t) x - log_sigmoid(x)
    g_sdf[a] += g (sigmoid(s_a) - [s_b > 0]) / M,  g_sdf[b] += g (sigmoid(s_b) - [s_a > 0]) / M
The loss is NaN and the gradient zero when M = 0.  The inputs are taken as float32 values (the product computes in
float32), everything after that in float64."""
from __future__ import annotations

import os

import numpy as np

from oracle import ref_loader


def _log_sigmoid(x):
    return np.minimum(x, 0.0) - np.log1p(np.exp(-np.abs(x)))


def _sigmoid(x):
    return np.exp(_log_sigmoid(x))


def selected(sdf, all_edges):
    """-> (a, b) int64 arrays of the selected edges, in the order of all_edges"""
    s = np.asarray(sdf, dtype=np.float32).reshape(-1).astype(np.float64)
    e = np.asarray(all_edges, dtype=np.int64).reshape(-1, 2)
    a, b = e[:, 0], e[:, 1]
    with np.errstate(invalid="ignore"):
        m = np.sign(s[a]) != np.sign(s[b])
    return a[m], b[m]


def sdf_reg_loss(sdf, all_edges):
    """-> float64 loss"""
    s = np.asarray(sdf, dtype=np.float32).reshape(-1).astype(np.float64)
    a, b = selected(sdf, all_edges)
    if a.shape[0] == 0:
        return float("nan")
    sa, sb = s[a], s[b]
    ta, tb = (sa > 0).astype(np.float64), (sb > 0).astype(np.float64)
    return float(np.mean((1.0 - tb) * sa - _log_sigmoid(sa)) + np.mean((1.0 - ta) * sb - _log_sigmoid(sb)))


def sdf_reg_grad(sdf, all_edges, g: float = 1.0):
    """-> float64 gradient (N,) for an upstream gradient g"""
    s = np.asarray(sdf, dtype=np.float32).reshape(-1).astype(np.float64)
    a, b = selected(sdf, all_edges)
    out = np.zeros(s.shape[0], dtype=np.float64)
    if a.shape[0] == 0:
        return out
    sa, sb = s[a], s[b]
    ta, tb = (sa > 0).astype(np.float64), (sb > 0).astype(np.float64)
    np.add.at(out, a, g * (_sigmoid(sa) - tb) / a.shape[0])
    np.add.at(out, b, g * (_sigmoid(sb) - ta) / a.shape[0])
    return out


def load_reference_sdf_reg_loss():
    """-> the reference's `compute_sdf_reg_loss` (geometry/hmsdf.py:162-170) from the checkout at D3H_REFERENCE_ROOT
    (oracle/ref_loader.py), compiled alone from the source text with `ast` as ref_loader.load_reference_lbs_methods does:
    hmsdf.py itself cannot be imported here (pysdf, trimesh, nvdiffrast).  Found at module level or as a method."""
    import ast
    import torch
    import torch.nn.functional as F

    path = os.path.join(ref_loader.REF_ROOT, "geometry", "hmsdf.py")
    with open(path) as fh:
        tree = ast.parse(fh.read())
    found = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name == "compute_sdf_reg_loss"]
    if not found:
        raise LookupError(f"compute_sdf_reg_loss not found in {path}")
    fn = found[0]
    fn.decorator_list = []
    ns = {"torch": torch, "F": F}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
    f = ns["compute_sdf_reg_loss"]
    if fn.args.args and fn.args.args[0].arg == "self":   # a method: `self` is not used by the loss
        return lambda sdf, all_edges: f(None, sdf, all_edges)
    return f
