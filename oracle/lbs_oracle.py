"""TEST INFRASTRUCTURE ONLY.

CPU restatement (numpy float64) of the linear-blend skinning D3-Human applies to the extracted vertices (SURVEY.md
section 8f row 4): deform/smplx_exavatar_deformer.py

    interpolate_weights  :363-383   K nearest template vertices (pytorch3d.ops.knn_points, squared Euclidean distances),
                                    inverse-distance weights normalised over the K neighbours, blended skinning weights
    apply_lbs_inverse    :385-421   M_p = sum_j w[p,j] A_j (4x4), optionally inverted, applied to [p; 1]
    lbs_forward          :472-476   canonical = M_p(init_A)^-1 p ;  posed = M_p(A) canonical + trans

The class hard-codes `self.k = 1` (:39): with one neighbour the normalised inverse-distance weight is exactly 1, so
w[p,:] = lbs_weights[nearest(p),:] and M_p = B[nearest(p)] with B[v] = sum_j lbs_weights[v,j] A_j.

`knn_points` belongs to pytorch3d (third-party, not installed here; the reference's README pins no version): K nearest
points by squared distance, ascending -- restated as a brute-force argmin.  Pinned against the reference's own two
methods, executed from the reference source with that brute-force stand-in for knn_points (tests/test_lbs_oracle.py).
"""
from __future__ import annotations

import numpy as np


def nearest(pts, template):
    """index of the nearest template vertex of every point (K = 1), squared distances in float64"""
    p = np.asarray(pts, np.float64)
    t = np.asarray(template, np.float64)
    out = np.empty(p.shape[0], np.int64)
    for lo in range(0, p.shape[0], 4096):
        d = ((p[lo:lo + 4096, None, :] - t[None, :, :]) ** 2).sum(-1)
        out[lo:lo + 4096] = d.argmin(1)
    return out


def blend(lbs_weights, A):
    """B[v] = sum_j lbs_weights[v, j] A[j]  ->  (Vt, 4, 4)"""
    return np.einsum("vj,jab->vab", np.asarray(lbs_weights, np.float64), np.asarray(A, np.float64))


def lbs_forward(pts, template, lbs_weights, init_A, A, trans, idx=None):
    """deformer.lbs_forward :472-476 for one frame.  -> (posed (P,3), cache).  idx (P): nearest template vertex of every
    point when already known (None: searched here)"""
    idx = nearest(pts, template) if idx is None else np.asarray(idx, np.int64)
    b_init, b_pose = blend(lbs_weights, init_A), blend(lbs_weights, A)
    inv = np.linalg.inv(b_init)
    ph = np.concatenate([np.asarray(pts, np.float64), np.ones((len(pts), 1))], 1)
    can = np.einsum("pab,pb->pa", inv[idx], ph)[:, :3]
    ch = np.concatenate([can, np.ones((len(pts), 1))], 1)
    posed = np.einsum("pab,pb->pa", b_pose[idx], ch)[:, :3] + np.asarray(trans, np.float64).reshape(1, 3)
    return posed, dict(idx=idx, inv=inv, b_pose=b_pose, can_h=ch, lbs_weights=np.asarray(lbs_weights, np.float64))


def lbs_forward_inverse(pts, template, lbs_weights, init_A, idx=None):
    """deformer.lbs_forward_inverse :424-430"""
    idx = nearest(pts, template) if idx is None else np.asarray(idx, np.int64)
    inv = np.linalg.inv(blend(lbs_weights, init_A))
    ph = np.concatenate([np.asarray(pts, np.float64), np.ones((len(pts), 1))], 1)
    return np.einsum("pab,pb->pa", inv[idx], ph)[:, :3]


def lbs_backward(cache, g_posed):
    """-> (g_pts (P,3), g_A (J,4,4), g_trans (3,)): init_A is a constant of the run (deformer.initialize :173-235), the
    nearest-neighbour index carries no gradient, and with K = 1 the weights do not depend on the distances."""
    g = np.asarray(g_posed, np.float64)
    idx, inv, b_pose, ch = cache["idx"], cache["inv"], cache["b_pose"], cache["can_h"]
    total = np.einsum("pab,pbc->pac", b_pose[idx], inv[idx])          # posed = total [p; 1] (+ trans)
    g_pts = np.einsum("pa,pab->pb", g, total[:, :3, :3])
    g_b = np.zeros_like(b_pose)
    np.add.at(g_b[:, :3, :], idx, g[:, :, None] * ch[:, None, :])
    g_a = np.einsum("vj,vab->jab", cache["lbs_weights"], g_b)
    return g_pts, g_a, g.sum(0)
