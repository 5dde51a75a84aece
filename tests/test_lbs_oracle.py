"""The skinning oracle (oracle/lbs_oracle.py, float64) against the reference's own methods
(deform/smplx_exavatar_deformer.py:363-421, executed from the reference source with a brute-force knn_points) -- build
container only -- and against the golden vectors written from them (tests/golden/lbs_*.npz)."""
import glob
import os
import types

import numpy as np
import pytest

from oracle import lbs_oracle as LO
from oracle import ref_loader

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "lbs_*.npz")))


def synthetic_rig(seed, vt=400, j=12):
    """A random articulated template: vertices, sparse-ish skinning weights (rows sum to one), rigid-ish 4x4 transforms."""
    rng = np.random.default_rng(seed)
    template = rng.uniform(-1, 1, size=(vt, 3)).astype(np.float32)
    w = rng.random((vt, j)).astype(np.float32) ** 4
    w /= w.sum(1, keepdims=True)

    def transforms():
        a = np.tile(np.eye(4, dtype=np.float32), (j, 1, 1))
        for k in range(j):       # moderate rotations (Rodrigues, |angle| ~ 0.6 rad): blends of them stay well conditioned,
            r = 0.35 * rng.standard_normal(3)     # like the joint transforms of a posed body
            th = np.linalg.norm(r) + 1e-12
            kx = np.array([[0, -r[2], r[1]], [r[2], 0, -r[0]], [-r[1], r[0], 0]]) / th
            rot = np.eye(3) + np.sin(th) * kx + (1 - np.cos(th)) * kx @ kx
            a[k, :3, :3] = rot.astype(np.float32)
            a[k, :3, 3] = (0.3 * rng.standard_normal(3)).astype(np.float32)
        return a
    return template, w.astype(np.float32), transforms(), transforms(), (0.2 * rng.standard_normal(3)).astype(np.float32)


def reference_lbs(pts, template, w, init_a, a, trans, grads=None):
    """deformer.lbs_forward :472-476 composed from the reference's two methods"""
    import torch
    interp, apply_inv = ref_loader.load_reference_lbs_methods()
    self = types.SimpleNamespace(vs_template=torch.tensor(template)[None], lbs_weights=torch.tensor(w), k=1)
    tp = torch.tensor(pts[None], requires_grad=True)
    ta = torch.tensor(a[None], requires_grad=True)
    tt = torch.tensor(trans.reshape(1, 3), requires_grad=True)
    w_pts = interp(self, tp)
    can = apply_inv(self, tp, torch.tensor(init_a[None]), w_pts)
    new = apply_inv(self, can, ta, w_pts, Inverse=False) + tt
    out = new.reshape(-1, 3)
    res = [out.detach().numpy(), can.detach().numpy()[0]]
    if grads is not None:
        (out * torch.tensor(grads)).sum().backward()
        res += [tp.grad.numpy()[0], ta.grad.numpy()[0], tt.grad.numpy()[0]]
    return res


@pytest.mark.parametrize("seed", range(4))
def test_oracle_matches_reference_methods(seed):
    if not ref_loader.reference_available():
        pytest.skip("needs a checkout of the original project (D3H_REFERENCE_ROOT)")
    template, w, init_a, a, trans = synthetic_rig(seed)
    rng = np.random.default_rng(100 + seed)
    pts = rng.uniform(-1.1, 1.1, size=(700, 3)).astype(np.float32)
    pts[::5] = 0.0                                       # the zeroed rows of verts_aug (gshell_tets.py:423-427)
    g = rng.standard_normal(pts.shape).astype(np.float32)
    posed, can, g_pts, g_a, g_t = reference_lbs(pts, template, w, init_a, a, trans, g)
    want, cache = LO.lbs_forward(pts, template, w, init_a, a, trans)
    assert np.abs(posed - want).max() < 2e-5 * max(1.0, np.abs(want).max())
    assert np.abs(can - LO.lbs_forward_inverse(pts, template, w, init_a)).max() < 2e-5
    o_pts, o_a, o_t = LO.lbs_backward(cache, g)
    assert np.abs(g_pts - o_pts).max() < 1e-4 * np.abs(o_pts).max()
    assert np.abs(g_a - o_a).max() < 1e-4 * np.abs(o_a).max()
    assert np.abs(g_t - o_t).max() < 1e-4 * np.abs(o_t).max()


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_reproduces_golden_vectors(path):
    d = np.load(path)
    want, cache = LO.lbs_forward(d["pts"], d["template"], d["w"], d["init_a"], d["a"], d["trans"])
    assert np.abs(d["posed"] - want).max() < 2e-5 * max(1.0, np.abs(want).max())
    o_pts, o_a, o_t = LO.lbs_backward(cache, d["g"])
    assert np.abs(d["g_pts"] - o_pts).max() < 1e-4 * np.abs(o_pts).max()
    assert np.abs(d["g_a"] - o_a).max() < 1e-4 * np.abs(o_a).max()
    assert np.abs(d["g_trans"] - o_t).max() < 1e-4 * np.abs(o_t).max()
