"""Skinning kernels (include/d3h_lbs.h, csrc/d3h_lbs.cu) at the edges they branch on, against the float64 oracle
(oracle/lbs_oracle.py): the 1024-vertex template tiles of the search, the origin's entry at index `count` of the search
list, ties, pivot swaps of the Gauss-Jordan inverse, exactly-zero weights, J = 1 / 128, NULL `trans` / `b_pose` / `pts`,
zero upstream rows, zero rows that do not share one table row, P = 0.  Most cases drive the C ABI directly; the module
cases go through deform/lbs.py.  Each case body takes the device; tests/test_emu_lbs.py runs the same bodies on the CPU
emulation of the kernels.

Positions and gradients to the points are computed row by row and are checked row by row: the largest error of a row,
relative to max(1, the row's largest entry), stays under POS_TOL / GPTS_TOL.  g_A and g_trans are sums over many rows
(float atomics in any order): relative to their largest entry, under SUM_TOL.  The emulation reproduces the GPU's float
op order except for the order of the atomics.  Largest errors seen on one B200: see the constants."""
import numpy as np
import pytest
import torch

from d3human_code_b200 import _cabi
from oracle import lbs_oracle as LO
from tests.test_lbs_oracle import synthetic_rig

pytestmark = pytest.mark.gpu
POS_TOL = 2e-6       # posed / canonical rows
GPTS_TOL = 2e-6      # g_pts rows
SUM_TOL = 2e-6       # g_A, g_trans (relative to the largest entry)
BENCH_SUM_TOL = 1e-5  # the same at the benchmark's shape: 207 000 zero rows summed in float


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture
def module_dev(dev):
    return dev


# ---------------------------------------------------------------------------------------------- helpers
def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else None


def _sync(dev):
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)


def _buf(dev, shape, dtype=torch.float32, fill=0):
    """a 16-byte aligned buffer (the ABI's tables and workspace need it; CPU tensors are not always 16-byte aligned)"""
    n = int(np.prod(shape))
    b = torch.full((n + 16,), fill, dtype=dtype, device=dev)
    off = (-b.data_ptr() % 16) // b.element_size()
    return b[off:off + n].view(shape)


def _put(dev, arr, dtype=torch.float32):
    arr = np.ascontiguousarray(arr)
    t = _buf(dev, arr.shape, dtype)
    t.copy_(torch.from_numpy(arr).to(dtype))
    return t


def _ptr(t):
    return t.data_ptr() if t is not None else None


def abi_skin(dev, template, w, init_a, a, trans, pts, g, use_pts=True, idx=None, g_trans=True):
    """The ABI chain of one frame: blend (init_A, inverted) -> nearest (unless idx is given) -> blend (A) -> apply ->
    apply_backward -> blend_backward.  Outputs that the ABI overwrites start as NaN."""
    L, st = _cabi.lib(), _stream(dev)
    vt, nj = w.shape
    p = pts.shape[0]
    tw, tia, ta, tm, tp, tg = (_put(dev, x) for x in (w, init_a, a, template, pts, g))
    tt = _put(dev, trans) if trans is not None else None
    binv, bpose = _buf(dev, (vt, 16), fill=np.nan), _buf(dev, (vt, 16), fill=np.nan)
    _cabi.check(L.d3h_lbs_blend(_ptr(tw), _ptr(tia), vt, nj, 1, _ptr(binv), st), "d3h_lbs_blend")
    _cabi.check(L.d3h_lbs_blend(_ptr(tw), _ptr(ta), vt, nj, 0, _ptr(bpose), st), "d3h_lbs_blend")
    if idx is None:
        tidx = _buf(dev, (p,), torch.int32, fill=-7)
        nb = int(L.d3h_lbs_nearest_workspace_bytes(p))
        ws = _buf(dev, (max(nb // 4, 16),), torch.int32, fill=-7)
        _cabi.check(L.d3h_lbs_nearest(_ptr(tp), p, _ptr(tm), vt, _ptr(tidx), _ptr(ws), nb, st), "d3h_lbs_nearest")
    else:
        tidx = _put(dev, idx, torch.int32)
    can, posed = _buf(dev, (p, 3), fill=np.nan), _buf(dev, (p, 3), fill=np.nan)
    _cabi.check(L.d3h_lbs_apply(_ptr(tp), p, _ptr(tidx), _ptr(binv), _ptr(bpose), _ptr(tt), _ptr(can), _ptr(posed), st), "d3h_lbs_apply")
    g_pts, g_b = _buf(dev, (p, 3), fill=np.nan), _buf(dev, (vt, 12))
    g_t = _buf(dev, (3,)) if g_trans else None
    _cabi.check(L.d3h_lbs_apply_backward(_ptr(tg), p, _ptr(tidx), _ptr(binv), _ptr(bpose), _ptr(can), _ptr(tp) if use_pts else None,
                                         _ptr(g_pts), _ptr(g_b), _ptr(g_t), st), "d3h_lbs_apply_backward")
    g_a = _buf(dev, (nj, 4, 4), fill=np.nan)
    _cabi.check(L.d3h_lbs_blend_backward(_ptr(tw), _ptr(g_b), vt, nj, _ptr(g_a), st), "d3h_lbs_blend_backward")
    _sync(dev)
    out = dict(idx=tidx.cpu().numpy(), can=can.cpu().numpy(), posed=posed.cpu().numpy(), g_pts=g_pts.cpu().numpy(),
               g_a=g_a.cpu().numpy(), g_b=g_b.cpu().numpy())
    out["g_trans"] = g_t.cpu().numpy() if g_t is not None else None
    return out


def _rows_close(got, want, tol, what):
    """every row: max |got - want| <= tol * max(1, max |want row|)"""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if got.size == 0:
        return
    assert np.isfinite(got).all(), (what, "not finite")
    err = np.abs(got - want).max(1) / np.maximum(1.0, np.abs(want).max(1))
    assert err.max() <= tol, (what, int(err.argmax()), float(err.max()))


def _sum_close(got, want, tol, what):
    assert got.shape == want.shape and np.isfinite(got).all(), (what, got.shape, want.shape)
    err = np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)
    assert err <= tol, (what, float(err))


def check_idx(idx, pts, template, exact=None):
    """-> the oracle's index.  Exact except for fp32 near-ties, which must be ties of the float64 distances too;
    `exact` (bool mask) rows must match exactly whatever the distances (designed ties: the lowest index wins)."""
    want = LO.nearest(pts, template)
    bad = idx != want
    if exact is not None:
        assert not (bad & exact).any(), np.nonzero(bad & exact)[0][:10]
    if bad.any():
        p64, t64 = pts[bad].astype(np.float64), template.astype(np.float64)
        d_got = ((p64 - t64[idx[bad]]) ** 2).sum(-1)
        d_want = ((p64 - t64[want[bad]]) ** 2).sum(-1)
        assert np.all(np.abs(d_got - d_want) <= 1e-6 * (1 + d_want)) and bad.mean() < 1e-3, np.nonzero(bad)[0][:10]
    return want


def check_against_oracle(r, pts, template, w, init_a, a, trans, g, idx=None, exact=None, sum_tol=SUM_TOL):
    """r = abi_skin(...); idx: the index the kernels were given (None: they searched, checked by check_idx).  The oracle
    then runs with the kernels' index, so a near-tie does not hide the rest."""
    if idx is None:
        check_idx(r["idx"], pts, template, exact)
    else:
        assert np.array_equal(r["idx"], idx)
    tr = trans if trans is not None else np.zeros(3, np.float32)
    want, cache = LO.lbs_forward(pts, template, w, init_a, a, tr, idx=r["idx"])
    _rows_close(r["can"], cache["can_h"][:, :3], POS_TOL, "canonical")
    _rows_close(r["posed"], want, POS_TOL, "posed")
    o_pts, o_a, o_t = LO.lbs_backward(cache, g)
    _rows_close(r["g_pts"], o_pts, GPTS_TOL, "g_pts")
    if np.abs(o_a).max() == 0:
        assert np.array_equal(r["g_a"], np.zeros_like(o_a))
    else:
        _sum_close(r["g_a"], o_a, sum_tol, "g_A")
    assert np.all(r["g_a"][:, 3, :] == 0), "last row of g_A"
    if r["g_trans"] is not None:
        if np.abs(o_t).max() == 0:
            assert np.array_equal(r["g_trans"], np.zeros(3, np.float32))
        else:
            _sum_close(r["g_trans"], o_t, sum_tol, "g_trans")
    return cache


def _points(rng, p, zero_frac=0.0, lo=-1.1, hi=1.1):
    pts = rng.uniform(lo, hi, size=(p, 3)).astype(np.float32)
    pts[rng.random(p) < zero_frac] = 0.0
    return pts


def _interleave(rng, n_live, n_zero):
    """n_live random rows and n_zero exact-zero rows, shuffled: the zero rows straddle every CTA boundary"""
    pts = np.zeros((n_live + n_zero, 3), np.float32)
    pts[rng.permutation(n_live + n_zero)[:n_live]] = rng.uniform(-1.1, 1.1, size=(n_live, 3)).astype(np.float32)
    return pts


def _gauss(rng, p):
    return rng.standard_normal((p, 3)).astype(np.float32)


def _rigid(rng, rot):
    m = np.eye(4, dtype=np.float32)
    m[:3, :3] = rot
    m[:3, 3] = (0.3 * rng.standard_normal(3)).astype(np.float32)
    return m


# ---------------------------------------------------------------------------------------------- nearest search
def live_count_case(dev, n_live, n_zero):
    """The search lists the live rows and puts the origin at entry `count`: with 256 live rows it is alone in a new CTA."""
    rng = np.random.default_rng(1000 + n_live + n_zero)
    template, w, init_a, a, trans = synthetic_rig(11, 1500, 12)
    pts = _interleave(rng, n_live, n_zero)
    g = _gauss(rng, pts.shape[0])
    check_against_oracle(abi_skin(dev, template, w, init_a, a, trans, pts, g), pts, template, w, init_a, a, trans, g)


def template_size_case(dev, vt):
    """Vt around the 1024-vertex tile of the search: one partial tile, exactly one tile, one vertex into the next, three."""
    rng = np.random.default_rng(2000 + vt)
    template, w, init_a, a, trans = synthetic_rig(12, vt, 9)
    pts = _interleave(rng, 257, 300)
    g = _gauss(rng, pts.shape[0])
    check_against_oracle(abi_skin(dev, template, w, init_a, a, trans, pts, g), pts, template, w, init_a, a, trans, g)


def ties_case(dev):
    """Exact duplicate template vertices inside one tile, across the 1023 / 1024 boundary and two tiles apart, the origin
    itself a template vertex (twice): the lowest index wins.  Points exactly on template vertices, and near them."""
    rng = np.random.default_rng(3)
    template, w, init_a, a, trans = synthetic_rig(13, 2200, 12)
    for lo, hi in ((10, 40), (1023, 1024), (500, 2100)):
        template[hi] = template[lo]
    template[600] = 0.0
    template[1800] = 0.0
    on = template[[10, 40, 1023, 1024, 500, 2100, 777, 1500, 2199]]
    near = np.concatenate([template[[10, 1023, 500]] + 1e-3 * rng.standard_normal((3, 3)).astype(np.float32) for _ in range(4)])
    pts = np.concatenate([on, near, np.zeros((300, 3), np.float32), _points(rng, 200)]).astype(np.float32)
    exact = np.zeros(pts.shape[0], bool)
    exact[:on.shape[0] + near.shape[0] + 300] = True
    g = _gauss(rng, pts.shape[0])
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g)
    check_against_oracle(r, pts, template, w, init_a, a, trans, g, exact=exact)
    assert list(r["idx"][:7]) == [10, 10, 1023, 1023, 500, 500, 777]
    assert np.all(r["idx"][on.shape[0] + near.shape[0]:][:300] == 600)


def zero_rows_case(dev, which):
    """all rows zero; no row zero; rows of -0.0 (and mixed signs of zero), which must act like zero rows"""
    rng = np.random.default_rng(4)
    template, w, init_a, a, trans = synthetic_rig(14, 1100, 12)
    if which == "all_zero":
        pts = np.zeros((700, 3), np.float32)
    elif which == "no_zero":
        pts = _points(rng, 700)
    else:
        pts = _interleave(rng, 300, 400)
        z = np.nonzero(~pts.any(1))[0]
        pts[z[::2]] = -0.0
        pts[z[1::4], 1] = -0.0
    g = _gauss(rng, pts.shape[0])
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g)
    check_against_oracle(r, pts, template, w, init_a, a, trans, g, exact=~pts.any(1))
    if which == "neg_zero":
        assert len(set(r["idx"][~pts.any(1)].tolist())) == 1


# ---------------------------------------------------------------------------------------------- blend and inverse
def sparse_weights_case(dev):
    """At most four nonzero weights per row, the rest exactly 0 (as in SMPL-X), and four joints with no weight at all:
    their g_A is exactly 0, like the last row of every g_A[j]."""
    rng = np.random.default_rng(5)
    template, _, init_a, a, trans = synthetic_rig(15, 1300, 24)
    w = np.zeros((1300, 24), np.float32)
    for v in range(1300):
        k = rng.integers(1, 5)
        w[v, rng.choice(20, k, replace=False)] = rng.random(k).astype(np.float32) + 0.05
    w /= w.sum(1, keepdims=True)
    pts = _interleave(rng, 500, 500)
    g = _gauss(rng, pts.shape[0])
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g)
    check_against_oracle(r, pts, template, w, init_a, a, trans, g)
    assert np.all(r["g_a"][20:] == 0) and np.abs(r["g_a"][:20]).max() > 0


def _rot90(k):
    c = [np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]]), np.array([[0, 0, 1], [0, 1, 0], [-1, 0, 0]]),
         np.array([[1, 0, 0], [0, 0, -1], [0, 1, 0]]), np.array([[0, 1, 0], [0, 0, 1], [1, 0, 0]])]
    return c[k % 4].astype(np.float32)


def pivot_case(dev):
    """One-hot weights over init_A of 90-degree rotations: the blended matrices have zeros on the diagonal, so the
    Gauss-Jordan inverse must swap rows."""
    rng = np.random.default_rng(6)
    template, _, _, a, trans = synthetic_rig(16, 900, 12)
    init_a = np.stack([_rigid(rng, _rot90(k)) for k in range(12)])
    w = np.zeros((900, 12), np.float32)
    w[np.arange(900), rng.integers(0, 12, 900)] = 1.0
    pts = _interleave(rng, 400, 200)
    g = _gauss(rng, pts.shape[0])
    check_against_oracle(abi_skin(dev, template, w, init_a, a, trans, pts, g), pts, template, w, init_a, a, trans, g)


def one_joint_case(dev):
    """J = 1: every point moves rigidly, posed = T1 T0^-1 p + trans, in closed form"""
    rng = np.random.default_rng(7)
    template = rng.uniform(-1, 1, size=(300, 3)).astype(np.float32)
    w = np.ones((300, 1), np.float32)
    t0, t1 = _rigid(rng, _rot90(1)), _rigid(rng, _rot90(2) @ _rot90(3))
    trans = np.array([0.1, -0.2, 0.3], np.float32)
    pts = _interleave(rng, 300, 100)
    g = _gauss(rng, pts.shape[0])
    r = abi_skin(dev, template, w, t0[None], t1[None], trans, pts, g)
    m = t1.astype(np.float64) @ np.linalg.inv(t0.astype(np.float64))
    can = pts @ np.linalg.inv(t0.astype(np.float64))[:3, :3].T + np.linalg.inv(t0.astype(np.float64))[:3, 3]
    _rows_close(r["posed"], pts @ m[:3, :3].T + m[:3, 3] + trans, POS_TOL, "posed")
    _rows_close(r["g_pts"], g @ m[:3, :3], GPTS_TOL, "g_pts")
    want_a = np.zeros((4, 4))
    want_a[:3, :3], want_a[:3, 3] = g.astype(np.float64).T @ can, g.sum(0)
    _sum_close(r["g_a"][0], want_a, SUM_TOL, "g_A")
    _sum_close(r["g_trans"], g.astype(np.float64).sum(0), SUM_TOL, "g_trans")


def max_joints_case(dev):
    """J = 128 (kMaxJoints: the joint table fills the blend kernel's shared memory)"""
    rng = np.random.default_rng(8)
    template, w, init_a, a, trans = synthetic_rig(18, 700, 128)
    pts = _interleave(rng, 300, 300)
    g = _gauss(rng, pts.shape[0])
    check_against_oracle(abi_skin(dev, template, w, init_a, a, trans, pts, g), pts, template, w, init_a, a, trans, g)


def joint_count_refused_case(dev):
    L, st = _cabi.lib(), _stream(dev)
    for nj in (0, 129):
        w, a, out, g_a = _buf(dev, (10, max(nj, 1))), _buf(dev, (max(nj, 1), 16)), _buf(dev, (10, 16)), _buf(dev, (max(nj, 1), 16))
        assert L.d3h_lbs_blend(_ptr(w), _ptr(a), 10, nj, 1, _ptr(out), st) == _cabi.D3H_E_BADARG
        assert L.d3h_lbs_blend_backward(_ptr(w), _ptr(out), 10, nj, _ptr(g_a), st) == _cabi.D3H_E_BADARG
    _sync(dev)


# ---------------------------------------------------------------------------------------------- apply and backward
def trans_case(dev, with_trans):
    """trans given / NULL (and then no g_trans either)"""
    rng = np.random.default_rng(9)
    template, w, init_a, a, trans = synthetic_rig(19, 800, 12)
    trans = trans if with_trans else None
    pts = _interleave(rng, 400, 400)
    g = _gauss(rng, pts.shape[0])
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g, g_trans=with_trans)
    check_against_oracle(r, pts, template, w, init_a, a, trans, g)


def forward_inverse_case(dev, seed):
    """b_pose == NULL: canonical points only (lbs_forward_inverse), posed untouched"""
    rng = np.random.default_rng(100 + seed)
    template, w, init_a, _, _ = synthetic_rig(seed, 900, 16)
    pts = _interleave(rng, 500, 300)
    L, st = _cabi.lib(), _stream(dev)
    p, (vt, nj) = pts.shape[0], w.shape
    tw, tia, tm, tp = (_put(dev, x) for x in (w, init_a, template, pts))
    binv = _buf(dev, (vt, 16))
    _cabi.check(L.d3h_lbs_blend(_ptr(tw), _ptr(tia), vt, nj, 1, _ptr(binv), st), "d3h_lbs_blend")
    idx = _buf(dev, (p,), torch.int32)
    nb = int(L.d3h_lbs_nearest_workspace_bytes(p))
    ws = _buf(dev, (max(nb // 4, 16),), torch.int32)
    _cabi.check(L.d3h_lbs_nearest(_ptr(tp), p, _ptr(tm), vt, _ptr(idx), _ptr(ws), nb, st), "d3h_lbs_nearest")
    can = _buf(dev, (p, 3), fill=np.nan)
    _cabi.check(L.d3h_lbs_apply(_ptr(tp), p, _ptr(idx), _ptr(binv), None, None, _ptr(can), None, st), "d3h_lbs_apply")
    _sync(dev)
    got_idx = idx.cpu().numpy()
    check_idx(got_idx, pts, template)
    _rows_close(can.cpu().numpy(), LO.lbs_forward_inverse(pts, template, w, init_a, idx=got_idx), POS_TOL, "canonical")


def _cta_layout(rng, template):
    """1400 rows, CTAs of 256: CTA 0 mixed; CTA 1 zero rows after a live first row; CTAs 2, 3 zero rows only; CTA 4 zero
    rows into mixed; CTA 5 partial.  A few live rows sit next to the origin's nearest vertex, so live-row atomics and
    the CTA sum of the zero rows meet on one table row."""
    pts = _points(rng, 1400, 0.5)
    pts[257:1100] = 0.0
    pts[0] = pts[256] = (0.9, -0.8, 0.7)
    v0 = int(LO.nearest(np.zeros((1, 3), np.float32), template)[0])
    near = [5, 100, 1200, 1399, 260]
    pts[near] = template[v0] + 1e-4 * rng.standard_normal((len(near), 3)).astype(np.float32)
    return pts, v0, near


def cta_boundaries_case(dev, use_pts):
    rng = np.random.default_rng(10)
    template, w, init_a, a, trans = synthetic_rig(20, 1200, 12)
    pts, v0, near = _cta_layout(rng, template)
    g = _gauss(rng, pts.shape[0])
    g[::7] = 0.0                                           # exact-zero upstream rows: exact-zero g_pts rows
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g, use_pts=use_pts)
    check_against_oracle(r, pts, template, w, init_a, a, trans, g)
    assert np.all(r["idx"][near] == v0) and r["idx"][256] != v0
    assert np.all(r["g_pts"][::7] == 0)


def pts_null_matches_case(dev):
    """pts given (zero rows summed per CTA) and pts NULL (twelve atomics per row): the same result"""
    rng = np.random.default_rng(11)
    template, w, init_a, a, trans = synthetic_rig(21, 1200, 12)
    pts, _, _ = _cta_layout(rng, template)
    g = _gauss(rng, pts.shape[0])
    r1 = abi_skin(dev, template, w, init_a, a, trans, pts, g, use_pts=True)
    r0 = abi_skin(dev, template, w, init_a, a, trans, pts, g, use_pts=False)
    assert np.array_equal(r1["g_pts"], r0["g_pts"])
    scale = np.abs(r0["g_b"]).max()
    assert np.abs(r1["g_b"] - r0["g_b"]).max() <= SUM_TOL * scale
    assert np.abs(r1["g_trans"] - r0["g_trans"]).max() <= SUM_TOL * np.abs(r0["g_trans"]).max()


def zero_upstream_case(dev):
    """an all-zero upstream gradient: every gradient exactly 0"""
    rng = np.random.default_rng(12)
    template, w, init_a, a, trans = synthetic_rig(22, 1200, 12)
    pts, _, _ = _cta_layout(rng, template)
    g = np.zeros_like(pts)
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g)
    for k in ("g_pts", "g_a", "g_b", "g_trans"):
        assert np.array_equal(r[k], np.zeros_like(r[k])), k


def mixed_zero_idx_case(dev, use_pts):
    """Zero rows whose idx differ (the header allows any idx): each table row gets its own zero rows' gradients.  600
    zero rows alternating between table rows 3 and 10, a live first row in CTA 1, live rows with their own idx."""
    rng = np.random.default_rng(13)
    template, w, init_a, a, trans = synthetic_rig(23, 300, 8)
    pts = np.zeros((700, 3), np.float32)
    idx = (np.arange(700) % 2 * 7 + 3).astype(np.int32)
    live = [256] + list(range(600, 700))
    pts[live] = rng.uniform(-1.1, 1.1, size=(len(live), 3)).astype(np.float32)
    idx[live] = rng.integers(0, 300, len(live))
    g = _gauss(rng, 700)
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g, use_pts=use_pts, idx=idx)
    cache = check_against_oracle(r, pts, template, w, init_a, a, trans, g, idx=idx)
    want_b = np.zeros((300, 3, 4))
    np.add.at(want_b, idx, g.astype(np.float64)[:, :, None] * cache["can_h"][:, None, :])
    for v in (3, 10):
        _sum_close(r["g_b"][v], want_b[v].reshape(12), SUM_TOL, f"g_b[{v}]")


def empty_case(dev):
    """P = 0 through the ABI: nothing written, zero gradients"""
    template, w, init_a, a, trans = synthetic_rig(24, 200, 6)
    pts, g = np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32)
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g)
    assert r["posed"].shape == (0, 3) and r["g_pts"].shape == (0, 3)
    assert np.array_equal(r["g_a"], np.zeros((6, 4, 4), np.float32)) and np.array_equal(r["g_trans"], np.zeros(3, np.float32))


# ---------------------------------------------------------------------------------------------- the module
def _rig(dev, template, w, init_a):
    from d3human_code_b200.deform.lbs import LinearBlendSkinning
    return LinearBlendSkinning(torch.tensor(template[None], device=dev), torch.tensor(w, device=dev), torch.tensor(init_a[None], device=dev))


def module_case(dev, which):
    rng = np.random.default_rng(15)
    template, w, init_a, a, trans = synthetic_rig(25, 900, 12)
    rig = _rig(dev, template, w, init_a)
    pts = _interleave(rng, 300, 300)
    g = _gauss(rng, pts.shape[0])
    ta = torch.tensor(a, device=dev, requires_grad=which != "a_no_grad")
    tt = torch.tensor(trans.reshape(1, 3), device=dev, requires_grad=True)
    if which == "view_f64":                                 # a strided float64 view: the gradient lands in its layout
        base = torch.zeros((pts.shape[0], 6), dtype=torch.float64, device=dev)
        base[:, ::2] = torch.tensor(pts, dtype=torch.float64, device=dev)
        base.requires_grad_(True)
        tp = base[:, ::2]
        assert not tp.is_contiguous()
    else:
        tp = torch.tensor(pts[None] if which == "batched" else pts, device=dev, requires_grad=True)
    out = rig.lbs_transform(tp, ta, None if which == "no_trans" else tt)
    assert out.shape == (pts.shape[0], 3) and out.dtype == torch.float32
    want, cache = LO.lbs_forward(pts, template, w, init_a, a, np.zeros(3, np.float32) if which == "no_trans" else trans)
    _rows_close(out.detach().cpu().numpy(), want, POS_TOL, "posed")
    (out * torch.tensor(g, device=dev)).sum().backward()
    o_pts, o_a, o_t = LO.lbs_backward(cache, g)
    if which == "view_f64":
        assert base.grad.dtype == torch.float64
        _rows_close(base.grad[:, ::2].cpu().numpy(), o_pts, GPTS_TOL, "g_pts")
        assert np.all(base.grad[:, 1::2].cpu().numpy() == 0)
    else:
        _rows_close(tp.grad.reshape(-1, 3).cpu().numpy(), o_pts, GPTS_TOL, "g_pts")
    if which == "a_no_grad":
        assert ta.grad is None
    else:
        _sum_close(ta.grad.cpu().numpy(), o_a, SUM_TOL, "g_A")
    if which == "no_trans":
        assert tt.grad is None
    else:
        _sum_close(tt.grad.cpu().numpy()[0], o_t, SUM_TOL, "g_trans")


def module_empty_case(dev):
    """P = 0 through the module: an empty result, zero gradients to A and trans"""
    template, w, init_a, a, trans = synthetic_rig(26, 200, 6)
    rig = _rig(dev, template, w, init_a)
    tp = torch.zeros((0, 3), device=dev, requires_grad=True)
    ta = torch.tensor(a, device=dev, requires_grad=True)
    tt = torch.tensor(trans.reshape(1, 3), device=dev, requires_grad=True)
    out = rig.lbs_transform(tp, ta, tt)
    assert out.shape == (0, 3)
    assert rig.lbs_forward_inverse(tp[None]).shape == (1, 0, 3)
    out.sum().backward()
    assert tp.grad.shape == (0, 3)
    assert torch.count_nonzero(ta.grad) == 0 and torch.count_nonzero(tt.grad) == 0


def module_weights_case(dev):
    """interpolate_weights with B = 2 frames: (B,P,J), each frame's rows its nearest vertex's weights"""
    rng = np.random.default_rng(16)
    template, w, init_a, _, _ = synthetic_rig(27, 700, 12)
    rig = _rig(dev, template, w, init_a)
    pts = np.stack([_interleave(rng, 200, 100), _interleave(rng, 250, 50)])
    got = rig.interpolate_weights(torch.tensor(pts, device=dev)).cpu().numpy()
    assert got.shape == (2, 300, 12)
    for b in range(2):
        idx = rig.nearest(torch.tensor(pts[b], device=dev)).cpu().numpy()
        check_idx(idx, pts[b], template, exact=~pts[b].any(1))
        assert np.array_equal(got[b], w[idx])


# ---------------------------------------------------------------------------------------------- the benchmark's shape
def bench_shape_case(dev):
    """230 286 rows, 90 % exact zeros, Vt = 10 475, J = 55 (DESIGN section 10).  The oracle's search runs on the distinct
    rows only."""
    rng = np.random.default_rng(17)
    template, w, init_a, a, trans = synthetic_rig(1, 10475, 55)
    template = (template * 0.9).astype(np.float32)
    pts = _points(rng, 230286, 0.9)
    g = _gauss(rng, pts.shape[0])
    r = abi_skin(dev, template, w, init_a, a, trans, pts, g)
    uniq, inv = np.unique(pts, axis=0, return_inverse=True)
    want_idx = LO.nearest(uniq, template)[inv.reshape(-1)]
    bad = r["idx"] != want_idx
    assert not bad[~pts.any(1)].any()
    if bad.any():
        p64, t64 = pts[bad].astype(np.float64), template.astype(np.float64)
        d_got, d_want = ((p64 - t64[r["idx"][bad]]) ** 2).sum(-1), ((p64 - t64[want_idx[bad]]) ** 2).sum(-1)
        assert np.all(np.abs(d_got - d_want) <= 1e-6 * (1 + d_want)) and bad.mean() < 1e-3
    check_against_oracle(r, pts, template, w, init_a, a, trans, g, idx=r["idx"], sum_tol=BENCH_SUM_TOL)


# ---------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.parametrize("n_zero", [0, 300])
@pytest.mark.parametrize("n_live", [255, 256, 257])
def test_live_row_counts_at_the_cta_edge(dev, n_live, n_zero):
    live_count_case(dev, n_live, n_zero)


@pytest.mark.parametrize("vt", [1, 1023, 1024, 1025, 2500])
def test_template_sizes_at_the_tile_edge(dev, vt):
    template_size_case(dev, vt)


def test_ties_go_to_the_lowest_index(dev):
    ties_case(dev)


@pytest.mark.parametrize("which", ["all_zero", "no_zero", "neg_zero"])
def test_zero_rows(dev, which):
    zero_rows_case(dev, which)


def test_sparse_weights(dev):
    sparse_weights_case(dev)


def test_inverse_swaps_rows(dev):
    pivot_case(dev)


def test_one_joint_is_rigid(dev):
    one_joint_case(dev)


def test_max_joints(dev):
    max_joints_case(dev)


def test_joint_counts_outside_the_table_are_refused(dev):
    joint_count_refused_case(dev)


@pytest.mark.parametrize("with_trans", [True, False])
def test_trans(dev, with_trans):
    trans_case(dev, with_trans)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_forward_inverse(dev, seed):
    forward_inverse_case(dev, seed)


@pytest.mark.parametrize("use_pts", [True, False])
def test_zero_rows_across_cta_boundaries(dev, use_pts):
    cta_boundaries_case(dev, use_pts)


def test_pts_null_gives_the_same_gradients(dev):
    pts_null_matches_case(dev)


def test_zero_upstream_gradient(dev):
    zero_upstream_case(dev)


@pytest.mark.parametrize("use_pts", [True, False])
def test_zero_rows_with_different_idx(dev, use_pts):
    mixed_zero_idx_case(dev, use_pts)


def test_no_points(dev):
    empty_case(dev)


@pytest.mark.parametrize("which", ["no_trans", "a_no_grad", "batched", "view_f64"])
def test_module(module_dev, which):
    module_case(module_dev, which)


def test_module_no_points(module_dev):
    module_empty_case(module_dev)


def test_module_interpolate_weights_of_two_frames(module_dev):
    module_weights_case(module_dev)


def test_benchmark_shape(dev):
    bench_shape_case(dev)
