"""The SDF sign-change regulariser (geometry/sdf_reg.py, csrc/d3h_sdf_reg.cu) against the float64 oracle
(oracle/sdf_reg_oracle.py) at the edges its kernels branch on: vertex counts around a multiple of 32 (the last partial
chunk and the spare bitmap word behind it), run-length entry counts around the 256-thread CTA, both table forms, the
selections with no edge, one edge and a NaN, input shapes and dtypes, row order, in-place edits of all_edges, an upstream
gradient other than 1 and the extraction's own edge table.  Each case body takes the device; tests/test_emu_sdf_reg.py
runs the same bodies on the CPU emulation of the kernels at small sizes.

Tolerances: loss relative error 2e-6, gradient 2e-6 of the largest gradient entry.  Largest errors seen on a B200
(1000 W power limit) at the benchmark shape, 128^3 Kuhn lattice and smplx_layout_grid(128) with the capsule field
(M = 38 270 selected edges in both): loss 9.1e-9 relative, gradient 1.8e-7 of the largest entry."""
import math

import numpy as np
import pytest
import torch

from d3human_code_b200 import extract as E
from d3human_code_b200 import grids
from d3human_code_b200.geometry import sdf_reg as R
from oracle import sdf_reg_oracle as O
from tests import _sdf_reg_util as S

pytestmark = pytest.mark.gpu
LOSS_TOL, GRAD_TOL = 2e-6, 2e-6


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture
def module_dev(dev):
    return dev


# ---------------------------------------------------------------------------------------------- helpers
def _edges(dev, e, dtype=torch.int64):
    return torch.as_tensor(np.ascontiguousarray(e)).to(dtype).to(dev)


def run(dev, sdf_np, edges_t, g=1.0, shape="n1", dtype=torch.float32):
    """-> (loss as float, gradient as float64 numpy (N,)) through compute_sdf_reg_loss and autograd"""
    s = torch.as_tensor(np.asarray(sdf_np, dtype=np.float32)).to(dtype)
    s = (s.reshape(-1, 1) if shape == "n1" else s.reshape(-1)).to(dev).requires_grad_()
    loss = R.compute_sdf_reg_loss(s, edges_t)
    assert loss.dim() == 0 and loss.dtype == torch.float32
    (loss * g).backward()
    assert s.grad.shape == s.shape and s.grad.dtype == dtype
    return float(loss.detach().cpu()), s.grad.detach().cpu().double().numpy().reshape(-1)


def check(dev, sdf_np, e_np, edges_t=None, g=1.0, shape="n1", dtype=torch.float32):
    """compare with the oracle; -> (loss relative error, gradient error / max |g|)"""
    if edges_t is None:
        edges_t = _edges(dev, e_np)
    loss, grad = run(dev, sdf_np, edges_t, g, shape, dtype)
    want = O.sdf_reg_loss(sdf_np, e_np)
    gwant = O.sdf_reg_grad(sdf_np, e_np, g)
    if math.isnan(want):
        assert math.isnan(loss), loss
        assert not grad.any()
        return 0.0, 0.0
    lerr = abs(loss - want) / abs(want)
    gerr = float(np.abs(grad - gwant).max() / max(np.abs(gwant).max(), 1e-30))
    assert lerr <= LOSS_TOL, (loss, want, lerr)
    assert gerr <= GRAD_TOL, gerr
    return lerr, gerr


# ---------------------------------------------------------------------------------------------- case bodies
def kuhn_case(dev, res, n, field):
    """Kuhn lattice with n vertices (the edges among the first n; None: all): the run-length table"""
    pos, e = S.kuhn_edges(res, n)
    s = S.capsule_field(pos, zeros_every=11) if field == "capsule" else S.random_field(pos.shape[0], res)
    t = _edges(dev, e)
    assert R.tables_for(t, pos.shape[0]).form == "runs"
    check(dev, s, e, t)


def single_tet_case(dev):
    """one tet, every assignment of {-1, -0.0, +0.0, +1, 2} to its corners that has both signs or a zero"""
    e = np.array([[0, 1], [0, 2], [0, 3], [1, 2], [1, 3], [2, 3]])
    t = _edges(dev, e)
    vals = [-1.0, -0.0, 0.0, 1.0, 2.0]
    rng = np.random.default_rng(0)
    for _ in range(40):
        s = np.array([vals[i] for i in rng.integers(0, len(vals), 4)], dtype=np.float32)
        check(dev, s, e, t)


def entries_case(dev, n_chunks, diffs):
    """a chain with about n_chunks * len(diffs) run-length entries (a difference d >= 32 has none in the last chunk): one
    CTA of the scan full, one short, one over"""
    n, e = S.chain_edges(n_chunks, diffs)
    t = _edges(dev, e)
    tab = R.tables_for(t, n)
    assert tab.form == "runs" and tab.n_runs == np.unique((e[:, 0] >> 5) * n + e[:, 1] - e[:, 0]).shape[0]
    check(dev, S.random_field(n, n_chunks), e, t)


def smplx_case(dev, res):
    """the unstructured SMPL-X layout: the transposed-rows table"""
    g = grids.smplx_layout_grid(res)
    n = g["v"].shape[0]
    e = S.generate_edges(torch.from_numpy(g["f"]), n).numpy()
    t = _edges(dev, e)
    assert R.tables_for(t, n).form == "rows"
    check(dev, S.capsule_field(g["v"], zeros_every=13), e, t)


def m_zero_case(dev, which):
    """no edge selected: NaN loss, zero gradient"""
    pos, e = S.kuhn_edges(3)
    n = pos.shape[0]
    s = {"positive": np.full(n, 0.5), "negative": np.full(n, -0.5), "zero": np.zeros(n)}.get(which)
    if which == "no_edges":
        e = np.zeros((0, 2), np.int64)
        s = S.random_field(n)
    loss, grad = run(dev, s, _edges(dev, e))
    assert math.isnan(loss) and not grad.any()


def m_one_case(dev):
    """exactly one selected edge: the last vertex of a chain has the other sign"""
    n, e = S.chain_edges(3)
    s = np.full(n, 0.25, np.float32)
    s[-1] = -1.5
    assert O.selected(s, e)[0].shape[0] == 1
    check(dev, s, e)


def nan_case(dev):
    """a NaN end point selects its edges: the loss is NaN"""
    pos, e = S.kuhn_edges(4)
    s = S.capsule_field(pos)
    s[37] = np.nan
    loss, _ = run(dev, s, _edges(dev, e))
    assert math.isnan(loss)


def shapes_case(dev):
    """(N,) and (N,1): the same loss and gradient, each in its own shape"""
    pos, e = S.kuhn_edges(5)
    s = S.random_field(pos.shape[0], 3)
    t = _edges(dev, e)
    l1, g1 = run(dev, s, t, shape="n1")
    l2, g2 = run(dev, s, t, shape="n")
    assert l1 == l2
    assert np.array_equal(g1, g2) or np.abs(g1 - g2).max() <= 1e-7 * np.abs(g1).max()


def f64_case(dev):
    """float64 sdf: computed in float32, gradient in float64"""
    pos, e = S.kuhn_edges(5)
    check(dev, S.capsule_field(pos, zeros_every=5), e, dtype=torch.float64)


def swapped_rows_case(dev):
    """rows as (max, min), in another order, and an int32 tensor: the same table, the same loss bits"""
    pos, e = S.kuhn_edges(6)
    s = S.random_field(pos.shape[0], 5)
    l0, _ = run(dev, s, _edges(dev, e))
    perm = np.random.default_rng(1).permutation(e.shape[0])
    l1, _ = run(dev, s, _edges(dev, e[perm][:, ::-1], torch.int32))
    assert l0 == l1
    check(dev, s, e[perm][:, ::-1])


def inplace_case(dev):
    """an in-place edit of all_edges (same address, same shape) builds a new table"""
    pos, e = S.kuhn_edges(5)
    n = pos.shape[0]
    s = S.capsule_field(pos)
    t = _edges(dev, e)
    check(dev, s, e, t)
    e2 = (e + 7) % n              # as many distinct edges, relabelled
    t.copy_(_edges(dev, e2))
    check(dev, s, e2, t)


def upstream_case(dev, g):
    pos, e = S.kuhn_edges(6)
    check(dev, S.capsule_field(pos, zeros_every=9), e, g=g)


def extraction_table_case(dev):
    """all_edges = the extraction's own sorted edge table (extract.build_edge_table, int32)"""
    pos, tets = grids.kuhn_grid(7)
    n = pos.shape[0]
    edge_ab = E.build_edge_table(torch.from_numpy(tets).to(torch.int32).to(dev), n)[1]
    e = edge_ab.cpu().numpy().astype(np.int64)
    assert np.array_equal(e, S.generate_edges(torch.from_numpy(tets), n).numpy())
    check(dev, S.capsule_field(pos, zeros_every=3), e, edge_ab)


def double_backward_case(dev):
    """the backward pass is not differentiable: a second derivative raises"""
    pos, e = S.kuhn_edges(3)
    s = torch.as_tensor(S.random_field(pos.shape[0])).to(dev).requires_grad_()
    w = torch.tensor(2.0, device=dev, requires_grad=True)
    loss = R.compute_sdf_reg_loss(s, _edges(dev, e)) * w
    (gs,) = torch.autograd.grad(loss, s, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gs.sum().backward()


# ---------------------------------------------------------------------------------------------- GPU sizes
@pytest.mark.parametrize("field", ["capsule", "random"])
@pytest.mark.parametrize("res", [30, 31, 32])     # N = 29791 = 32k - 1, 32768 = 32k, 35937 = 32k + 1
def test_kuhn_vertex_counts_around_32(module_dev, res, field):
    kuhn_case(module_dev, res, None, field)


def test_single_tet(module_dev):
    single_tet_case(module_dev)


@pytest.mark.parametrize("n_chunks,diffs", [(255, (1,)), (256, (1,)), (257, (1,)), (128, (1, 40)), (257, (1, 33))])
def test_entry_counts_around_the_cta(module_dev, n_chunks, diffs):
    entries_case(module_dev, n_chunks, diffs)


def test_smplx_layout_takes_the_rows(module_dev):
    smplx_case(module_dev, 24)


@pytest.mark.parametrize("which", ["positive", "negative", "zero", "no_edges"])
def test_no_edge_selected(module_dev, which):
    m_zero_case(module_dev, which)


def test_one_edge_selected(module_dev):
    m_one_case(module_dev)


def test_nan(module_dev):
    nan_case(module_dev)


def test_shapes(module_dev):
    shapes_case(module_dev)


def test_float64(module_dev):
    f64_case(module_dev)


def test_row_order(module_dev):
    swapped_rows_case(module_dev)


def test_inplace_edit(module_dev):
    inplace_case(module_dev)


@pytest.mark.parametrize("g", [3.5, -0.25])
def test_upstream_gradient(module_dev, g):
    upstream_case(module_dev, g)


def test_extraction_edge_table(module_dev):
    extraction_table_case(module_dev)


def test_double_backward_raises(module_dev):
    double_backward_case(module_dev)


# ---------------------------------------------------------------------------------------------- benchmark shape
def _bench_inputs(which):
    if which == "kuhn128":
        pos, tets = grids.kuhn_grid(128)
        n = pos.shape[0]
        e = S.generate_edges(torch.from_numpy(tets).cuda(), n)
        return grids.capsule_garment_field(pos)[0], e, "runs"
    g = grids.smplx_layout_grid(128)
    n = g["v"].shape[0]
    e = S.generate_edges(torch.from_numpy(g["f"]).cuda(), n)
    return grids.capsule_garment_field(g["v"])[0], e, "rows"


@pytest.mark.parametrize("which", ["kuhn128", "smplx128"])
def test_benchmark_shape(dev, which):
    s_np, e, form = _bench_inputs(which)
    assert R.tables_for(e, s_np.shape[0]).form == form
    s = torch.from_numpy(s_np).to(dev).reshape(-1, 1).requires_grad_()
    loss = R.compute_sdf_reg_loss(s, e)
    loss.backward()
    e_np = e.cpu().numpy()
    want, gwant = O.sdf_reg_loss(s_np, e_np), O.sdf_reg_grad(s_np, e_np)
    lerr = abs(loss.item() - want) / abs(want)
    gerr = float(np.abs(s.grad.cpu().double().numpy().reshape(-1) - gwant).max() / np.abs(gwant).max())
    print(f"SDF_REG_ERRORS {which} loss_rel={lerr:.3e} grad_rel_max={gerr:.3e} M={O.selected(s_np, e_np)[0].shape[0]}")
    assert lerr <= LOSS_TOL and gerr <= GRAD_TOL, (lerr, gerr)
    # the same inputs give the same loss bits
    again = R.compute_sdf_reg_loss(s.detach(), e)
    assert again.item() == loss.item()
    # after the first call: forward and backward never wait for the device
    s.grad = None
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        loss = R.compute_sdf_reg_loss(s, e)
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert s.grad is not None
