"""The float64 oracle of the SDF regulariser (oracle/sdf_reg_oracle.py) against a float64 torch restatement of the
reference's `compute_sdf_reg_loss` (geometry/hmsdf.py:162-170) and its autograd; hand-checked tiny cases for every sign
pair; the live reference when a checkout is available; the validation of the one-time table build
(geometry/sdf_reg.py).  CPU only."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from d3human_code_b200 import grids
from d3human_code_b200.geometry import sdf_reg as R
from oracle import ref_loader
from oracle import sdf_reg_oracle as O
from tests import _sdf_reg_util as S


def reference_form(sdf, all_edges):
    """the reference snippet, verbatim but for the name"""
    sdf_f1x6x2 = sdf[all_edges.reshape(-1)].reshape(-1, 2)
    mask = torch.sign(sdf_f1x6x2[..., 0]) != torch.sign(sdf_f1x6x2[..., 1])
    sdf_f1x6x2 = sdf_f1x6x2[mask]
    sdf_diff = F.binary_cross_entropy_with_logits(sdf_f1x6x2[..., 0], (sdf_f1x6x2[..., 1] > 0).float().to(sdf.dtype)) + \
        F.binary_cross_entropy_with_logits(sdf_f1x6x2[..., 1], (sdf_f1x6x2[..., 0] > 0).float().to(sdf.dtype))
    return sdf_diff


def _torch64(sdf_np, e_np, g=1.0):
    s = torch.tensor(np.asarray(sdf_np, np.float32).astype(np.float64), requires_grad=True)
    loss = reference_form(s, torch.as_tensor(e_np))
    if not math.isnan(float(loss.detach())):
        (loss * g).backward()
    grad = s.grad.numpy() if s.grad is not None else np.zeros(s.shape[0])
    return float(loss.detach()), grad


@pytest.mark.parametrize("case", ["kuhn6_capsule", "kuhn5_random", "smplx10", "chain"])
@pytest.mark.parametrize("g", [1.0, -2.5])
def test_oracle_matches_torch_float64(case, g):
    if case.startswith("kuhn"):
        pos, e = S.kuhn_edges(int(case[4]))
        s = S.capsule_field(pos, 7) if "capsule" in case else S.random_field(pos.shape[0], 2)
    elif case == "smplx10":
        gr = grids.smplx_layout_grid(10)
        e = S.generate_edges(torch.from_numpy(gr["f"]), gr["v"].shape[0]).numpy()
        s = S.capsule_field(gr["v"], 5)
    else:
        n, e = S.chain_edges(4, (1, 3))
        s = S.random_field(n, 9)
    want, gwant = _torch64(s, e, g)
    assert abs(O.sdf_reg_loss(s, e) - want) <= 1e-12 * abs(want)
    assert np.abs(O.sdf_reg_grad(s, e, g) - gwant).max() <= 1e-14
    # row order and orientation do not change the result
    perm = np.random.default_rng(0).permutation(e.shape[0])
    assert abs(O.sdf_reg_loss(s, e[perm][:, ::-1]) - want) <= 1e-12 * abs(want)


# every sign pair on one edge (a, b): selected?, loss by hand
_LS = lambda x: min(x, 0.0) - math.log1p(math.exp(-abs(x)))   # noqa: E731
PAIRS = [
    (1.0, -1.0, True), (-1.0, 1.0, True), (0.0, -2.0, True), (0.0, 3.0, True), (-0.0, 0.5, True), (2.0, 0.0, True),
    (0.0, 0.0, False), (0.0, -0.0, False), (-0.0, 0.0, False), (1.0, 2.0, False), (-1.0, -3.0, False),
]


@pytest.mark.parametrize("sa,sb,sel", PAIRS)
def test_every_sign_pair(sa, sb, sel):
    s = np.array([sa, sb], np.float32)
    e = np.array([[0, 1]])
    loss = O.sdf_reg_loss(s, e)
    want_t, _ = _torch64(s, e)
    if not sel:
        assert math.isnan(loss) and math.isnan(want_t)
        assert not O.sdf_reg_grad(s, e).any()
        return
    ta, tb = float(sa > 0), float(sb > 0)
    hand = (1 - tb) * sa - _LS(sa) + (1 - ta) * sb - _LS(sb)
    assert abs(loss - hand) <= 1e-15 and abs(want_t - hand) <= 1e-15
    sig = lambda x: 1 / (1 + math.exp(-x))   # noqa: E731
    assert np.allclose(O.sdf_reg_grad(s, e), [sig(sa) - tb, sig(sb) - ta], rtol=0, atol=1e-15)


def test_self_edge_and_nan():
    s = np.array([1.0, -1.0, np.nan], np.float32)
    assert math.isnan(O.sdf_reg_loss(s, np.array([[0, 0], [1, 1]])))            # self edges: nothing selected
    assert math.isnan(O.sdf_reg_loss(s, np.array([[0, 1], [1, 2]])))            # NaN end point: selected, NaN
    assert O.selected(s, np.array([[0, 1], [1, 2], [2, 2]]))[0].shape[0] == 3     # NaN != NaN


def test_generate_edges_equals_the_reference_construction():
    _, tets = grids.kuhn_grid(4)
    t = torch.from_numpy(tets)
    assert torch.equal(S.generate_edges(t, 125), S.generate_edges_reference(t))


@pytest.mark.reference
def test_live_reference():
    if not ref_loader.reference_available():
        pytest.skip("D3H_REFERENCE_ROOT not set")
    ref = O.load_reference_sdf_reg_loss()
    pos, e = S.kuhn_edges(6)
    s = S.capsule_field(pos, 7)
    st = torch.tensor(s.astype(np.float64), requires_grad=True)
    loss = ref(st, torch.as_tensor(e))
    loss.backward()
    assert abs(float(loss) - O.sdf_reg_loss(s, e)) <= 1e-12 * abs(float(loss))
    assert np.abs(st.grad.numpy() - O.sdf_reg_grad(s, e)).max() <= 1e-14


# ---------------------------------------------------------------------------------------------- table build
def test_table_validation():
    ok = torch.tensor([[0, 1], [1, 2]])
    with pytest.raises(ValueError, match="integer"):
        R.tables_for(ok.float(), 3)
    with pytest.raises(ValueError, match="shape"):
        R.tables_for(torch.tensor([0, 1, 2]), 3)
    with pytest.raises(ValueError, match="shape"):
        R.tables_for(torch.tensor([[0, 1, 2]]), 3)
    with pytest.raises(ValueError, match="outside"):
        R.tables_for(torch.tensor([[0, 1], [-1, 2]]), 3)
    with pytest.raises(ValueError, match="outside"):
        R.tables_for(torch.tensor([[0, 3]]), 3)
    with pytest.raises(ValueError, match="twice"):
        R.tables_for(torch.tensor([[0, 1], [1, 0]]), 3)
    with pytest.raises(ValueError, match="twice"):
        R.tables_for(torch.tensor([[1, 2], [0, 1], [1, 2]]), 3)
    assert R.tables_for(ok.to(torch.int32), 3).n_edges == 2


def test_table_form_follows_the_structure():
    pos, e = S.kuhn_edges(8)
    tab = R.tables_for(torch.as_tensor(e), pos.shape[0])
    assert tab.form == "runs" and tab.n_edges == e.shape[0]
    gr = grids.smplx_layout_grid(12)
    e = S.generate_edges(torch.from_numpy(gr["f"]), gr["v"].shape[0])
    assert R.tables_for(e, gr["v"].shape[0]).form == "rows"
