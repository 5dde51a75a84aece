"""Second derivative of the SDF network on the tensor cores (the eikonal term of hmsdf.py:856-880:
autograd.grad(sdf, x, create_graph=True), then a loss on that gradient): the kernels of include/d3h_mlp.h, "Second
derivative", against float64, and MLP / Embedding double backward against the float64 `second_order` of
tests/_mlp_second_order.py.  GPU only.

Tolerances as tests/test_zzzzzz_mlp.py; the double backward through the whole network is held to 1e-4 normwise (torch fp32
itself is ~1e-6 to 3e-6 away from float64 on these networks)."""
import numpy as np
import pytest
import torch

from d3human_code_b200 import _cabi
from oracle import mlp_oracle as MO
from tests import _mlp_second_order as SO

pytestmark = pytest.mark.gpu
GEMM_TOL, SO_TOL = 1e-5, 1e-4
D3H = dict(n_freq=6, d_hidden=256, n_hidden=6, skip_in=[3])
CFGS = {"d3human": D3H, "d128": dict(n_freq=6, d_hidden=128, n_hidden=4, skip_in=[2]),
        "two_skips": dict(n_freq=4, d_hidden=128, n_hidden=3, skip_in=[0, 2])}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _st(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _nrel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _np(t):
    return t.detach().cpu().numpy()


def _curv(y):
    return np.where(100.0 * y <= 20.0, 100.0 * np.exp(-100.0 * y), 0.0)


# ------------------------------------------------------------------------------------------------ building blocks
@pytest.mark.parametrize("m,k,n", [(1, 64, 256), (300, 256, 256), (77, 320, 128), (4133, 256, 64), (20000, 256, 256)])
def test_linear_tangent_and_adjoint_epilogues_match_float64(dev, m, k, n):
    """d3h_mlp_linear_tangent: zdot = a B^T, adot = zdot softplus'(y); d3h_mlp_linear_adjoint: c = (a B^T) softplus'(y) +
    beta [beta y <= 20] exp(-beta y) delta zdot.  y spans both sides of the softplus threshold; leading dimensions larger
    than the rows; nothing is written outside the N columns."""
    rng = np.random.default_rng(m + k + n)
    lda, ldw, ldy, ldd, ldz, ldc = k + 8, k + 4, n + 4, n + 8, n + 12, n + 16
    a = rng.standard_normal((m, lda)).astype(np.float32)
    w = (rng.standard_normal((n, ldw)) / np.sqrt(k)).astype(np.float32)
    y = rng.uniform(0.0, 0.4, size=(m, ldy)).astype(np.float32)
    d = rng.standard_normal((m, ldd)).astype(np.float32)
    zd = rng.standard_normal((m, ldz)).astype(np.float32)
    ta, tw, ty, td, tzd = (torch.tensor(t, device=dev) for t in (a, w, y, d, zd))
    L = _cabi.lib()
    wp = torch.empty(2 * n * k, device=dev)
    _cabi.check(L.d3h_mlp_pack_weight(tw.data_ptr(), ldw, n, k, 0, 0, 0, n, k, wp.data_ptr(), _st(dev)), "d3h_mlp_pack_weight")
    z_out = torch.full((m, ldz), 7.0, device=dev)
    a_out = torch.full((m, ldc), 7.0, device=dev)
    _cabi.check(L.d3h_mlp_linear_tangent(ta.data_ptr(), lda, m, k, wp.data_ptr(), n, ty.data_ptr(), ldy, z_out.data_ptr(), ldz,
                                         a_out.data_ptr(), ldc, _st(dev)), "d3h_mlp_linear_tangent")
    c_out = torch.full((m, ldc), 7.0, device=dev)
    _cabi.check(L.d3h_mlp_linear_adjoint(ta.data_ptr(), lda, m, k, wp.data_ptr(), n, ty.data_ptr(), ldy, td.data_ptr(), ldd,
                                         tzd.data_ptr(), ldz, c_out.data_ptr(), ldc, _st(dev)), "d3h_mlp_linear_adjoint")
    z = a[:, :k].astype(np.float64) @ w[:, :k].astype(np.float64).T
    y64 = y[:, :n].astype(np.float64)
    spd = 1.0 - np.exp(-100.0 * y64)
    got_z, got_a, got_c = _np(z_out), _np(a_out), _np(c_out)
    assert _rel(got_z[:, :n], z) < GEMM_TOL and (got_z[:, n:] == 7.0).all()
    assert _rel(got_a[:, :n], z * spd) < GEMM_TOL and (got_a[:, n:] == 7.0).all()
    want_c = z * spd + _curv(y64) * d[:, :n].astype(np.float64) * zd[:, :n].astype(np.float64)
    assert _rel(got_c[:, :n], want_c) < GEMM_TOL and (got_c[:, n:] == 7.0).all()


@pytest.mark.parametrize("n_freq,ld,n_cols", [(6, 64, 64), (6, 320, 64), (1, 12, 9), (8, 64, 51)])
def test_embedding_tangent_and_second_backward_match_float64(dev, n_freq, ld, n_cols):
    rng = np.random.default_rng(n_freq + ld)
    m = 1001
    e = 3 * (2 * n_freq + 1)
    x = rng.uniform(-1.2, 1.2, size=(m, 3)).astype(np.float32)
    v = rng.standard_normal((m, 3)).astype(np.float32)
    g = rng.standard_normal((m, ld)).astype(np.float32)
    gbar = rng.standard_normal((m, ld)).astype(np.float32)
    tx, tv, tg, tgb = (torch.tensor(t, device=dev) for t in (x, v, g, gbar))
    L = _cabi.lib()
    out = torch.full((m, ld), 7.0, device=dev)
    _cabi.check(L.d3h_mlp_embed_tangent(tx.data_ptr(), tv.data_ptr(), m, n_freq, out.data_ptr(), ld, n_cols, _st(dev)),
                "d3h_mlp_embed_tangent")
    got = _np(out)
    want = SO.embed_tangent(x, n_freq, v)
    assert np.abs(got[:, :e] - want).max() < 4e-6 * 2 ** n_freq * max(np.abs(want).max(), 1.0)
    assert (got[:, e:n_cols] == 0).all() and (got[:, n_cols:] == 7.0).all()
    g64, gb64 = g[:, :e].astype(np.float64), gbar[:, :e].astype(np.float64)
    for with_bar in (True, False):
        hx = torch.empty((m, 3), device=dev)
        _cabi.check(L.d3h_mlp_embed_second_backward(tx.data_ptr(), tv.data_ptr(), m, n_freq, tgb.data_ptr() if with_bar else None,
                                                    ld, tg.data_ptr(), ld, hx.data_ptr(), _st(dev)), "d3h_mlp_embed_second_backward")
        want = SO.embed_second_backward(x, n_freq, v, g64) + (MO.embed_backward(x, n_freq, gb64) if with_bar else 0.0)
        assert _rel(_np(hx), want) < 4e-6 * 2 ** n_freq, (with_bar, _rel(_np(hx), want))


@pytest.mark.parametrize("m,d_out", [(1, 1), (515, 1), (4133, 3), (100000, 1)])
def test_head_second_backward_matches_float64(dev, m, d_out):
    """d3h_mlp_head_second_backward: dw += g^T adot (accumulating), mu = beta [beta a <= 20] exp(-beta a) delta zdot."""
    rng = np.random.default_rng(m + 7 * d_out)
    k, ld = 256, 260
    adot = rng.standard_normal((m, ld)).astype(np.float32)
    a = rng.uniform(0.0, 0.4, size=(m, ld)).astype(np.float32)
    dl = rng.standard_normal((m, ld)).astype(np.float32)
    zd = rng.standard_normal((m, ld)).astype(np.float32)
    g = rng.standard_normal((m, d_out)).astype(np.float32)
    tad, ta, tdl, tzd, tg = (torch.tensor(t, device=dev) for t in (adot, a, dl, zd, g))
    dw = torch.full((d_out, k), 1.0, device=dev)
    mu = torch.full((m, 264), 5.0, device=dev)
    _cabi.check(_cabi.lib().d3h_mlp_head_second_backward(tad.data_ptr(), ld, ta.data_ptr(), ld, tdl.data_ptr(), ld, tzd.data_ptr(),
                                                         ld, m, k, tg.data_ptr(), d_out, dw.data_ptr(), mu.data_ptr(), 264,
                                                         _st(dev)), "d3h_mlp_head_second_backward")
    want_mu = _curv(a[:, :k].astype(np.float64)) * dl[:, :k] * zd[:, :k]
    got = _np(mu)
    assert _rel(got[:, :k], want_mu) < 1e-5 and (got[:, k:] == 5.0).all()
    want_dw = g.astype(np.float64).T @ adot[:, :k].astype(np.float64)
    assert np.abs(_np(dw) - 1.0 - want_dw).max() < 1e-5 * np.sqrt(m) * 4


# ------------------------------------------------------------------------------------------------ the modules
def _net(dev, cfg, seed, d_out=1):
    from d3human_code_b200.geometry.mlp import MLP
    torch.manual_seed(seed)
    net = MLP(d_out=d_out, **cfg).to(dev)
    lin = [mod for mod in net.net if isinstance(mod, torch.nn.Linear)]
    return net, lin


def _oracle_cache(x, lin, cfg):
    return MO.forward(x, [_np(l.weight) for l in lin], [_np(l.bias) for l in lin], cfg["n_freq"], tuple(cfg["skip_in"]))


@pytest.mark.parametrize("m", [1, 127, 4097, 100000])
@pytest.mark.parametrize("name", list(CFGS))
def test_mlp_eikonal_plus_first_order_loss_matches_oracle(dev, name, m):
    """The training step of hmsdf.py:856-880: gx = autograd.grad(sdf, x, ones, create_graph=True), loss = a first-order
    term on sdf + the eikonal term ((|gx| - 1)^2).mean(), loss.backward().  Gradients on x and every parameter against
    backward + second_order of the float64 oracle; the output bias gets the first-order share only."""
    cfg = CFGS[name]
    net, lin = _net(dev, cfg, seed=m)
    rng = np.random.default_rng(m)
    x = rng.uniform(-1, 1, size=(m, 3)).astype(np.float32)
    g1 = rng.standard_normal((m, 1)).astype(np.float32)
    tx = torch.tensor(x, device=dev, requires_grad=True)
    y = net(tx)
    gx, = torch.autograd.grad(y, tx, torch.ones_like(y), create_graph=True)
    assert gx.requires_grad and gx.grad_fn is not None
    eik = ((gx.norm(dim=-1) - 1.0) ** 2).mean()
    ((y * torch.tensor(g1, device=dev)).sum() + eik).backward()

    yo, cache = _oracle_cache(x, lin, cfg)
    ones = np.ones((m, 1))
    gx_o, _, _ = MO.backward(cache, ones)
    assert _nrel(_np(gx), gx_o) < SO_TOL
    nrm = np.linalg.norm(gx_o, axis=-1, keepdims=True)
    v = 2.0 * (nrm - 1.0) * gx_o / nrm / m
    hx, hw, hb, _ = SO.second_order(cache, ones, v)
    fx, fw, fb = MO.backward(cache, g1)
    errs = {"x": _nrel(_np(tx.grad), hx + fx)}
    for i, l in enumerate(lin):
        errs[f"w{i}"] = _nrel(_np(l.weight.grad), hw[i] + fw[i])
        errs[f"b{i}"] = _nrel(_np(l.bias.grad), hb[i] + fb[i])
    assert max(errs.values()) < SO_TOL, errs


def test_mlp_eikonal_alone_leaves_output_bias_without_gradient_and_takes_a_differentiable_upstream(dev):
    """torch semantics of the double backward: the output bias does not enter gx (its .grad stays None), and an upstream
    gy that itself requires grad receives ydot = J(x) v."""
    cfg = dict(n_freq=6, d_hidden=256, n_hidden=3, skip_in=[1])
    net, lin = _net(dev, cfg, seed=5, d_out=2)
    rng = np.random.default_rng(5)
    m = 777
    x = rng.uniform(-1, 1, size=(m, 3)).astype(np.float32)
    gy = rng.standard_normal((m, 2)).astype(np.float32)
    v = rng.standard_normal((m, 3)).astype(np.float32)
    tx = torch.tensor(x, device=dev, requires_grad=True)
    tgy = torch.tensor(gy, device=dev, requires_grad=True)
    gx, = torch.autograd.grad(net(tx), tx, tgy, create_graph=True)
    (gx * torch.tensor(v, device=dev)).sum().backward()
    assert lin[-1].bias.grad is None
    _, cache = _oracle_cache(x, lin, cfg)
    hx, hw, hb, ydot = SO.second_order(cache, gy, v)
    assert _nrel(_np(tx.grad), hx) < SO_TOL and _nrel(_np(tgy.grad), ydot) < SO_TOL
    for i, l in enumerate(lin):
        assert _nrel(_np(l.weight.grad), hw[i]) < SO_TOL, i
        if i < len(lin) - 1:
            assert _nrel(_np(l.bias.grad), hb[i]) < SO_TOL, i


def test_embedding_double_backward_matches_oracle(dev):
    from d3human_code_b200.geometry.embedding import Embedding
    rng = np.random.default_rng(1)
    for n_freq in (1, 6, 8):
        m, c = 1001, 3 * (2 * n_freq + 1)
        x = rng.uniform(-1.2, 1.2, size=(m, 3)).astype(np.float32)
        g = rng.standard_normal((m, c)).astype(np.float32)
        v = rng.standard_normal((m, 3)).astype(np.float32)
        tx = torch.tensor(x, device=dev, requires_grad=True)
        tg = torch.tensor(g, device=dev, requires_grad=True)
        gx, = torch.autograd.grad(Embedding(3, n_freq)(tx), tx, tg, create_graph=True)
        assert gx.requires_grad
        (gx * torch.tensor(v, device=dev)).sum().backward()
        tol = 4e-6 * 2 ** n_freq
        assert _rel(_np(gx), MO.embed_backward(x, n_freq, g.astype(np.float64))) < tol
        assert _rel(_np(tx.grad), SO.embed_second_backward(x, n_freq, v, g.astype(np.float64))) < tol
        assert _rel(_np(tg.grad), SO.embed_tangent(x, n_freq, v)) < tol


def test_unsupported_derivatives_raise(dev):
    from d3human_code_b200.geometry.embedding import Embedding
    net, lin = _net(dev, D3H, seed=2)
    tx = torch.rand(300, 3, device=dev, requires_grad=True)
    # a loss on the first-order weight gradients
    gw, = torch.autograd.grad(net(tx).sum(), lin[2].weight, create_graph=True)
    with pytest.raises(NotImplementedError):
        gw.square().sum().backward()
    # a third derivative of the network
    gx, = torch.autograd.grad(net(tx).sum(), tx, create_graph=True)
    with pytest.raises(NotImplementedError):
        torch.autograd.grad(gx.square().sum(), tx, create_graph=True)
    # ... and of the encoding
    gx, = torch.autograd.grad(Embedding(3, 6)(tx).sum(), tx, create_graph=True)
    with pytest.raises(NotImplementedError):
        torch.autograd.grad(gx.square().sum(), tx, create_graph=True)


def test_launch_counts(dev):
    """The first-order pass enqueues what it always did; the double backward adds its own kernels on top."""
    from d3human_code_b200.geometry import mlp as M
    net, _ = _net(dev, D3H, seed=3)
    tx = torch.rand(1000, 3, device=dev, requires_grad=True)
    nh, ns = 6, 1
    fwd = 2 + 2 * (nh + 1) + ns
    bwd = 2 + 3 * (nh + 1) + nh + 3 * ns + 2
    l0 = M.launch_counter()
    net(tx).sum().backward()
    assert M.launch_counter() - l0 == fwd + bwd
    l0 = M.launch_counter()
    gx, = torch.autograd.grad(net(tx).sum(), tx, create_graph=True)
    assert M.launch_counter() - l0 == fwd + bwd
    gx.square().sum().backward()
    second = (1 + ns) + (nh + 1) + 1 + 4 * (nh + 1) + 4 * ns + (1 + ns) + nh + 1
    assert M.launch_counter() - l0 == fwd + bwd + second


def test_extraction_loss_plus_eikonal_in_one_backward_is_the_sum_of_both(dev):
    """MLP -> hmSDF_Tets (hmsdf.py:434-455) plus the eikonal term on the same network in one backward pass gives the sum of
    the gradients of the two losses back-propagated separately."""
    from d3human_code_b200 import grids
    from d3human_code_b200.geometry.hmsdf_tets_split import hmSDF_Tets
    pos, tets = grids.kuhn_grid(16)
    msdf = torch.tensor(grids.capsule_garment_field(pos)[1], device=dev)
    tt = torch.tensor(tets, device=dev)
    net, lin = _net(dev, D3H, seed=4)
    with torch.no_grad():      # bias the output so that the zero level set crosses the grid
        net.net[14].bias -= net(torch.tensor(pos, device=dev)).median()
    params = [p for l in lin for p in (l.weight, l.bias)]

    def losses(which):
        tp = torch.tensor(pos, device=dev, requires_grad=True)
        sdf = net(tp)
        out = []
        if "ext" in which:
            verts = hmSDF_Tets()(tp, sdf, msdf, tt, "cloth")[0]
            assert verts.shape[0] > 0
            out.append(verts.square().sum())
        if "eik" in which:
            gx, = torch.autograd.grad(sdf, tp, torch.ones_like(sdf), create_graph=True)
            out.append(((gx.norm(dim=-1) - 1.0) ** 2).mean())
        for p in params:
            p.grad = None
        sum(out).backward()
        return [torch.zeros_like(tp) if tp.grad is None else tp.grad.clone()] + \
               [torch.zeros_like(p) if p.grad is None else p.grad.clone() for p in params]

    both, ext, eik = losses(("ext", "eik")), losses(("ext",)), losses(("eik",))
    assert float(eik[1].abs().max()) > 0 and float(ext[1].abs().max()) > 0
    for i, (b, e1, e2) in enumerate(zip(both, ext, eik)):
        assert _nrel(_np(b), _np(e1 + e2)) < 1e-5, i
