"""SDF field query on the tensor cores (SURVEY 8f row 3; include/d3h_mlp.h, d3human-code_b200/geometry/mlp.py) against
the float64 oracle (oracle/mlp_oracle.py) and the golden vectors written from the live reference module
(tests/golden/mlp_*.npz).  GPU only (the edge cases of tests/test_zzzzzzzzz_mlp_edges.py also run on the CPU emulation).  Last file of the suite: a new stage must not stop
(-x) the tests of the extraction.

Tolerances.  The reference computes in fp32 (TF32 off, torch default); the kernels use the 3xTF32 split with fp32
accumulation in tensor memory, whose error is that of a re-ordered fp32 sum.  Forward: |y - y_oracle| <= 1e-5 max|y|;
gradients: normwise 5e-5 (the reference's own fp32 backward is 2e-5 away from the float64 oracle, tests/test_mlp_oracle.py).
"""
import ctypes as C
import glob
import os

import numpy as np
import pytest
import torch

from d3human_code_b200 import _cabi
from oracle import mlp_oracle as MO

pytestmark = pytest.mark.gpu
FWD_TOL, GRAD_TOL, GEMM_TOL = 1e-5, 5e-5, 1e-5
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "mlp_*.npz")))


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


# ------------------------------------------------------------------------------------------------ building blocks
@pytest.mark.parametrize("m,k,n,mode", [(128, 64, 256, 0), (1000, 256, 256, 1), (77, 320, 256, 1), (4133, 256, 64, 0),
                                        (300, 256, 256, 2), (129, 32, 128, 0), (20000, 256, 256, 1)])
def test_linear_tensor_core_gemm_matches_float64(dev, m, k, n, mode):
    """d3h_mlp_linear: c = f(a w^T + bias) for the three epilogues, M not a multiple of the 128-row tile, leading
    dimensions larger than the row lengths.  Reference: float64 matmul of the same fp32 inputs."""
    rng = np.random.default_rng(m + k + n + mode)
    lda, ldw, ldc, ldy = k + 8, k + 4, n + 12, n + 4
    a = rng.standard_normal((m, lda)).astype(np.float32)
    w = (rng.standard_normal((n, ldw)) / np.sqrt(k)).astype(np.float32)
    bias = (0.1 * rng.standard_normal(n)).astype(np.float32)
    y = np.abs(rng.standard_normal((m, ldy)) * 0.02).astype(np.float32)
    ta, tw, tb, ty = (torch.tensor(t, device=dev) for t in (a, w, bias, y))
    tc = torch.full((m, ldc), 7.0, device=dev)
    L = _cabi.lib()
    assert L.d3h_mlp_packed_weight_bytes(n, k) == 8 * n * k
    wp = torch.empty(2 * n * k, device=dev)
    _cabi.check(L.d3h_mlp_pack_weight(tw.data_ptr(), ldw, n, k, 0, 0, 0, n, k, wp.data_ptr(), _st(dev)), "d3h_mlp_pack_weight")
    _cabi.check(L.d3h_mlp_linear(ta.data_ptr(), lda, m, k, wp.data_ptr(), n, tb.data_ptr() if mode != 2 else None, mode,
                                 ty.data_ptr() if mode == 2 else None, ldy if mode == 2 else 0, tc.data_ptr(), ldc, _st(dev)),
                "d3h_mlp_linear")
    z = a[:, :k].astype(np.float64) @ w[:, :k].astype(np.float64).T
    if mode != 2:
        z = z + bias
    want = {0: z, 1: MO.softplus(z), 2: z * (1.0 - np.exp(-100.0 * y[:, :n].astype(np.float64)))}[mode]
    got = tc.cpu().numpy()
    assert _rel(got[:, :n], want) < GEMM_TOL, _rel(got[:, :n], want)
    assert (got[:, n:] == 7.0).all()          # nothing written outside the N columns


@pytest.mark.parametrize("m,n,k", [(64, 128, 64), (1000, 256, 256), (4133, 256, 64), (33, 128, 256), (50000, 256, 256)])
def test_wgrad_contraction_over_points_matches_float64(dev, m, n, k):
    """d3h_mlp_wgrad: dw += dz^T a, db += sum dz (accumulating), M not a multiple of the 32-point slice."""
    rng = np.random.default_rng(m + n + k)
    ldz, lda, lddw = n + 4, k + 8, k + 4
    dz = rng.standard_normal((m, ldz)).astype(np.float32)
    a = rng.standard_normal((m, lda)).astype(np.float32)
    tdz, ta = torch.tensor(dz, device=dev), torch.tensor(a, device=dev)
    dw = torch.full((n, lddw), 1.0, device=dev)
    db = torch.full((n,), 2.0, device=dev)
    L = _cabi.lib()
    nbytes = int(L.d3h_mlp_wgrad_workspace_bytes(m, n, k))
    ws = torch.empty(nbytes // 4, device=dev)
    assert L.d3h_mlp_wgrad(tdz.data_ptr(), ldz, ta.data_ptr(), lda, m, n, k, dw.data_ptr(), lddw, db.data_ptr(), ws.data_ptr(),
                           nbytes - 16, _st(dev)) == _cabi.D3H_E_SMALLWS
    _cabi.check(L.d3h_mlp_wgrad(tdz.data_ptr(), ldz, ta.data_ptr(), lda, m, n, k, dw.data_ptr(), lddw, db.data_ptr(),
                                ws.data_ptr(), nbytes, _st(dev)), "d3h_mlp_wgrad")
    want = dz[:, :n].astype(np.float64).T @ a[:, :k].astype(np.float64)
    scale = np.sqrt(m)
    got = dw.cpu().numpy()
    assert np.abs(got[:, :k] - 1.0 - want).max() < 1e-5 * scale * 4, np.abs(got[:, :k] - 1.0 - want).max()
    assert (got[:, k:] == 1.0).all()
    assert np.abs(db.cpu().numpy() - 2.0 - dz[:, :n].astype(np.float64).sum(0)).max() < 1e-5 * scale * 4


def test_embedding_and_head_match_oracle(dev):
    from d3human_code_b200.geometry.embedding import Embedding
    rng = np.random.default_rng(0)
    x = rng.uniform(-1.2, 1.2, size=(1001, 3)).astype(np.float32)
    for n_freq in (1, 6, 8):
        tx = torch.tensor(x, device=dev, requires_grad=True)
        emb = Embedding(3, n_freq)
        y = emb(tx)
        assert y.shape == (1001, emb.out_channels)
        assert np.abs(y.detach().cpu().numpy() - MO.embed(x, n_freq)).max() < 4e-6 * 2 ** n_freq    # argument 2^k x: ulp(2^k)
        g = rng.standard_normal(tuple(y.shape)).astype(np.float32)
        (y * torch.tensor(g, device=dev)).sum().backward()
        assert _rel(tx.grad.cpu().numpy(), MO.embed_backward(x, n_freq, g.astype(np.float64))) < 1e-5
    a = rng.standard_normal((515, 256)).astype(np.float32)
    w, b = rng.standard_normal((3, 256)).astype(np.float32), rng.standard_normal(3).astype(np.float32)
    ta, tw, tb = (torch.tensor(t, device=dev) for t in (a, w, b))
    out = torch.empty((515, 3), device=dev)
    _cabi.check(_cabi.lib().d3h_mlp_head(ta.data_ptr(), 256, 515, 256, tw.data_ptr(), tb.data_ptr(), 3, out.data_ptr(), _st(dev)),
                "d3h_mlp_head")
    assert _rel(out.cpu().numpy(), a.astype(np.float64) @ w.astype(np.float64).T + b) < 3e-6


# ------------------------------------------------------------------------------------------------ the module
def _load_into(net, w, b):
    lin = [m for m in net.net if isinstance(m, torch.nn.Linear)]
    with torch.no_grad():
        for l, wi, bi in zip(lin, w, b):
            l.weight.copy_(torch.tensor(wi))
            l.bias.copy_(torch.tensor(bi))
    return lin


@pytest.mark.parametrize("path", [p for p in GOLDEN if "two_skips" not in p], ids=lambda p: os.path.basename(p)[:-4])
def test_mlp_matches_golden_vectors_of_the_reference(dev, path):
    """Same parameters / inputs as the live reference module produced the goldens with: outputs and every gradient."""
    from d3human_code_b200.geometry.mlp import MLP
    d = np.load(path)
    n_freq, d_hidden, n_hidden, _m = (int(v) for v in d["cfg"])
    skip_in = [int(s) for s in d["skip_in"]]
    n = n_hidden + 2
    net = MLP(n_freq=n_freq, d_hidden=d_hidden, d_out=1, n_hidden=n_hidden, skip_in=skip_in).to(dev)
    lin = _load_into(net, [d[f"w{i}"] for i in range(n)], [d[f"b{i}"] for i in range(n)])
    x = torch.tensor(d["x"], device=dev, requires_grad=True)
    y = net(x)
    assert _rel(y.detach().cpu().numpy(), d["y"]) < FWD_TOL, _rel(y.detach().cpu().numpy(), d["y"])
    (y * torch.tensor(d["gy"], device=dev)).sum().backward()
    errs = {"gx": _rel(x.grad.cpu().numpy(), d["gx"])}
    for i, l in enumerate(lin):
        errs[f"gw{i}"] = _rel(l.weight.grad.cpu().numpy(), d[f"gw{i}"])
        errs[f"gb{i}"] = _rel(l.bias.grad.cpu().numpy(), d[f"gb{i}"])
    assert max(errs.values()) < GRAD_TOL, errs


@pytest.mark.parametrize("seed,m", [(0, 1), (1, 127), (2, 4097), (3, 100000)])
def test_mlp_matches_oracle_on_random_networks(dev, seed, m):
    """The D3-Human configuration (n_freq 6, 256 wide, 6 hidden layers, skip_in [3]; train.py:1622-1625) and variations, at
    batch sizes around the tile size and at the reference's batch_point_num = 100000 (hmsdf.py:187)."""
    from d3human_code_b200.geometry.mlp import MLP
    rng = np.random.default_rng(seed)
    cfg = [dict(n_freq=6, d_hidden=256, n_hidden=6, skip_in=[3]), dict(n_freq=4, d_hidden=128, n_hidden=2, skip_in=[0, 1]),
           dict(n_freq=8, d_hidden=256, n_hidden=1, skip_in=[]), dict(n_freq=6, d_hidden=256, n_hidden=6, skip_in=[3])][seed]
    torch.manual_seed(seed)
    net = MLP(d_out=1, **cfg).to(dev)
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(1.5)
    lin = [mod for mod in net.net if isinstance(mod, torch.nn.Linear)]
    x = rng.uniform(-1, 1, size=(m, 3)).astype(np.float32)
    tx = torch.tensor(x, device=dev, requires_grad=True)
    y = net(tx)
    yo, cache = MO.forward(x, [l.weight.detach().cpu().numpy() for l in lin], [l.bias.detach().cpu().numpy() for l in lin],
                           cfg["n_freq"], tuple(cfg["skip_in"]))
    assert y.shape == (m, 1)
    assert _rel(y.detach().cpu().numpy(), yo) < FWD_TOL, _rel(y.detach().cpu().numpy(), yo)
    gy = rng.standard_normal((m, 1)).astype(np.float32)
    (y * torch.tensor(gy, device=dev)).sum().backward()
    gx, gw, gb = MO.backward(cache, gy)
    errs = {"gx": _rel(tx.grad.cpu().numpy(), gx)}
    for i, l in enumerate(lin):
        errs[f"gw{i}"] = _rel(l.weight.grad.cpu().numpy(), gw[i])
        errs[f"gb{i}"] = _rel(l.bias.grad.cpu().numpy(), gb[i])
    assert max(errs.values()) < GRAD_TOL, errs


def test_mlp_state_dict_is_the_reference_layout_and_feeds_the_extraction(dev):
    """Drop-in: parameter names of the reference module; its output goes straight into hmSDF_Tets and the loss
    back-propagates through the extraction into the network's weights (hmsdf.py:434-455)."""
    from d3human_code_b200 import grids
    from d3human_code_b200.geometry.hmsdf_tets_split import hmSDF_Tets
    from d3human_code_b200.geometry.mlp import MLP
    net = MLP(n_freq=6, d_hidden=256, n_hidden=6, skip_in=[3]).to(dev)
    keys = list(net.state_dict().keys())
    assert keys[:2] == ["net.0.weight", "net.0.bias"] and keys[-2:] == ["net.14.weight", "net.14.bias"] and len(keys) == 16
    assert net.net[8].weight.shape == (256, 256 + 39)
    pos, tets = grids.kuhn_grid(16)
    tp = torch.tensor(pos, device=dev)
    with torch.no_grad():      # bias the output so that the zero level set crosses the grid
        sdf0 = net(tp)
        net.net[14].bias -= sdf0.median()
    sdf = net(tp)
    msdf = torch.tensor(grids.capsule_garment_field(pos)[1], device=dev)
    verts, faces, _, _, _, extra = hmSDF_Tets()(tp, sdf, msdf, torch.tensor(tets, device=dev), "cloth")
    assert faces.shape[0] > 0
    verts.square().sum().backward()
    g = net.net[0].weight.grad
    assert g is not None and torch.isfinite(g).all() and float(g.abs().max()) > 0
    with pytest.raises(NotImplementedError):
        MLP(use_float16=True).to(dev)(tp)


def test_packed_weight_transposed_slice_with_padding(dev):
    """d3h_mlp_pack_weight with transpose / column offset / zero padding (the operands of the input-gradient GEMMs):
    c = a B^T with B[n][k] = w[k][col0 + n] for n < 39, zero up to 64."""
    rng = np.random.default_rng(5)
    m, dh, e, ep = 333, 256, 39, 64
    w = rng.standard_normal((dh, dh + e)).astype(np.float32)
    a = rng.standard_normal((m, dh)).astype(np.float32)
    tw, ta = torch.tensor(w, device=dev), torch.tensor(a, device=dev)
    L = _cabi.lib()
    wp = torch.empty(2 * ep * dh, device=dev)
    _cabi.check(L.d3h_mlp_pack_weight(tw.data_ptr(), dh + e, e, dh, 1, 0, dh, ep, dh, wp.data_ptr(), _st(dev)), "d3h_mlp_pack_weight")
    out = torch.empty((m, ep), device=dev)
    _cabi.check(L.d3h_mlp_linear(ta.data_ptr(), dh, m, dh, wp.data_ptr(), ep, None, 0, None, 0, out.data_ptr(), ep, _st(dev)),
                "d3h_mlp_linear")
    want = a.astype(np.float64) @ w[:, dh:].astype(np.float64)
    got = out.cpu().numpy()
    assert _rel(got[:, :e], want) < GEMM_TOL and (got[:, e:] == 0).all()


def test_packed_weight_cache_follows_in_place_updates_and_new_modules(dev):
    """The operand images of the weights are cached per module on (storage, version): an optimiser step (in-place update)
    must be seen by the next call, and a NEW module whose parameters land on the addresses of a freed one must not find the
    old images (the allocator recycles them at once)."""
    from d3human_code_b200.geometry.mlp import MLP
    rng = np.random.default_rng(11)
    x = rng.uniform(-1, 1, size=(500, 3)).astype(np.float32)
    tx = torch.tensor(x, device=dev)

    def check(net):
        lin = [mod for mod in net.net if isinstance(mod, torch.nn.Linear)]
        y = net(tx)
        yo, _ = MO.forward(x, [l.weight.detach().cpu().numpy() for l in lin], [l.bias.detach().cpu().numpy() for l in lin], 6, (3,))
        assert _rel(y.detach().cpu().numpy(), yo) < FWD_TOL

    for seed in range(3):
        torch.manual_seed(100 + seed)
        net = MLP(n_freq=6, d_hidden=256, n_hidden=6, skip_in=[3]).to(dev)
        check(net)
        check(net)                                   # second call: cache hit
        opt = torch.optim.SGD(net.parameters(), lr=1e-4)
        w_before = net.net[4].weight.detach().clone()
        net(tx).sum().backward()
        opt.step()                                   # in-place update of every weight
        assert not torch.equal(w_before, net.net[4].weight.detach())
        check(net)
        del net, opt


@pytest.mark.parametrize("m,d_out", [(1, 1), (515, 1), (4133, 3), (100000, 1)])
def test_head_backward_matches_float64(dev, m, d_out):
    """d3h_mlp_head_backward: dz = (g w) * softplus'(a), dw += g^T a, db += sum g (accumulating)."""
    rng = np.random.default_rng(m + d_out)
    k, lda, ldz = 256, 260, 264
    a = np.abs(rng.standard_normal((m, lda)) * 0.02).astype(np.float32)
    w = rng.standard_normal((d_out, k)).astype(np.float32)
    g = rng.standard_normal((m, d_out)).astype(np.float32)
    ta, tw, tg = (torch.tensor(t, device=dev) for t in (a, w, g))
    dz = torch.full((m, ldz), 5.0, device=dev)
    dw = torch.full((d_out, k), 1.0, device=dev)
    db = torch.full((d_out,), 2.0, device=dev)
    _cabi.check(_cabi.lib().d3h_mlp_head_backward(ta.data_ptr(), lda, m, k, tw.data_ptr(), d_out, tg.data_ptr(), dz.data_ptr(), ldz,
                                                  dw.data_ptr(), db.data_ptr(), _st(dev)), "d3h_mlp_head_backward")
    a64, g64 = a[:, :k].astype(np.float64), g.astype(np.float64)
    want_dz = (g64 @ w.astype(np.float64)) * (1.0 - np.exp(-100.0 * a64))
    got = dz.cpu().numpy()
    assert _rel(got[:, :k], want_dz) < 1e-5 and (got[:, k:] == 5.0).all()
    assert np.abs(dw.cpu().numpy() - 1.0 - g64.T @ a64).max() < 1e-5 * np.sqrt(m) * 4
    assert np.abs(db.cpu().numpy() - 2.0 - g64.sum(0)).max() < 1e-5 * np.sqrt(m) * 4
