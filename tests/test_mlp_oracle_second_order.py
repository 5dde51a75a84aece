"""Second derivative of the SDF network (the eikonal term of hmsdf.py:856-880): `second_order` of
tests/_mlp_second_order.py (float64, hand-derived, on the cache of oracle/mlp_oracle.py) against torch float64 double
backward through the same nn.Linear / nn.Softplus chain and against the live reference module, and the argument checks of
the second-derivative entry points of include/d3h_mlp.h.  CPU only."""
import numpy as np
import pytest
import torch
from torch import nn

from d3human_code_b200 import _cabi
from oracle import mlp_oracle as MO
from oracle import ref_loader
from tests import _mlp_second_order as SO


def _nrel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _torch_chain(x, ws, bs, n_freq, skip_in):
    """geometry/embedding.py + geometry/mlp.py as plain torch ops (nn.Softplus(beta=100), default threshold 20)."""
    sp = nn.Softplus(beta=100)
    out = [x]
    for k in range(n_freq):
        out += [torch.sin(2.0 ** k * x), torch.cos(2.0 ** k * x)]
    emb = torch.cat(out, -1)
    h = emb
    n_hidden = len(ws) - 2
    for li in range(len(ws)):
        if 1 <= li <= n_hidden and (li - 1) in skip_in:
            h = torch.cat([h, emb], -1)
        h = nn.functional.linear(h, ws[li], bs[li])
        if li < len(ws) - 1:
            h = sp(h)
    return h


def _torch_second_order(x, ws, bs, n_freq, skip_in, gy, v):
    dt = torch.float64
    tx = torch.tensor(x, dtype=dt, requires_grad=True)
    tw = [torch.tensor(w, dtype=dt, requires_grad=True) for w in ws]
    tb = [torch.tensor(b, dtype=dt, requires_grad=True) for b in bs]
    tgy = torch.tensor(gy, dtype=dt, requires_grad=True)
    y = _torch_chain(tx, tw, tb, n_freq, skip_in)
    gx, = torch.autograd.grad(y, tx, tgy, create_graph=True)
    grads = torch.autograd.grad((gx * torch.tensor(v, dtype=dt)).sum(), [tx, tgy] + tw + tb, allow_unused=True)
    return [None if g is None else g.numpy() for g in grads]


CONFIGS = [   # (n_freq, d_hidden, d_out, n_hidden, skip_in, weight scale, point range)
    (3, 16, 2, 3, (1,), 1.0, 1.0),          # one skip layer
    (4, 24, 1, 4, (0, 2), 1.0, 1.0),        # two skips
    (2, 16, 3, 2, (), 1.0, 1.0),            # d_out 3, no skip
    (6, 32, 1, 6, (3,), 1.5, 1.0),          # the D3-Human layout (narrower)
    (3, 16, 1, 2, (1,), 0.05, 0.02),        # small pre-activations: most of the chain inside the softplus threshold
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=[f"nf{c[0]}_dh{c[1]}_out{c[2]}_nh{c[3]}_skip{'-'.join(map(str, c[4])) or 'none'}_s{c[5]}"
                                              for c in CONFIGS])
def test_second_order_matches_torch_float64_double_backward(cfg):
    n_freq, dh, d_out, nh, skip_in, scale, span = cfg
    rng = np.random.default_rng(sum(cfg[:4]))
    shapes = MO.layer_shapes(n_freq, dh, d_out, nh, skip_in)
    ws = [rng.standard_normal(s) * scale / np.sqrt(s[1]) for s in shapes]
    bs = [0.1 * scale * rng.standard_normal(s[0]) for s in shapes]
    m = 97
    x = rng.uniform(-span, span, size=(m, 3))
    gy, v = rng.standard_normal((m, d_out)), rng.standard_normal((m, 3))
    _, cache = MO.forward(x, ws, bs, n_freq, skip_in)
    pre = np.concatenate([p.ravel() for p in cache["pre"][:-1]]) * MO.BETA
    assert (pre > MO.THRESHOLD).any() or scale < 0.1          # both branches of the threshold are exercised
    assert (np.abs(pre) < MO.THRESHOLD).any()
    gx, gw, gb, ydot = SO.second_order(cache, gy, v)
    ref = _torch_second_order(x, ws, bs, n_freq, skip_in, gy, v)
    n = len(ws)
    assert _nrel(gx, ref[0]) < 1e-10
    assert _nrel(ydot, ref[1]) < 1e-10
    for i in range(n):
        assert gw[i].shape == shapes[i]
        assert _nrel(gw[i], ref[2 + i]) < 1e-10, i
    for i in range(n - 1):
        assert _nrel(gb[i], ref[2 + n + i]) < 1e-10, i
    assert ref[2 + 2 * n - 1] is None and not gb[-1].any()     # the output bias does not enter the gradient


def test_embedding_second_derivative_matches_torch_float64():
    rng = np.random.default_rng(3)
    x, v = rng.uniform(-1.5, 1.5, size=(50, 3)), rng.standard_normal((50, 3))
    n_freq = 5
    g = rng.standard_normal((50, 3 * (2 * n_freq + 1)))
    tx = torch.tensor(x, requires_grad=True)
    tg = torch.tensor(g, requires_grad=True)
    emb = torch.cat([tx] + sum([[torch.sin(2.0 ** k * tx), torch.cos(2.0 ** k * tx)] for k in range(n_freq)], []), -1)
    gx, = torch.autograd.grad(emb, tx, tg, create_graph=True)
    assert _nrel(gx.detach().numpy(), MO.embed_backward(x, n_freq, g)) < 1e-12
    hx, hg = torch.autograd.grad((gx * torch.tensor(v)).sum(), [tx, tg])
    assert _nrel(SO.embed_second_backward(x, n_freq, v, g), hx.numpy()) < 1e-12
    assert _nrel(SO.embed_tangent(x, n_freq, v), hg.numpy()) < 1e-12


@pytest.mark.parametrize("seed", range(3))
def test_second_order_matches_live_reference(seed):
    if not ref_loader.reference_available():
        pytest.skip("needs a checkout of the original project (D3H_REFERENCE_ROOT)")
    ref = ref_loader.load_reference_mlp()
    rng = np.random.default_rng(seed)
    n_freq, d_hidden, n_hidden = int(rng.integers(2, 7)), int(rng.choice([16, 32])), int(rng.integers(2, 6))
    skip_in = sorted(set(int(s) for s in rng.integers(0, n_hidden, size=int(rng.integers(1, 3)))))
    d_out = int(rng.choice([1, 3]))
    torch.manual_seed(seed)
    net = ref.MLP(n_freq=n_freq, d_hidden=d_hidden, d_out=d_out, n_hidden=n_hidden, skip_in=skip_in).double()
    x = torch.tensor(rng.uniform(-1, 1, size=(120, 3)), requires_grad=True)
    y = net(x)
    gy, v = rng.standard_normal(tuple(y.shape)), rng.standard_normal((120, 3))
    gx, = torch.autograd.grad(y, x, torch.tensor(gy), create_graph=True)
    lin = [m for m in net.net if isinstance(m, nn.Linear)]
    params = [l.weight for l in lin] + [l.bias for l in lin]
    got = torch.autograd.grad((gx * torch.tensor(v)).sum(), [x] + params, allow_unused=True)
    _, cache = MO.forward(x.detach().numpy(), [l.weight.detach().numpy() for l in lin], [l.bias.detach().numpy() for l in lin],
                          n_freq, tuple(skip_in))
    hx, gw, gb, _ = SO.second_order(cache, gy, v)
    assert _nrel(hx, got[0].numpy()) < 1e-9
    n = len(lin)
    for i in range(n):
        assert _nrel(gw[i], got[1 + i].numpy()) < 1e-9
        if got[1 + n + i] is not None:
            assert _nrel(gb[i], got[1 + n + i].numpy()) < 1e-9


def test_second_derivative_entry_points_validate_their_arguments():
    """include/d3h_mlp.h: the second-derivative entry points check shapes, alignment and operands before launching."""
    lib = _cabi.lib()
    E = _cabi.D3H_E_BADARG
    buf = np.zeros(4096, dtype=np.float32)
    p = buf.ctypes.data + (-buf.ctypes.data % 16)
    # linear_tangent(a, lda, m, k, w, n, y, ldy, zdot, ldzd, adot, ldad)
    assert lib.d3h_mlp_linear_tangent(p, 64, 0, 64, p, 256, p, 256, p, 256, p, 256, None) == 0          # M = 0
    assert lib.d3h_mlp_linear_tangent(p, 64, 8, 48, p, 256, p, 256, p, 256, p, 256, None) == E          # K % 32
    assert lib.d3h_mlp_linear_tangent(p, 64, 8, 64, p, 96, p, 256, p, 256, p, 256, None) == E           # N
    assert lib.d3h_mlp_linear_tangent(p, 64, 8, 64, p, 256, None, 256, p, 256, p, 256, None) == E       # no y
    assert lib.d3h_mlp_linear_tangent(p, 64, 8, 64, p, 256, p, 256, None, 256, p, 256, None) == E       # no zdot
    assert lib.d3h_mlp_linear_tangent(p, 64, 8, 64, p, 256, p, 256, p, 128, p, 256, None) == E          # zdot too narrow
    assert lib.d3h_mlp_linear_tangent(p, 64, 8, 64, p, 256, p, 256, p + 4, 256, p, 256, None) == E      # alignment
    assert b"d3h_mlp_linear_tangent" in lib.d3h_last_error_string()
    # linear_adjoint(a, lda, m, k, w, n, y, ldy, delta, ldd, zdot, ldzd, c, ldc)
    assert lib.d3h_mlp_linear_adjoint(p, 64, 0, 64, p, 256, p, 256, p, 256, p, 256, p, 256, None) == 0
    assert lib.d3h_mlp_linear_adjoint(p, 64, 8, 64, p, 256, p, 256, None, 256, p, 256, p, 256, None) == E   # no delta
    assert lib.d3h_mlp_linear_adjoint(p, 64, 8, 64, p, 256, p, 256, p, 256, None, 256, p, 256, None) == E   # no zdot
    assert lib.d3h_mlp_linear_adjoint(p, 64, 8, 64, p, 256, p, 254, p, 256, p, 256, p, 256, None) == E      # ldy % 4
    assert lib.d3h_mlp_linear_adjoint(p, 64, 8, 64, p, 256, p, 256, p, 256, p, 256, p + 8, 256, None) == E  # alignment
    assert lib.d3h_mlp_linear_adjoint(p, 30, 8, 32, p, 256, p, 256, p, 256, p, 256, p, 256, None) == E      # lda < K
    assert b"d3h_mlp_linear_adjoint" in lib.d3h_last_error_string()
    # embed_tangent(x, v, m, n_freq, out, ld, n_cols); embed_second_backward(x, v, m, n_freq, gbar, ldbar, g_emb, ld, g_x)
    assert lib.d3h_mlp_embed_tangent(p, p, 0, 6, p, 64, 64, None) == 0
    assert lib.d3h_mlp_embed_tangent(p, p, 8, 6, p, 64, 32, None) == E                 # 39 channels do not fit
    assert lib.d3h_mlp_embed_tangent(p, None, 8, 6, p, 64, 64, None) == E              # no v
    assert lib.d3h_mlp_embed_second_backward(p, p, 0, 6, None, 0, p, 64, p, None) == 0
    assert lib.d3h_mlp_embed_second_backward(p, p, 8, 6, p, 32, p, 64, p, None) == E   # gbar too narrow
    assert lib.d3h_mlp_embed_second_backward(p, p, 8, 6, None, 0, None, 64, p, None) == E   # no g_emb
    assert lib.d3h_mlp_embed_second_backward(p, p, 8, 17, None, 0, p, 256, p, None) == E    # n_freq > 16
    # head_second_backward(adot, ldad, a, lda, delta, ldd, zdot, ldzd, m, k, g, d_out, dw, mu, ldmu)
    assert lib.d3h_mlp_head_second_backward(p, 256, p, 256, p, 256, p, 256, 0, 256, p, 1, p, p, 256, None) == 0
    assert lib.d3h_mlp_head_second_backward(p, 256, p, 256, p, 256, p, 256, 8, 256, p, 9, p, p, 256, None) == E   # d_out > 8
    assert lib.d3h_mlp_head_second_backward(p, 256, p, 256, p, 256, p, 256, 8, 260, p, 1, p, p, 260, None) == E   # K > 256
    assert lib.d3h_mlp_head_second_backward(p, 256, p, 256, None, 256, p, 256, 8, 256, p, 1, p, p, 256, None) == E  # no delta
    assert lib.d3h_mlp_head_second_backward(p, 256, p, 256, p, 256, p, 256, 8, 256, p, 1, p, p + 4, 256, None) == E  # alignment
    assert lib.d3h_mlp_head_second_backward(p, 256, p, 256, p, 256, p, 256, 8, 256, p, 1, None, p, 256, None) == E  # no dw
    assert b"d3h_mlp_head_second_backward" in lib.d3h_last_error_string()
