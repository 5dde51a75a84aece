"""The SDF-MLP oracle (oracle/mlp_oracle.py, float64) against the golden vectors written from the live reference
(`geometry/mlp.py`, fp32) and against the live reference itself (build container only)."""
import glob
import os

import numpy as np
import pytest

from oracle import mlp_oracle as MO
from oracle import ref_loader

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "mlp_*.npz")))
FWD_TOL = 2e-6      # fp32 reference vs float64 oracle, relative to max |y|
GRAD_TOL = 2e-5     # normwise, gradients


def _params(d):
    n = len([k for k in d.files if k.startswith("w")])
    return [d[f"w{i}"] for i in range(n)], [d[f"b{i}"] for i in range(n)]


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_reproduces_golden_vectors(path):
    d = np.load(path)
    n_freq = int(d["cfg"][0])
    w, b = _params(d)
    y, cache = MO.forward(d["x"], w, b, n_freq, tuple(int(s) for s in d["skip_in"]))
    assert _rel(y, d["y"]) < FWD_TOL
    gx, gw, gb = MO.backward(cache, d["gy"])
    assert _rel(gx, d["gx"]) < GRAD_TOL
    for i in range(len(w)):
        assert gw[i].shape == d[f"gw{i}"].shape
        assert _rel(gw[i], d[f"gw{i}"]) < GRAD_TOL and _rel(gb[i], d[f"gb{i}"]) < GRAD_TOL


def test_layer_shapes_match_the_reference_module():
    if not ref_loader.reference_available():
        pytest.skip("needs a checkout of the original project (D3H_REFERENCE_ROOT)")
    import torch
    ref = ref_loader.load_reference_mlp()
    for cfg in (dict(n_freq=6, d_hidden=256, n_hidden=6, skip_in=[3]), dict(), dict(n_freq=3, d_hidden=32, n_hidden=2, skip_in=[0, 1])):
        net = ref.MLP(**cfg)
        lin = [tuple(m.weight.shape) for m in net.net if isinstance(m, torch.nn.Linear)]
        assert lin == MO.layer_shapes(cfg.get("n_freq", 6), cfg.get("d_hidden", 128), 1, cfg.get("n_hidden", 3), tuple(cfg.get("skip_in", [])))


@pytest.mark.parametrize("seed", range(6))
def test_oracle_matches_live_reference(seed):
    if not ref_loader.reference_available():
        pytest.skip("needs a checkout of the original project (D3H_REFERENCE_ROOT)")
    import torch
    ref = ref_loader.load_reference_mlp()
    rng = np.random.default_rng(seed)
    n_freq, d_hidden, n_hidden = int(rng.integers(1, 8)), int(rng.choice([16, 64, 96])), int(rng.integers(1, 7))
    skip_in = sorted(set(int(s) for s in rng.integers(0, n_hidden, size=int(rng.integers(0, 3)))))
    d_out = int(rng.choice([1, 3]))
    torch.manual_seed(seed)
    net = ref.MLP(n_freq=n_freq, d_hidden=d_hidden, d_out=d_out, n_hidden=n_hidden, skip_in=skip_in)
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(float(rng.uniform(0.5, 3.0)))
    x = torch.tensor(rng.uniform(-1.5, 1.5, size=(200, 3)).astype(np.float32), requires_grad=True)
    y = net(x)
    gy = torch.tensor(rng.standard_normal(tuple(y.shape)).astype(np.float32))
    (y * gy).sum().backward()
    lin = [m for m in net.net if isinstance(m, torch.nn.Linear)]
    yo, cache = MO.forward(x.detach().numpy(), [l.weight.detach().numpy() for l in lin], [l.bias.detach().numpy() for l in lin],
                           n_freq, tuple(skip_in))
    assert _rel(yo, y.detach().numpy()) < 5 * FWD_TOL
    gx, gw, gb = MO.backward(cache, gy.numpy())
    assert _rel(gx, x.grad.numpy()) < 5 * GRAD_TOL
    for i, l in enumerate(lin):
        assert _rel(gw[i], l.weight.grad.numpy()) < 5 * GRAD_TOL and _rel(gb[i], l.bias.grad.numpy()) < 5 * GRAD_TOL
