"""SDF network kernels (include/d3h_mlp.h, csrc/d3h_mlp.cu) at the edges they branch on, against float64 (numpy,
oracle/mlp_oracle.py, tests/_mlp_second_order.py): every epilogue of the tensor-core GEMM with N = 192 (three 32-column
loads per epilogue half), odd slice counts (the second register set of the producers' two-slice pipeline on the last
slice), K = 384 (the skip layer of a 128-wide encoding), rows at and past M left untouched; the packed weight image with
offsets, transposition and zero fill; the contraction over points around the 512-point range boundary; every output
width 1..8 of the output layer with K < 256 (idle threads); both forward paths of the encoding up to n_freq = 16; the
modules with a 128-wide encoding, n_freq = 0 and skip layers at the first and the last hidden layer.  Each case body takes
the device; tests/test_emu_mlp.py runs the same bodies on the CPU emulation of the kernels at small sizes.

Tolerances are those of tests/test_zzzzzz_mlp.py and tests/test_zzzzzzzz_mlp_second_order.py: GEMM outputs 1e-5 of the
largest entry, module outputs 1e-5 and gradients 5e-5 (max-relative), second order 1e-4 normwise plus the change that
fp32-level errors of the pre-activations cause in the float64 result (_pre_activation_sensitivity: softplus'' with
beta = 100 is that sensitive where one point and a 128-wide encoding leave few units to carry the result).  The encoding is
checked element by element against the float64 value with an error bound of its fp32 evaluation: 4e-6 times the same
sum taken over absolute values (its arguments 2^k x are exact, so n_freq does not widen the bound)."""
import numpy as np
import pytest
import torch

from d3human_code_b200 import _cabi
from oracle import mlp_oracle as MO
from tests import _mlp_second_order as SO

pytestmark = pytest.mark.gpu
GEMM_TOL, FWD_TOL, GRAD_TOL, SO_TOL, ENC_TOL = 1e-5, 1e-5, 5e-5, 1e-4, 4e-6
SENTINEL = 7.0


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture
def module_dev(dev):
    return dev


# ---------------------------------------------------------------------------------------------- helpers
def _st(dev):
    return torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else None


def _buf(dev, shape, fill=SENTINEL):
    """a 16-byte aligned float32 buffer (the GEMM operands need it; CPU tensors are not always 16-byte aligned)"""
    n = int(np.prod(shape))
    b = torch.full((n + 16,), fill, dtype=torch.float32, device=dev)
    off = (-b.data_ptr() % 16) // 4
    return b[off:off + n].view(shape)


def _put(dev, arr):
    t = _buf(dev, np.shape(arr))
    t.copy_(torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float32)))
    return t


def _np(t):
    return t.detach().cpu().numpy()


def _f64(a):
    return np.asarray(a, dtype=np.float64)


def _rel(a, b):
    a, b = _f64(a), _f64(b)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _nrel(a, b):
    a, b = _f64(a), _f64(b)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _spd(y):
    return 1.0 - np.exp(-100.0 * y)


def _curv(y):
    return np.where(100.0 * y <= 20.0, 100.0 * np.exp(-100.0 * y), 0.0)


def _pack(dev, w, ldw, n_valid, k_valid, transpose, row0, col0, n_pad, k_pad):
    L = _cabi.lib()
    wp = _buf(dev, (2 * n_pad * k_pad,))
    _cabi.check(L.d3h_mlp_pack_weight(w.data_ptr(), ldw, n_valid, k_valid, transpose, row0, col0, n_pad, k_pad, wp.data_ptr(),
                                      _st(dev)), "d3h_mlp_pack_weight")
    return wp


# ---------------------------------------------------------------------------------------------- linear: five epilogues
EPILOGUES = ("mode0", "mode1", "mode2", "tangent", "adjoint")


def linear_case(dev, m, n, k, epi):
    """One GEMM c = f(a w^T [+ bias]) with the epilogue `epi`; leading dimensions larger than the rows; three sentinel rows
    after M and sentinel columns after N in every output.  Columns [0, n/4) put the pre-activation on beta z = 20 +- 0.3,
    columns [n/4, n/2) on e^{beta z} = 2^-12 (the two branch points of softplus); columns [n/2, 3n/4) put y on both sides
    of beta y = 20 (where the curvature term of the adjoint switches off) with delta and z-dot 1000 times larger, so that a
    curvature term on the wrong side of the threshold moves the result by far more than the tolerance."""
    rng = np.random.default_rng(1000 * m + 10 * n + k + EPILOGUES.index(epi))
    lda, ldw, ldc, ldy, ldd, ldzd = k + 4, k + 8, n + 8, n + 12, n + 4, n + 16
    q = n // 4
    a = rng.standard_normal((m, lda)).astype(np.float32)
    w = rng.standard_normal((n, ldw)) / np.sqrt(k)
    w[:2 * q] *= 1e-3
    w = w.astype(np.float32)
    bias = 0.1 * rng.standard_normal(n)
    bias[:q] = 0.2 + rng.uniform(-2e-3, 2e-3, q)
    bias[q:2 * q] = -12.0 * np.log(2.0) / 100.0 + rng.uniform(-2e-3, 2e-3, q)
    bias = bias.astype(np.float32)
    y = rng.uniform(0.0, 0.4, size=(m, ldy))
    s = rng.uniform(1e-5, 1e-2, size=(m, q)) * rng.choice([-1.0, 1.0], size=(m, q))
    y[:, 2 * q:3 * q] = 0.2 * (1.0 + s)
    y = y.astype(np.float32)
    d = rng.standard_normal((m, ldd))
    zd = rng.standard_normal((m, ldzd))
    d[:, 2 * q:3 * q] *= 1e3
    zd[:, 2 * q:3 * q] *= 1e3
    d, zd = d.astype(np.float32), zd.astype(np.float32)
    ta, tw, tb, ty, td, tzd = (_put(dev, t) for t in (a, w, bias, y, d, zd))
    wp = _pack(dev, tw, ldw, n, k, 0, 0, 0, n, k)
    L, st = _cabi.lib(), _st(dev)
    c = _buf(dev, (m + 3, ldc))
    c2 = _buf(dev, (m + 3, ldzd))
    if epi in ("mode0", "mode1", "mode2"):
        mode = int(epi[-1])
        _cabi.check(L.d3h_mlp_linear(ta.data_ptr(), lda, m, k, wp.data_ptr(), n, tb.data_ptr() if mode != 2 else None, mode,
                                     ty.data_ptr() if mode == 2 else None, ldy if mode == 2 else 0, c.data_ptr(), ldc, st),
                    "d3h_mlp_linear")
    elif epi == "tangent":
        _cabi.check(L.d3h_mlp_linear_tangent(ta.data_ptr(), lda, m, k, wp.data_ptr(), n, ty.data_ptr(), ldy, c2.data_ptr(), ldzd,
                                             c.data_ptr(), ldc, st), "d3h_mlp_linear_tangent")
    else:
        _cabi.check(L.d3h_mlp_linear_adjoint(ta.data_ptr(), lda, m, k, wp.data_ptr(), n, ty.data_ptr(), ldy, td.data_ptr(), ldd,
                                             tzd.data_ptr(), ldzd, c.data_ptr(), ldc, st), "d3h_mlp_linear_adjoint")
    z = _f64(a[:, :k]) @ _f64(w[:, :k]).T
    y64 = _f64(y[:, :n])
    want = {"mode0": lambda: z + bias, "mode1": lambda: MO.softplus(z + bias), "mode2": lambda: z * _spd(y64),
            "tangent": lambda: z * _spd(y64),
            "adjoint": lambda: z * _spd(y64) + _curv(y64) * _f64(d[:, :n]) * _f64(zd[:, :n])}[epi]()
    got = _np(c)
    assert _rel(got[:m, :n], want) < GEMM_TOL, (epi, _rel(got[:m, :n], want))
    assert (got[:m, n:] == SENTINEL).all(), "written past column N"
    assert (got[m:] == SENTINEL).all(), "written past row M"
    got2 = _np(c2)
    if epi == "tangent":
        assert _rel(got2[:m, :n], z) < GEMM_TOL, _rel(got2[:m, :n], z)
        assert (got2[:m, n:] == SENTINEL).all() and (got2[m:] == SENTINEL).all(), "z-dot written outside M x N"
    else:
        assert (got2 == SENTINEL).all()


LINEAR_M = (1, 127, 128, 129, 255, 257)
LINEAR_N = (64, 128, 192, 256)
LINEAR_K = (32, 64, 96, 288, 384)


@pytest.mark.parametrize("epi", EPILOGUES)
@pytest.mark.parametrize("k", LINEAR_K)
@pytest.mark.parametrize("n", LINEAR_N)
@pytest.mark.parametrize("m", LINEAR_M)
def test_linear_epilogues_at_the_edges(dev, m, n, k, epi):
    linear_case(dev, m, n, k, epi)


# ---------------------------------------------------------------------------------------------- packed weight image
PACK_CASES = [  # transpose, n_valid, k_valid, n_pad, k_pad, row0, col0
    (0, 150, 90, 192, 96, 3, 5),
    (1, 192, 70, 192, 96, 2, 7),
    (1, 39, 256, 64, 256, 0, 256),
    (0, 64, 32, 64, 32, 0, 0),
    (1, 100, 200, 128, 224, 5, 1),
]


def pack_case(dev, transpose, n_valid, k_valid, n_pad, k_pad, row0, col0):
    """d3h_mlp_pack_weight, checked through a linear call: B[n][k] = w[row0 + k][col0 + n] (transposed) or
    w[row0 + n][col0 + k] for n < n_valid, k < k_valid, zero elsewhere.  The columns of a beyond k_valid are not zero, so a
    missing zero fill in K shows; the output columns beyond n_valid must come out exactly zero."""
    rng = np.random.default_rng(n_valid + k_valid + transpose)
    m = 129
    rows = row0 + (k_valid if transpose else n_valid) + 2
    ldw = col0 + (n_valid if transpose else k_valid) + 3
    w = rng.standard_normal((rows, ldw)).astype(np.float32)
    a = rng.standard_normal((m, k_pad)).astype(np.float32)
    tw, ta = _put(dev, w), _put(dev, a)
    wp = _pack(dev, tw, ldw, n_valid, k_valid, transpose, row0, col0, n_pad, k_pad)
    out = _buf(dev, (m, n_pad))
    _cabi.check(_cabi.lib().d3h_mlp_linear(ta.data_ptr(), k_pad, m, k_pad, wp.data_ptr(), n_pad, None, 0, None, 0,
                                           out.data_ptr(), n_pad, _st(dev)), "d3h_mlp_linear")
    if transpose:
        bmat = w[row0:row0 + k_valid, col0:col0 + n_valid].T
    else:
        bmat = w[row0:row0 + n_valid, col0:col0 + k_valid]
    want = _f64(a[:, :k_valid]) @ _f64(bmat).T
    got = _np(out)
    assert _rel(got[:, :n_valid], want) < GEMM_TOL, _rel(got[:, :n_valid], want)
    assert (got[:, n_valid:] == 0).all(), "padding rows of the weight image are not zero"


@pytest.mark.parametrize("case", PACK_CASES, ids=lambda c: "t%d_n%d_k%d_np%d_kp%d" % c[:5])
def test_packed_weight_offsets_transpose_and_zero_fill(dev, case):
    pack_case(dev, *case)


# ---------------------------------------------------------------------------------------------- wgrad
WGRAD_M = (1, 31, 33, 511, 512, 513, 2000)
WGRAD_NK = [(n, k) for n in (128, 256) for k in (64, 128, 192, 256)]


def wgrad_case(dev, m, n, k, with_db):
    """d3h_mlp_wgrad: dw += dz^T a and db += sum dz onto non-zero values, or db null; the contraction runs over point
    ranges of >= 512 points (several ranges from M = 513 on, the last one partial); columns of dw beyond K untouched."""
    rng = np.random.default_rng(m * 7 + n + k + with_db)
    ldz, lda, lddw = n + 4, k + 8, k + 12
    dz = rng.standard_normal((m, ldz)).astype(np.float32)
    a = rng.standard_normal((m, lda)).astype(np.float32)
    base = rng.standard_normal((n, lddw)).astype(np.float32)
    base[:, k:] = SENTINEL
    bbase = rng.standard_normal(n).astype(np.float32)
    tdz, ta, dw, db = _put(dev, dz), _put(dev, a), _put(dev, base), _put(dev, bbase)
    L = _cabi.lib()
    nbytes = int(L.d3h_mlp_wgrad_workspace_bytes(m, n, k))
    ws = _buf(dev, (nbytes // 4,), fill=np.nan)
    _cabi.check(L.d3h_mlp_wgrad(tdz.data_ptr(), ldz, ta.data_ptr(), lda, m, n, k, dw.data_ptr(), lddw,
                                db.data_ptr() if with_db else None, ws.data_ptr(), nbytes, _st(dev)), "d3h_mlp_wgrad")
    want = _f64(dz[:, :n]).T @ _f64(a[:, :k])
    bound = 1e-5 * np.sqrt(m) * 4
    got = _np(dw)
    assert np.abs(got[:, :k] - _f64(base[:, :k]) - want).max() < bound, np.abs(got[:, :k] - base[:, :k] - want).max()
    assert (got[:, k:] == SENTINEL).all(), "written past column K of dw"
    gb = _np(db)
    if with_db:
        assert np.abs(gb - _f64(bbase) - _f64(dz[:, :n]).sum(0)).max() < bound
    else:
        assert (gb == bbase).all()


@pytest.mark.parametrize("nk", WGRAD_NK, ids=lambda p: "n%d_k%d" % p)
@pytest.mark.parametrize("m", WGRAD_M)
def test_wgrad_point_ranges_and_bias(dev, m, nk):
    wgrad_case(dev, m, nk[0], nk[1], with_db=(m + nk[1]) % 2 == 1)
    if m in (1, 513):
        wgrad_case(dev, m, nk[0], nk[1], with_db=(m + nk[1]) % 2 == 0)


# ---------------------------------------------------------------------------------------------- output layer
HEAD_K = (4, 128, 252, 256)
HEAD_M = (1, 127, 128, 129, 513)


def head_case(dev, d_out, k, m):
    """d3h_mlp_head, d3h_mlp_head_backward and d3h_mlp_head_second_backward for one output width: dw / db accumulate onto
    non-zero values; dz and mu untouched past column K and past row M.  The second derivative's activations straddle
    beta a = 20 with large delta and z-dot there (see linear_case)."""
    rng = np.random.default_rng(100 * d_out + k + m)
    lda, ldz = k + 4, k + 8
    a = rng.uniform(0.0, 0.4, size=(m, lda))
    h = max(k // 4, 1)
    s = rng.uniform(1e-5, 1e-2, size=(m, h)) * rng.choice([-1.0, 1.0], size=(m, h))
    a[:, :h] = 0.2 * (1.0 + s)
    a = a.astype(np.float32)
    w = rng.standard_normal((d_out, k)).astype(np.float32)
    bias = rng.standard_normal(d_out).astype(np.float32)
    g = rng.standard_normal((m, d_out)).astype(np.float32)
    adot = rng.standard_normal((m, lda)).astype(np.float32)
    dl = rng.standard_normal((m, lda))
    zd = rng.standard_normal((m, lda))
    dl[:, :h] *= 1e3
    zd[:, :h] *= 1e3
    dl, zd = dl.astype(np.float32), zd.astype(np.float32)
    dw0 = rng.standard_normal((d_out, k)).astype(np.float32)
    db0 = rng.standard_normal(d_out).astype(np.float32)
    ta, tw, tb, tg, tad, tdl, tzd = (_put(dev, t) for t in (a, w, bias, g, adot, dl, zd))
    L, st = _cabi.lib(), _st(dev)
    a64, g64 = _f64(a[:, :k]), _f64(g)

    out = _buf(dev, (m + 2, d_out))
    _cabi.check(L.d3h_mlp_head(ta.data_ptr(), lda, m, k, tw.data_ptr(), tb.data_ptr(), d_out, out.data_ptr(), st), "d3h_mlp_head")
    got = _np(out)
    assert _rel(got[:m], a64 @ _f64(w).T + bias) < GEMM_TOL and (got[m:] == SENTINEL).all()

    dz = _buf(dev, (m + 2, ldz))
    dw, db = _put(dev, dw0), _put(dev, db0)
    _cabi.check(L.d3h_mlp_head_backward(ta.data_ptr(), lda, m, k, tw.data_ptr(), d_out, tg.data_ptr(), dz.data_ptr(), ldz,
                                        dw.data_ptr(), db.data_ptr(), st), "d3h_mlp_head_backward")
    got = _np(dz)
    assert _rel(got[:m, :k], (g64 @ _f64(w)) * _spd(a64)) < GEMM_TOL
    assert (got[:m, k:] == SENTINEL).all() and (got[m:] == SENTINEL).all(), "dz written outside M x K"
    bound = 1e-5 * np.sqrt(m) * 4
    assert np.abs(_np(dw) - _f64(dw0) - g64.T @ a64).max() < bound
    assert np.abs(_np(db) - _f64(db0) - g64.sum(0)).max() < bound

    mu = _buf(dev, (m + 2, ldz))
    dw = _put(dev, dw0)
    _cabi.check(L.d3h_mlp_head_second_backward(tad.data_ptr(), lda, ta.data_ptr(), lda, tdl.data_ptr(), lda, tzd.data_ptr(), lda,
                                               m, k, tg.data_ptr(), d_out, dw.data_ptr(), mu.data_ptr(), ldz, st),
                "d3h_mlp_head_second_backward")
    got = _np(mu)
    want_mu = _curv(a64) * _f64(dl[:, :k]) * _f64(zd[:, :k])
    assert _rel(got[:m, :k], want_mu) < GEMM_TOL, _rel(got[:m, :k], want_mu)
    assert (got[:m, k:] == SENTINEL).all() and (got[m:] == SENTINEL).all(), "mu written outside M x K"
    assert np.abs(_np(dw) - _f64(dw0) - g64.T @ _f64(adot[:, :k])).max() < bound


@pytest.mark.parametrize("m", HEAD_M)
@pytest.mark.parametrize("k", HEAD_K)
@pytest.mark.parametrize("d_out", range(1, 9))
def test_output_layer_every_width(dev, d_out, k, m):
    head_case(dev, d_out, k, m)


# ---------------------------------------------------------------------------------------------- encoding
ENC_FREQ = (0, 1, 6, 10, 11, 16)
ENC_LAYOUTS = ("vec4", "offset", "cols", "ld")


def _enc_scales(x, n_freq, v, g, gbar):
    """the float64 sums of the encoding's kernels taken over absolute values: the scale of their fp32 rounding error"""
    ax, av = np.abs(_f64(x)), np.abs(_f64(v))
    one = np.ones_like(ax)
    tang, bwd, sec = [av], np.abs(g[:, :3]).copy(), np.zeros_like(ax)
    for kk in range(n_freq):
        f = 2.0 ** kk
        gs, gc = np.abs(g[:, 3 + 6 * kk:6 + 6 * kk]), np.abs(g[:, 6 + 6 * kk:9 + 6 * kk])
        tang += [f * av, f * av]
        bwd += f * (gs + gc)
        sec += f * f * av * (gs + gc)
    bbar = np.abs(gbar[:, :3]).copy()
    for kk in range(n_freq):
        f = 2.0 ** kk
        bbar += f * (np.abs(gbar[:, 3 + 6 * kk:6 + 6 * kk]) + np.abs(gbar[:, 6 + 6 * kk:9 + 6 * kk]))
    return one, np.concatenate(tang, -1), bwd, sec, bbar


def encoding_case(dev, n_freq, layout, m=1001):
    """d3h_mlp_embed on its vectorised path (n_cols, ld multiples of 4, `out` 16-byte aligned) and on the scalar path
    (`out` 4 bytes off, n_cols % 4 != 0, ld % 4 != 0), zero padding up to n_cols, nothing written past n_cols or M;
    d3h_mlp_embed_backward (accumulate 0 / 1), d3h_mlp_embed_tangent, d3h_mlp_embed_second_backward (gbar null or not)."""
    rng = np.random.default_rng(10 * n_freq + ENC_LAYOUTS.index(layout))
    e = 3 * (2 * n_freq + 1)
    n_cols = {"vec4": (e + 3) // 4 * 4 + 4, "offset": (e + 3) // 4 * 4, "cols": e + 2 - (e + 2) % 4 + 1, "ld": (e + 3) // 4 * 4}[layout]
    ld = {"vec4": n_cols + 8, "offset": n_cols + 4, "cols": n_cols + 3, "ld": n_cols + 5}[layout]
    x = rng.uniform(-1.2, 1.2, size=(m, 3)).astype(np.float32)
    v = rng.standard_normal((m, 3)).astype(np.float32)
    g = rng.standard_normal((m, ld)).astype(np.float32)
    gbar = rng.standard_normal((m, ld)).astype(np.float32)
    tx, tv, tg, tgb = (_put(dev, t) for t in (x, v, g, gbar))
    L, st = _cabi.lib(), _st(dev)
    g64, gb64 = _f64(g[:, :e]), _f64(gbar[:, :e])
    one, s_tang, s_bwd, s_sec, s_bar = _enc_scales(x, n_freq, v, g64, gb64)

    def check(got, want, scale, what):
        err = np.abs(_f64(got) - want) - ENC_TOL * scale
        assert err.max() <= 0.0, (what, float((np.abs(_f64(got) - want) / scale).max()))

    for kernel in ("embed", "tangent"):
        raw = _buf(dev, ((m + 2) * ld + 1,))
        out = raw[1:] if layout == "offset" else raw[:-1]      # 4 bytes off the 16-byte alignment
        if kernel == "embed":
            _cabi.check(L.d3h_mlp_embed(tx.data_ptr(), m, n_freq, out.data_ptr(), ld, n_cols, st), "d3h_mlp_embed")
            want, scale = MO.embed(x, n_freq), np.concatenate([np.abs(_f64(x))] + [one] * (2 * n_freq), -1)
        else:
            _cabi.check(L.d3h_mlp_embed_tangent(tx.data_ptr(), tv.data_ptr(), m, n_freq, out.data_ptr(), ld, n_cols, st),
                        "d3h_mlp_embed_tangent")
            want, scale = SO.embed_tangent(x, n_freq, v), s_tang
        got = _np(out).reshape(m + 2, ld)
        check(got[:m, :e], want, scale, kernel)
        assert (got[:m, e:n_cols] == 0).all(), "padding columns not zero"
        assert (got[:m, n_cols:] == SENTINEL).all() and (got[m:] == SENTINEL).all(), "written past n_cols or M"

    gx0 = rng.standard_normal((m, 3)).astype(np.float32)
    for accumulate in (0, 1):
        gx = _put(dev, gx0)
        _cabi.check(L.d3h_mlp_embed_backward(tx.data_ptr(), m, n_freq, tg.data_ptr(), ld, gx.data_ptr(), accumulate, st),
                    "d3h_mlp_embed_backward")
        want = MO.embed_backward(x, n_freq, g64) + (_f64(gx0) if accumulate else 0.0)
        check(_np(gx), want, s_bwd + (np.abs(_f64(gx0)) if accumulate else 0.0), "backward")
    for with_bar in (True, False):
        hx = _put(dev, gx0)
        _cabi.check(L.d3h_mlp_embed_second_backward(tx.data_ptr(), tv.data_ptr(), m, n_freq, tgb.data_ptr() if with_bar else None,
                                                    ld, tg.data_ptr(), ld, hx.data_ptr(), st), "d3h_mlp_embed_second_backward")
        want = SO.embed_second_backward(x, n_freq, v, g64) + (MO.embed_backward(x, n_freq, gb64) if with_bar else 0.0)
        check(_np(hx), want, s_sec + (s_bar if with_bar else 0.0) + 1e-30, "second backward")


@pytest.mark.parametrize("layout", ENC_LAYOUTS)
@pytest.mark.parametrize("n_freq", ENC_FREQ)
def test_encoding_paths_and_frequencies(dev, n_freq, layout):
    encoding_case(dev, n_freq, layout)


# ---------------------------------------------------------------------------------------------- modules
MODULE_CFGS = {   # 128-wide encodings (n_freq >= 11), no frequencies, skip layers first / last, one hidden layer
    "f0_d128_o2_skip_first": dict(n_freq=0, d_hidden=128, d_out=2, n_hidden=2, skip_in=[0]),
    "f11_d256_o8_skip_last": dict(n_freq=11, d_hidden=256, d_out=8, n_hidden=3, skip_in=[2]),
    "f16_d128_o8_one_hidden": dict(n_freq=16, d_hidden=128, d_out=8, n_hidden=1, skip_in=[]),
    "f11_d128_o2_one_hidden_skip": dict(n_freq=11, d_hidden=128, d_out=2, n_hidden=1, skip_in=[0]),
}


def module_case(dev, name, m, eikonal):
    """MLP through the real module path, against the float64 oracle: first order (forward, every gradient), or the eikonal
    training step (first-order loss + ((|gx| - 1)^2).mean() through autograd.grad(create_graph=True))."""
    from d3human_code_b200.geometry.mlp import MLP
    cfg = MODULE_CFGS[name]
    torch.manual_seed(m + len(name))
    net = MLP(**cfg).to(dev)
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(1.5)
    lin = [mod for mod in net.net if isinstance(mod, torch.nn.Linear)]
    rng = np.random.default_rng(m)
    x = rng.uniform(-1, 1, size=(m, 3)).astype(np.float32)
    g1 = rng.standard_normal((m, cfg["d_out"])).astype(np.float32)
    tx = torch.tensor(x, device=dev, requires_grad=True)
    y = net(tx)
    assert y.shape == (m, cfg["d_out"])
    yo, cache = MO.forward(x, [_np(l.weight) for l in lin], [_np(l.bias) for l in lin], cfg["n_freq"], tuple(cfg["skip_in"]))
    assert _rel(_np(y), yo) < FWD_TOL, _rel(_np(y), yo)
    fx, fw, fb = MO.backward(cache, g1)
    if not eikonal:
        (y * torch.tensor(g1, device=dev)).sum().backward()
        errs = {"x": _rel(_np(tx.grad), fx)}
        for i, l in enumerate(lin):
            errs[f"w{i}"] = _rel(_np(l.weight.grad), fw[i])
            errs[f"b{i}"] = _rel(_np(l.bias.grad), fb[i])
        assert max(errs.values()) < GRAD_TOL, errs
        return
    ones = torch.ones_like(y)
    gx, = torch.autograd.grad(y, tx, ones, create_graph=True)
    eik = ((gx.norm(dim=-1) - 1.0) ** 2).mean()
    ((y * torch.tensor(g1, device=dev)).sum() + eik).backward()
    ones64 = np.ones((m, cfg["d_out"]))
    gx_o, _, _ = MO.backward(cache, ones64)
    assert _nrel(_np(gx), gx_o) < SO_TOL
    nrm = np.linalg.norm(gx_o, axis=-1, keepdims=True)
    v = 2.0 * (nrm - 1.0) * gx_o / nrm / m
    hx, hw, hb, _ = SO.second_order(cache, ones64, v)
    errs = {"x": _nrel(_np(tx.grad), hx + fx)}
    for i, l in enumerate(lin):
        errs[f"w{i}"] = _nrel(_np(l.weight.grad), hw[i] + fw[i])
        errs[f"b{i}"] = _nrel(_np(l.bias.grad), hb[i] + fb[i])
    tol = SO_TOL + _pre_activation_sensitivity(cache, [_np(l.bias) for l in lin], ones64, v, (hx, hw, hb))
    assert max(errs.values()) < tol, (tol, errs)


def _pre_activation_sensitivity(cache, biases, g_out, v, exact):
    """Largest normwise change of the float64 second derivative when every pre-activation moves by 2^-22 of the sum of
    its terms' magnitudes, with random signs: the error any fp32-accurate GEMM (the 3xTF32 split included) may leave in
    a pre-activation.  Softplus(beta=100)'s second derivative turns an absolute error dz there into a relative error of
    about beta dz in the unit's curvature term, so where few units carry the result (one point, a wide encoding) fp32
    itself cannot reach 1e-4; on the other configurations this adds a few 1e-5."""
    rng = np.random.default_rng(0)
    pert = dict(cache)
    pert["pre"] = [z + 2.0 ** -22 * (np.abs(h) @ np.abs(w).T + np.abs(_f64(b))) * rng.choice([-1.0, 1.0], size=z.shape)
                   for z, h, w, b in zip(cache["pre"], cache["inputs"], cache["w"], biases)]
    px, pw, pb, _ = SO.second_order(pert, g_out, v)
    hx, hw, hb = exact
    return max([_nrel(px, hx)] + [_nrel(a, b) for a, b in zip(pw, hw)] + [_nrel(a, b) for a, b in zip(pb[:-1], hb[:-1])])


@pytest.mark.parametrize("eikonal", [False, True], ids=["first_order", "eikonal"])
@pytest.mark.parametrize("m", [1, 128, 129, 4097])
@pytest.mark.parametrize("name", list(MODULE_CFGS))
def test_module_configurations(module_dev, name, m, eikonal):
    module_case(module_dev, name, m, eikonal)


# ---------------------------------------------------------------------------------------------- several devices
def test_linear_and_wgrad_on_every_device(dev):
    """The GEMM kernels need more than 48 KB of dynamic shared memory, a per-kernel attribute of each device: a process
    that runs the network on a second device after the first must launch there as well."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    for i in list(range(torch.cuda.device_count())) + [0]:
        d = torch.device(f"cuda:{i}")
        with torch.cuda.device(d):
            linear_case(d, 129, 256, 288, "mode1")
            wgrad_case(d, 513, 256, 256, with_db=True)
