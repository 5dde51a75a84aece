"""The dense gradient buffers of a batched extraction are zero-filled by the backward call, not by the forward call.

A batch's forward call allocates its gradient buffers uninitialised; its backward call zeroes them in ONE launch ahead of
the adjoints: every frame, also frames without a surface or without upstream gradients, and a buffer that several
frames share (sdf / msdf) once.  D3H_ZERO_IN_FORWARD=1 brings back the fill on the forward call.

The cases run on memory the caching allocator has handed out before, filled with NaN, so a row the call forgets to
zero shows up: every frame's grad_pos must be finite, exactly zero away from the rows the frame touched (the end points
of its crossing edges, FramesFuture.tape_edges) and equal to the oracle on them."""
import numpy as np
import pytest
import torch

from oracle import gshell_oracle as O
from d3human_code_b200 import grids
from d3human_code_b200 import extract as E
from tests import _util as U
from tests import test_fused_batch_shapes as T
from tests.test_cuda_parity import dev, edges_mode  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu


@pytest.fixture
def dirty(dev):
    """dirty(*shapes): allocates float tensors of these shapes on the device, fills them with NaN and frees them, so the
    caching allocator hands the same blocks to the next allocations of those sizes."""
    def poison(*shapes):
        blocks = [torch.full(s, float("nan"), dtype=torch.float32, device=dev) for s in shapes for _ in range(3)]
        del blocks
    return poison


class _AsyncBatch(T._Batch):
    """T._Batch through extract_frames_async, keeping the future (for tape_edges)."""

    def run(self, lanes, presize=True):
        self.tp = torch.tensor(self.pos_b, device=self.dev, requires_grad=True)
        s_arg, self.ts, self.s_keys = self._leaves(self.sdfs, self.form == "shared")
        m_arg, self.tm, self.m_keys = self._leaves(self.msdfs, False)
        tt = torch.tensor(self.tets, device=self.dev)
        if presize:
            T._presize(self.dev, self.tets.shape[0], self.pos_b.shape[1], self.fwds)
        self.fut = E.extract_frames_async(self.tp, s_arg, m_arg, tt, types=self.types, lanes=lanes)
        self.outs = self.fut.result()
        return self.outs


def _check_untouched_rows(b):
    g = b.tp.grad.cpu().numpy()
    assert np.isfinite(g).all(), "grad_pos holds rows the backward call did not zero"
    for i in range(b.B):
        rows = np.unique(b.fut.tape_edges(i).cpu().numpy().reshape(-1))
        off = np.ones(g.shape[1], dtype=bool)
        off[rows] = False
        assert not g[i][off].any(), f"grad_pos[{i}]: a row away from the frame's crossing edges is not zero"


def dirty_case(dev, dirty, res, B, skip=(), empty_first=0, seed=0):
    """B frames on 8 lanes on NaN-filled memory; `skip`: frames without upstream gradients; the first `empty_first`
    frames on a field without a surface."""
    pos, tets, pos_b = T._frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    sdfs = [np.ones_like(sdf)] * empty_first + [sdf] * (B - empty_first)
    b = _AsyncBatch(dev, pos_b, sdfs, [msdf] * B, tets, ["cloth"] * B, form="list" if empty_first else "shared")
    N = pos.shape[0]
    dirty((B, N, 3), (N,), (N, 1))
    b.run(8)
    T._check_forward(b.outs, b.fwds)
    back = b.backward_and_check(np.random.default_rng(seed), skip)
    assert back.get("zero") == 1, back
    _check_untouched_rows(b)
    if empty_first:
        assert all(o[0].shape[0] == 0 for o in b.outs[:empty_first])
    return b


@pytest.mark.parametrize("B", [8, 17])
def test_dirty_memory(dev, edges_mode, dirty, B):
    """8 and 17 frames on 8 lanes; with 17 frames one frame gets no upstream gradient: its grad_pos is exactly zero."""
    T._skip_unless_scan(edges_mode)
    dirty_case(dev, dirty, 16, B, skip=(11,) if B == 17 else ())


def test_dirty_memory_empty_frames(dev, edges_mode, dirty):
    """17 frames whose first 8 have no surface: the adjoints skip them, the zero-fill does not."""
    T._skip_unless_scan(edges_mode)
    dirty_case(dev, dirty, 16, 17, empty_first=8)


def path_case(dev, dirty, monkeypatch, res):
    """Launch counts: a forward-only batched call launches no zero-fill, its backward exactly one; with
    D3H_ZERO_IN_FORWARD=1 the forward call launches it (once per fused launch) and the backward none."""
    lanes, B = 8, 8
    pos, tets, pos_b = T._frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    for in_forward in (False, True):
        if in_forward:
            monkeypatch.setenv("D3H_ZERO_IN_FORWARD", "1")
        else:
            monkeypatch.delenv("D3H_ZERO_IN_FORWARD", raising=False)
        b = _AsyncBatch(dev, pos_b, [sdf] * B, [msdf] * B, tets, ["cloth"] * B)
        dirty((B, pos.shape[0], 3), (pos.shape[0],))
        _, fwd, _ = T._observed(lambda: b.run(lanes))
        T._assert_fused(fwd, B, lanes)
        back = b.backward_and_check(np.random.default_rng(9))
        _check_untouched_rows(b)
        assert back.get("adjoint") == 1, back
        if in_forward:
            assert fwd.get("zero") == len(T._rounds(B, lanes)) and "zero" not in back, (fwd, back)
        else:
            assert "zero" not in fwd and back.get("zero") == 1, (fwd, back)


def test_zero_fill_path(dev, edges_mode, dirty, monkeypatch):
    T._skip_unless_scan(edges_mode)
    path_case(dev, dirty, monkeypatch, 16)


def shared_gradient_case(dev, dirty, res, api):
    """Two groups of frames on the same sdf / msdf leaves, one backward call per group: each call zero-fills its own
    buffers, autograd sums them into .grad, and the sums match the oracle (per-frame or packed API)."""
    lanes, groups, per = 8, 2, 9
    B = groups * per
    pos, tets, pos_b = T._frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    N = pos.shape[0]
    fwds = [O.extract_forward(pos_b[i], sdf, msdf, tets, 1, True) for i in range(B)]
    T._presize(dev, tets.shape[0], N, fwds)
    rng = np.random.default_rng(10)
    ups = [(rng.standard_normal(f["verts_aug"].shape).astype(np.float32),
            rng.standard_normal(f["msdf"].shape).astype(np.float32)) for f in fwds]
    dirty((per, N, 3), (N,), (N, 1))
    tt = torch.tensor(tets, device=dev)
    ts = torch.tensor(sdf[:, None], device=dev, requires_grad=True)
    tm = torch.tensor(msdf, device=dev, requires_grad=True)
    pgs = [torch.tensor(pos_b[g * per:(g + 1) * per], device=dev, requires_grad=True) for g in range(groups)]
    futs = [E.extract_frames_async(pg, ts, tm, tt, types="cloth", lanes=lanes) for pg in pgs]
    for g, fut in enumerate(futs):
        u = ups[g * per:(g + 1) * per]
        if api == "packed":
            pk = fut.packed()
            gv = torch.zeros(pk.verts_aug.shape, device=dev)
            gm = torch.zeros(pk.msdf.shape, device=dev)
            for i, (a, m) in enumerate(u):
                gv[i, :a.shape[0]] = torch.tensor(a, device=dev)
                gm[i, :m.shape[0]] = torch.tensor(m, device=dev)
            torch.autograd.backward([pk.verts_aug, pk.msdf], [gv, gm])
        else:
            outs = fut.result()
            torch.autograd.backward([o[0] for o in outs] + [o[5]["msdf"] for o in outs],
                                    [torch.tensor(a, device=dev) for a, _ in u] + [torch.tensor(m, device=dev) for _, m in u])
    want_s, want_m = np.zeros(N, np.float64), np.zeros(N, np.float64)
    for i in range(B):
        g_pos, g_sdf, g_msdf = O.extract_backward(fwds[i], *ups[i])
        want_s += g_sdf.reshape(-1)
        want_m += g_msdf
        got = pgs[i // per].grad[i % per].cpu().numpy()
        assert np.isfinite(got).all(), i
        U.assert_close_normwise(f"grad_pos[{i}]", got, g_pos, U.GRAD_RTOL)
    U.assert_close_normwise("grad_sdf", ts.grad.cpu().numpy().reshape(-1), want_s, U.GRAD_RTOL)
    U.assert_close_normwise("grad_msdf", tm.grad.cpu().numpy(), want_m, U.GRAD_RTOL)


@pytest.mark.parametrize("api", ["frames", "packed"])
def test_shared_gradient_over_two_backward_calls(dev, edges_mode, dirty, api):
    T._skip_unless_scan(edges_mode)
    shared_gradient_case(dev, dirty, 16, api)
