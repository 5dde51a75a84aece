"""Fused frame batches in the shapes a training step runs, against the numpy oracle.

bench.py runs 8 lanes, so every fused launch has kMaxFused = 8 rows (grid.y = frame) and a backward pass takes more than
kAdjBatch = 16 frames.  This covers what only those shapes reach: the topology tiles split over 8 rows, the per-frame
tables of the topology CTAs filled to 8 entries, the corner ids copied onto the tapes of frames 1..7 and read back by the
tangent adjoint, several adjoint launches per backward, polygon counts at the edges of the 64- and 256-polygon tiles
(none at all included), and the host's decisions whether the frames of a launch share one topology and whether a launch
keeps the topology of the launch before.

Every frame is checked against the oracle: integer outputs, positions and mSDF bit-exact, tangents with the
condition-aware bound, and gradients normwise, each frame with its own upstream gradients on verts_aug, msdf,
vertices_watertight and both tangent outputs (the shared sdf / msdf receive the sum over the frames).  Each case also
asserts the path it took, so that a fall-back to one frame per launch fails instead of passing: launches per kernel kind
(d3h_profile_*: a fused launch is ONE poly_faces launch for all its frames) and, per frame, whether it searched for a
topology of its own (the device trace: the edge-scan compaction stamps the row of every frame it runs for; a frame that
takes the topology of the first frame of its launch, or of the launch before, runs none)."""
import numpy as np
import pytest
import torch

from oracle import gshell_oracle as O
from d3human_code_b200 import _cabi, grids
from d3human_code_b200 import extract as E
from tests import _util as U
from tests.test_cuda_parity import _tangent_upstream, dev, edges_mode  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

#: gradients that also flow through the tangent branch (tests/test_cuda_parity.py: test_tangent_gradients_*)
TNG_GRAD_RTOL = 1e-4
#: the fused launches of a batch have at most this many rows (kMaxFused, csrc/d3h_internal.cuh)
MAX_FUSED = 8
#: frames per adjoint launch (kAdjBatch, csrc/d3h_backward.cu)
ADJ_BATCH = 16

#: sphere fields cut by the grid boundary (odd polygon counts need that on the Kuhn lattice): centre and, per resolution,
#: (radius, polygons) with fewer than 64 polygons (one poly_cut tile), exactly 256 k and 256 k + 1 (poly_faces tiles)
TILE_CENTRE = (0.97, 0.93, -0.2)
TILE_RADII = {
    12: {"small": (0.086, 8), "tiles": (0.737, 512), "tiles_plus_one": (1.173, 1025)},
    16: {"small": (0.084, 12), "tiles": (0.783, 1024), "tiles_plus_one": (0.369, 257)},
}


def _skip_unless_scan(edges_mode):
    if edges_mode != "scan":
        pytest.skip("frames are fused on the run-length path only")


def _rounds(B, lanes):
    """Sizes of the fused launches of a batch: frame i runs in workspace i % lanes, a launch takes consecutive frames
    with distinct workspaces, at most MAX_FUSED."""
    r = min(lanes, E.MAX_LANES, MAX_FUSED, B)
    return [r] * (B // r) + ([B % r] if B % r else [])


def _presize(dev, n_tets, n_grid, fwds):
    """Capacities of the grid's plan from the oracle's sizes: the call runs once, without a counting run or a regrowth,
    so its launches and trace rows are those of the fused batch alone.  The records get twice the room: the edge-scan
    work queues are cut from that capacity in sub-queues, and one that fills up makes the call re-run."""
    plan = E._plan_for(dev, n_tets, n_grid)
    fv = max(int(f["t1"]) + int(f["t2"]) for f in fwds)
    v = max(int(f["n_verts_watertight"]) for f in fwds)
    va = max(f["verts_aug"].shape[0] for f in fwds)
    fw = max(f["faces_watertight"].shape[0] for f in fwds)
    fa = max(f["faces_aug"].shape[0] for f in fwds)
    plan.cap_tets, plan.cap_v, plan.cap_va, plan.cap_fw, plan.cap_fa = (E._grow(x) for x in (2 * fv, v, va, fw, fa))
    return plan


def _observed(fn, plan=None, B=0):
    """Runs fn() with the launch profiler and the device trace on.
    -> (fn(), {kernel kind: launches}, per frame of the last batch of `plan`: did it search for its own topology)"""
    L = _cabi.lib()
    kinds = [L.d3h_profile_kernel_name(k).decode() for k in range(L.d3h_profile_kinds())]
    _cabi.profile_read()
    _cabi.profile_enable(True)
    _cabi.trace_enable(True)
    try:
        out = fn()
        launches = {k: n for k, (_, n) in _cabi.profile_read().items()}
        table = np.zeros((64, 24, 2), dtype=np.uint64)
        _cabi.check(L.d3h_trace_read(table.ctypes.data), "d3h_trace_read")
    finally:
        _cabi.profile_enable(False)
        _cabi.trace_enable(False)
    own = None
    if plan is not None:
        assert B <= 64
        seqs = [plan.seq - B + 1 + i for i in range(B)]        # the frames of the batch launched last
        own = [bool(table[s % 64, kinds.index("compact"), 1]) for s in seqs]
    return out, launches, own


def _shared_own(B, lanes):
    """Frames that search for a topology when every frame shares sdf / msdf / type: the first frame of a launch, unless
    the launch keeps the topology of the launch before (both have more than one frame)."""
    own, prev = [], 0
    for n in _rounds(B, lanes):
        own += [not (n > 1 and prev > 1)] + [False] * (n - 1)
        prev = n
    return own


def _check_forward(outs, fwds, max_unchecked=0.01):
    assert len(outs) == len(fwds)
    for i, (verts, faces, uvs, uv_idx, v_tng, extra) in enumerate(outs):
        f = fwds[i]
        nv = int(f["n_verts_watertight"])
        assert extra["n_verts_watertight"] == nv, (i, extra["n_verts_watertight"], nv)
        U.assert_exact(f"faces_aug[{i}]", faces.cpu().numpy(), f["faces_aug"])
        U.assert_exact(f"verts_aug[{i}]", verts.detach().cpu().numpy(), f["verts_aug"])
        U.assert_exact(f"msdf[{i}]", extra["msdf"].detach().cpu().numpy(), f["msdf"])
        U.assert_exact(f"msdf_boundary[{i}]", extra["msdf_boundary"].detach().cpu().numpy(), f["msdf_boundary"])
        U.assert_exact(f"faces_watertight[{i}]", extra["faces_watertight"].cpu().numpy(), f["faces_watertight"])
        U.assert_exact(f"vertices_watertight[{i}]", extra["vertices_watertight"].detach().cpu().numpy(),
                       f["vertices_watertight"])
        if nv:
            kappa = O.tangent_condition(f)
            limit = max(max_unchecked, 1.0 / nv)       # (a tiny surface: one row may be ill-conditioned)
            U.assert_tangents_conditioned(f"v_tng_aug[{i}]", v_tng.detach().cpu().numpy(), f["v_tng_aug"], kappa,
                                          max_unchecked_frac=limit)
            U.assert_tangents_conditioned(f"v_tng_watertight[{i}]", extra["v_tng_watertight"].detach().cpu().numpy(),
                                          f["v_tng_watertight"], kappa[:nv], max_unchecked_frac=limit)


def _upstream(fwd, rng):
    """verts_aug, msdf, vertices_watertight, v_tng_aug, v_tng_watertight (tangent rows of ill-conditioned vertices: 0)"""
    nv = int(fwd["n_verts_watertight"])
    g_aug, g_wt = _tangent_upstream(fwd, rng) if nv else (np.zeros_like(fwd["v_tng_aug"]), np.zeros((0, 3), np.float32))
    return (rng.standard_normal(fwd["verts_aug"].shape).astype(np.float32),
            rng.standard_normal(fwd["msdf"].shape).astype(np.float32),
            rng.standard_normal((nv, 3)).astype(np.float32), g_aug, g_wt)


class _Batch:
    """One extract_frames call on per-frame fields: `sdfs` / `msdfs` list the frame's array; frames that name the SAME
    array object share one tensor (form="list") or the one shared tensor (form="shared", sdf as (N,1) like the SDF
    network's output); form="stacked" passes (B,N) tensors, one row per frame."""

    def __init__(self, dev, pos_b, sdfs, msdfs, tets, types, form="shared"):
        self.dev, self.pos_b, self.sdfs, self.msdfs, self.tets, self.types = dev, pos_b, sdfs, msdfs, tets, types
        self.B = pos_b.shape[0]
        self.form = form
        self.fwds = [O.extract_forward(pos_b[i], sdfs[i], msdfs[i], tets, -1 if types[i] == "body" else 1, True)
                     for i in range(self.B)]

    def _leaves(self, arrays, col):
        if self.form == "stacked":
            t = torch.tensor(np.stack(arrays), device=self.dev, requires_grad=True)
            return t, [t], [(0, i) for i in range(self.B)]
        uniq, keys = [], []
        for a in arrays:
            k = next((j for j, u in enumerate(uniq) if u is a), None)
            if k is None:
                k = len(uniq)
                uniq.append(a)
            keys.append((k, None))
        ts = [torch.tensor(a[:, None] if col else a, device=self.dev, requires_grad=True) for a in uniq]
        if self.form == "shared":
            assert len(ts) == 1
            return ts[0], ts, keys
        return [ts[k] for k, _ in keys], ts, keys

    def run(self, lanes, presize=True):
        """-> (outputs, {kernel kind: forward launches}, per frame: searched for its own topology)"""
        self.tp = torch.tensor(self.pos_b, device=self.dev, requires_grad=True)
        s_arg, self.ts, self.s_keys = self._leaves(self.sdfs, self.form == "shared")
        m_arg, self.tm, self.m_keys = self._leaves(self.msdfs, False)
        tt = torch.tensor(self.tets, device=self.dev)
        plan = _presize(self.dev, self.tets.shape[0], self.pos_b.shape[1], self.fwds) if presize else None
        outs, launches, own = _observed(lambda: E.extract_frames(self.tp, s_arg, m_arg, tt, types=self.types, lanes=lanes),
                                        plan, self.B)
        if presize:
            assert E._ExtractFn.last_launches < 2 * self.B * E.LAUNCHES_FORWARD_SCAN, "the call re-ran"
        self.outs = outs
        return outs, launches, own

    def backward_and_check(self, rng, skip=()):
        """Each frame but those in `skip` gets its own upstream gradients on the five differentiable outputs.
        -> {kernel kind: backward launches}"""
        tensors, grads = [], []
        want_pos = np.zeros(self.pos_b.shape, np.float64)
        want_s = [np.zeros(tuple(t.shape), np.float64) for t in self.ts]
        want_m = [np.zeros(tuple(t.shape), np.float64) for t in self.tm]
        m_used = [False] * len(self.tm)
        for i, (verts, _, _, _, v_tng, extra) in enumerate(self.outs):
            if i in skip:
                continue
            gv, gm, gw, g_aug, g_wt = _upstream(self.fwds[i], rng)
            for out, g in ((verts, gv), (extra["msdf"], gm), (extra["vertices_watertight"], gw), (v_tng, g_aug),
                           (extra["v_tng_watertight"], g_wt)):
                tensors.append(out)
                grads.append(torch.tensor(g, device=self.dev))
            g_pos, g_sdf, g_msdf = O.extract_backward(self.fwds[i], gv, gm, gw, None, g_aug, g_wt)
            want_pos[i] = g_pos
            k, _ = self.s_keys[i]
            if self.form == "stacked":
                want_s[0][i] += g_sdf
            else:
                want_s[k] += g_sdf.reshape(want_s[k].shape)
            if self.types[i] != "body":
                k, _ = self.m_keys[i]
                if self.form == "stacked":
                    want_m[0][i] += g_msdf
                else:
                    want_m[k] += g_msdf
                m_used[k if self.form != "stacked" else 0] = True
        _, launches, _ = _observed(lambda: torch.autograd.backward(tensors, grads))
        got_pos = self.tp.grad.cpu().numpy()
        for i in range(self.B):
            if i in skip:
                assert not got_pos[i].any(), f"grad_pos[{i}]: a frame without upstream gradients got one"
            else:
                U.assert_close_normwise(f"grad_pos[{i}]", got_pos[i], want_pos[i], TNG_GRAD_RTOL)
        for j, t in enumerate(self.ts):
            U.assert_close_normwise(f"grad_sdf[{j}]", t.grad.cpu().numpy(), want_s[j], TNG_GRAD_RTOL)
        for j, t in enumerate(self.tm):
            if m_used[j]:
                U.assert_close_normwise(f"grad_msdf[{j}]", t.grad.cpu().numpy(), want_m[j], TNG_GRAD_RTOL)
            else:
                assert t.grad is None or not t.grad.any(), "body frames do not back-propagate into msdf"
        return launches


def _frames(res, B):
    pos, tets = grids.kuhn_grid(res)
    pos_b = np.stack([pos + grids.frame_offsets(pos.shape[0], res, f) for f in range(B)]).astype(np.float32)
    assert all(not np.array_equal(pos_b[0], pos_b[i]) for i in range(1, B))
    return pos, tets, pos_b


def _assert_fused(launches, B, lanes):
    rounds = _rounds(B, lanes)
    assert launches.get("poly_faces") == len(rounds) and launches.get("poly_cut") == len(rounds), (launches, rounds)


# ------------------------------------------------------------------------------------------------ 1. eight rows
def eight_rows_case(dev, res, B, typ, skip=(), seed=0):
    """B frames on the shared capsule field, lanes = 8: launches of 8 rows, later launches keep the topology."""
    lanes = 8
    pos, tets, pos_b = _frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    b = _Batch(dev, pos_b, [sdf] * B, [msdf] * B, tets, [typ] * B)
    outs, launches, own = b.run(lanes)
    assert lanes == MAX_FUSED and max(_rounds(B, lanes)) == MAX_FUSED
    _assert_fused(launches, B, lanes)
    assert own == _shared_own(B, lanes), own
    assert launches.get("compact") == sum(_shared_own(B, lanes)), launches
    _check_forward(outs, b.fwds)
    back = b.backward_and_check(np.random.default_rng(seed), skip)
    live = B - len(skip)
    assert back.get("adjoint") == (live + ADJ_BATCH - 1) // ADJ_BATCH, back
    return b


@pytest.mark.parametrize("typ", ["cloth", "body"])
@pytest.mark.parametrize("B", [8, 9, 17])
def test_eight_rows_per_launch(dev, edges_mode, B, typ):
    """8, 9 and 17 frames on 8 lanes: launches of 8 / 8+1 / 8+8+1 frames, the second launch of 17 keeps the topology of
    the first.  With 17 frames one frame gets no upstream gradient at all: the other 16 fill exactly one adjoint launch."""
    _skip_unless_scan(edges_mode)
    eight_rows_case(dev, 16, B, typ, skip=(11,) if B == 17 else ())


def test_thirty_three_frames_three_adjoint_launches(dev, edges_mode):
    """33 frames on 8 lanes: five launches (8+8+8+8+1; launches 2-4 keep the topology) and three adjoint launches
    (16+16+1) in the backward pass."""
    _skip_unless_scan(edges_mode)
    assert (33 + ADJ_BATCH - 1) // ADJ_BATCH == 3
    eight_rows_case(dev, 16, 33, "cloth")


# ------------------------------------------------------------------------------------------------ 2. tile edges
def _tile_field(pos, radius):
    p = pos.astype(np.float64)
    sdf = (radius - np.linalg.norm(p - np.asarray(TILE_CENTRE), axis=-1)).astype(np.float32)
    msdf = (p[:, 1] - TILE_CENTRE[1] + 0.3 * radius).astype(np.float32)
    return sdf, msdf


def tile_edge_case(dev, res, which):
    """8 frames on 8 lanes sharing one field whose polygon count sits at a tile edge; 'empty': sdf > 0 everywhere."""
    lanes, B = 8, 8
    pos, tets, pos_b = _frames(res, B)
    if which == "empty":
        sdf, msdf = np.ones(pos.shape[0], np.float32), grids.capsule_garment_field(pos)[1]
        want = 0
    else:
        radius, want = TILE_RADII[res][which]
        sdf, msdf = _tile_field(pos, radius)
    b = _Batch(dev, pos_b, [sdf] * B, [msdf] * B, tets, ["cloth"] * B)
    npoly = int(b.fwds[0]["t1"]) + int(b.fwds[0]["t2"])
    assert npoly == want, (which, npoly)
    assert {"empty": npoly == 0, "small": 0 < npoly < 64, "tiles": npoly % 256 == 0 and npoly > 0,
            "tiles_plus_one": npoly % 256 == 1 and npoly > 256}[which]
    outs, launches, own = b.run(lanes)
    _assert_fused(launches, B, lanes)
    assert own == _shared_own(B, lanes), own
    counts = E.last_counts_frames()
    assert len(counts) == B
    for i, c in enumerate(counts):      # every frame's counts were published (the host waited for each of them)
        assert (c["n_tri_tets"] + c["n_quad_tets"], c["n_verts"]) == (npoly, int(b.fwds[i]["n_verts_watertight"])), c
    # (a sphere cut off by the grid boundary has more vertices whose face normals cancel than the capsule)
    _check_forward(outs, b.fwds, max_unchecked=0.05)
    if which == "empty":
        assert all(o[0].shape == (0, 3) and o[1].shape == (0, 3) and o[5]["faces_watertight"].shape == (0, 3)
                   for o in outs)
    back = b.backward_and_check(np.random.default_rng(3))
    if which == "empty":
        assert back.get("adjoint", 0) == 0, back     # every frame is dropped from the adjoint batch
        assert not b.tp.grad.any() and not b.ts[0].grad.any() and not b.tm[0].grad.any()
    else:
        assert b.tp.grad.any()


@pytest.mark.parametrize("which", ["empty", "small", "tiles", "tiles_plus_one"])
def test_polygon_counts_at_tile_edges(dev, edges_mode, which):
    """8 rows sharing one topology at polygon counts where the tiles of the surface kernels end: none at all, fewer than
    64 (one poly_cut tile: most topology CTAs of both kernels have no data but still count towards the last-CTA-out
    scan), exactly 256 k and 256 k + 1 (poly_faces tiles)."""
    _skip_unless_scan(edges_mode)
    tile_edge_case(dev, 16, which)


def empty_frames_in_adjoint_batch_case(dev, res):
    """17 frames, the first 8 on an empty field: the first adjoint launch compacts its 16 frames to the 8 non-empty ones,
    the second takes frame 16."""
    lanes, B = 8, 17
    pos, tets, pos_b = _frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    empty = np.ones_like(sdf)
    b = _Batch(dev, pos_b, [empty] * 8 + [sdf] * 9, [msdf] * B, tets, ["cloth"] * B, form="list")
    outs, launches, own = b.run(lanes)
    _assert_fused(launches, B, lanes)
    assert own == [True] + [False] * 7 + [True] + [False] * 7 + [True], own   # another field: nothing kept
    _check_forward(outs, b.fwds)
    assert all(o[0].shape[0] == 0 for o in outs[:8]) and all(o[0].shape[0] > 0 for o in outs[8:])
    back = b.backward_and_check(np.random.default_rng(4))
    assert back.get("adjoint") == 2, back
    assert not b.ts[0].grad.any()


def test_empty_frames_with_gradients_in_an_adjoint_batch(dev, edges_mode):
    _skip_unless_scan(edges_mode)
    empty_frames_in_adjoint_batch_case(dev, 16)


# ------------------------------------------------------------------------------------------------ 3. share / reuse
def _second_field(pos):
    """another surface and another garment than capsule_garment_field's (a wrong reuse keeps the capsule's topology)"""
    p = pos.astype(np.float64)
    return grids.capsule_sdf(pos, 0.06).astype(np.float32), np.minimum(p[:, 1] + 0.2, 0.6 - p[:, 1]).astype(np.float32)


def alternating_fields_case(dev, res, vary):
    """[A]*4 + [B]*4 + [A]*4 on 4 lanes, sdf or msdf varied: three launches that each share a topology, none keeps the
    topology of the launch before."""
    lanes, B = 4, 12
    pos, tets, pos_b = _frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    sdf2, msdf2 = _second_field(pos)
    if vary == "sdf":
        sdfs, msdfs = [sdf] * 4 + [sdf2] * 4 + [sdf] * 4, [msdf] * B
    else:
        sdfs, msdfs = [sdf] * B, [msdf] * 4 + [msdf2] * 4 + [msdf] * 4
    b = _Batch(dev, pos_b, sdfs, msdfs, tets, ["cloth"] * B, form="list")
    assert not np.array_equal(b.fwds[0]["faces_aug"], b.fwds[4]["faces_aug"])
    outs, launches, own = b.run(lanes)
    _assert_fused(launches, B, lanes)
    assert own == [True, False, False, False] * 3, own
    assert launches.get("compact") == 3, launches
    _check_forward(outs, b.fwds)
    b.backward_and_check(np.random.default_rng(5))


@pytest.mark.parametrize("vary", ["sdf", "msdf"])
def test_alternating_fields_never_reuse_the_launch_before(dev, edges_mode, vary):
    _skip_unless_scan(edges_mode)
    alternating_fields_case(dev, 16, vary)


def stacked_equal_rows_case(dev, res):
    """A stacked (B,N) sdf and msdf whose rows are equal: different pointers, so no launch shares (or keeps) a topology;
    every frame searches its own.  (A stacked field needs N % 4 == 0.)"""
    lanes, B = 4, 8
    pos, tets, pos_b = _frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    b = _Batch(dev, pos_b, [sdf.copy() for _ in range(B)], [msdf.copy() for _ in range(B)], tets, ["cloth"] * B,
               form="stacked")
    outs, launches, own = b.run(lanes)
    _assert_fused(launches, B, lanes)
    assert own == [True] * B, own
    assert launches.get("compact") == len(_rounds(B, lanes)), launches
    _check_forward(outs, b.fwds)
    b.backward_and_check(np.random.default_rng(6))


def test_stacked_equal_rows_do_not_share(dev, edges_mode):
    _skip_unless_scan(edges_mode)
    stacked_equal_rows_case(dev, 19)      # (stacked rows need N % 4 == 0: 20^3 vertices)


def mixed_types_case(dev, res):
    """cloth and body frames alternating on 8 lanes: ONE launch of 8 rows that does not share (msdf_negate differs)."""
    lanes, B = 8, 8
    pos, tets, pos_b = _frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    types = ["cloth", "body"] * 4
    b = _Batch(dev, pos_b, [sdf] * B, [msdf] * B, tets, types)
    outs, launches, own = b.run(lanes)
    _assert_fused(launches, B, lanes)
    assert own == [True] * B, own
    _check_forward(outs, b.fwds)
    b.backward_and_check(np.random.default_rng(7))


def test_mixed_types_in_one_launch_do_not_share(dev, edges_mode):
    _skip_unless_scan(edges_mode)
    mixed_types_case(dev, 16)


def regrowth_case(dev, res, B=11):
    """test_fused_frames_shared_topology_and_regrowth on 8 lanes: 11 frames (8 + 3, the second launch keeps the
    topology), the second call after the plan's capacities were cut down (every list overflows, the host re-runs)."""
    lanes = 8
    pos, tets, pos_b = _frames(res, B)
    sdf, msdf = grids.capsule_garment_field(pos)
    b = _Batch(dev, pos_b, [sdf] * B, [msdf] * B, tets, ["cloth"] * B)
    outs, launches, own = b.run(lanes)
    assert own == _shared_own(B, lanes) == [True] + [False] * (B - 1), own
    _assert_fused(launches, B, lanes)
    _check_forward(outs, b.fwds)
    b.backward_and_check(np.random.default_rng(8))
    for plan in E._plans.values():
        plan.cap_tets, plan.cap_v, plan.cap_va, plan.cap_fw, plan.cap_fa = 96, 48, 96, 48, 48
    outs, launches, _ = b.run(lanes, presize=False)
    per_attempt = B * E.LAUNCHES_FORWARD_SCAN
    assert E._ExtractFn.last_launches >= 2 * per_attempt, "the cut-down capacities did not overflow"
    n = len(_rounds(B, lanes))
    assert launches["poly_faces"] % n == 0 and launches["poly_faces"] < B, launches   # every attempt fused
    _check_forward(outs, b.fwds)
    b.backward_and_check(np.random.default_rng(8))


def test_regrowth_on_eight_lanes(dev, edges_mode):
    _skip_unless_scan(edges_mode)
    regrowth_case(dev, 16)


# ------------------------------------------------------------------------------------------------ 4. full size
def test_bench_pattern_full_size(dev, edges_mode):
    """bench.py's calling pattern at its size: 128^3, the capsule field, 2 groups of 16 frames on 8 lanes, both groups
    launched (extract_frames_async) before either is read, a backward pass per group.  Every frame against a drop-in
    hmSDF_Tets call on the same positions (integer outputs and positions bit-exact, gradients within GRAD_RTOL); frames
    0 and 31 against the oracle."""
    _skip_unless_scan(edges_mode)
    if dev.type != "cuda":
        pytest.skip("128^3: GPU only")
    from d3human_code_b200.geometry.hmsdf_tets_split import hmSDF_Tets
    res, groups, per, lanes = 128, 2, 16, 8
    B = groups * per
    pos, tets = grids.kuhn_grid(res)
    sdf, msdf = grids.capsule_garment_field(pos)
    N = pos.shape[0]
    tt = torch.tensor(tets, device=dev)
    pos_all = torch.tensor(np.stack([pos + grids.frame_offsets(N, res, f) for f in range(B)]), device=dev)
    ts = torch.tensor(sdf[:, None], device=dev, requires_grad=True)
    tm = torch.tensor(msdf, device=dev, requires_grad=True)
    pgs = [pos_all[g * per:(g + 1) * per].clone().requires_grad_(True) for g in range(groups)]
    futs = [E.extract_frames_async(pg, ts, tm, tt, types="cloth", lanes=lanes) for pg in pgs]
    gen = torch.Generator(device=dev).manual_seed(1234)
    outs, ups = [], []
    for fut in futs:
        o = fut.result()
        assert len(o) == per
        u = [(torch.randn(f[0].shape, device=dev, generator=gen), torch.randn(f[5]["msdf"].shape, device=dev, generator=gen),
              torch.randn(f[5]["vertices_watertight"].shape, device=dev, generator=gen)) for f in o]
        torch.autograd.backward([f[0] for f in o] + [f[5]["msdf"] for f in o] + [f[5]["vertices_watertight"] for f in o],
                                [x[0] for x in u] + [x[1] for x in u] + [x[2] for x in u])
        outs += o
        ups += u
    hm = hmSDF_Tets()
    g_sdf, g_msdf = torch.zeros_like(ts), torch.zeros_like(tm)
    for i in range(B):
        p1 = pos_all[i].clone().requires_grad_(True)
        s1, m1 = ts.detach().clone().requires_grad_(True), tm.detach().clone().requires_grad_(True)
        v, f, _, _, _, ex = hm(p1, s1, m1, tt, "cloth")
        o = outs[i]
        assert torch.equal(o[1], f) and torch.equal(o[5]["faces_watertight"], ex["faces_watertight"]), i
        assert torch.equal(o[0].detach(), v.detach()) and torch.equal(o[5]["msdf"].detach(), ex["msdf"].detach()), i
        assert torch.equal(o[5]["vertices_watertight"].detach(), ex["vertices_watertight"].detach()), i
        assert torch.equal(o[5]["msdf_boundary"].detach(), ex["msdf_boundary"].detach()), i
        torch.autograd.backward([v, ex["msdf"], ex["vertices_watertight"]], list(ups[i]))
        grad_group = pgs[i // per].grad[i % per]
        U.assert_close_normwise(f"grad_pos[{i}]", grad_group.cpu().numpy(), p1.grad.cpu().numpy(), U.GRAD_RTOL)
        g_sdf += s1.grad
        g_msdf += m1.grad
    U.assert_close_normwise("grad_sdf", ts.grad.cpu().numpy(), g_sdf.cpu().numpy(), U.GRAD_RTOL)
    U.assert_close_normwise("grad_msdf", tm.grad.cpu().numpy(), g_msdf.cpu().numpy(), U.GRAD_RTOL)
    for i in (0, B - 1):
        fwd = O.extract_forward(pos_all[i].cpu().numpy(), sdf, msdf, tets, 1, True, n_threads=8)
        o = outs[i]
        U.assert_exact(f"faces_aug[{i}]", o[1].cpu().numpy(), fwd["faces_aug"])
        U.assert_exact(f"verts_aug[{i}]", o[0].detach().cpu().numpy(), fwd["verts_aug"])
        U.assert_exact(f"msdf[{i}]", o[5]["msdf"].detach().cpu().numpy(), fwd["msdf"])
        U.assert_exact(f"faces_watertight[{i}]", o[5]["faces_watertight"].cpu().numpy(), fwd["faces_watertight"])
        U.assert_exact(f"vertices_watertight[{i}]", o[5]["vertices_watertight"].detach().cpu().numpy(),
                       fwd["vertices_watertight"])
        U.assert_exact(f"msdf_boundary[{i}]", o[5]["msdf_boundary"].detach().cpu().numpy(), fwd["msdf_boundary"])
        U.assert_tangents_conditioned(f"v_tng_aug[{i}]", o[4].detach().cpu().numpy(), fwd["v_tng_aug"],
                                      O.tangent_condition(fwd), max_unchecked_frac=0.01)
        g_pos, _, _ = O.extract_backward(fwd, *(u.cpu().numpy() for u in ups[i]))
        U.assert_close_normwise(f"oracle grad_pos[{i}]", pgs[i // per].grad[i % per].cpu().numpy(), g_pos, U.GRAD_RTOL)
