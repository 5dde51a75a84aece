"""The `-m gpu` parity tests, run on the CPU against a functional emulation of the CUDA kernels.

`tests/emu/build_emu.py` compiles the product's .cu files unchanged with g++ against `tests/emu/cuda_runtime.h`
(every CUDA thread is a fibre; barriers and warp collectives are rendezvous points) and this module points the ctypes
binding at the result, then calls the very test functions of `tests/test_cuda_parity.py` / `tests/test_z_configs.py`
with a CPU device.  What this checks is the LOGIC of the kernels (indexing, scans, sorts, tables, float op order) and
the whole host path through the real C ABI; it cannot see data races, memory-ordering bugs or anything about speed --
those are what the GPU runs are for.  Test infrastructure only: the product loads `lib/libd3h_tets.so` (nvcc, sm_100a)
and nothing else.
"""
import contextlib
import os
import sys

import numpy as np
import pytest
import torch

from d3human_code_b200 import _cabi
from d3human_code_b200 import extract as E
from tests import _util as U
from tests import test_cuda_parity as G
from tests import test_z_configs as Z

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import build_emu  # noqa: E402


class _Stream:
    cuda_stream = 0

    def synchronize(self):
        pass


def _packed_tets_cpu(tet_fx4, n_grid):
    """extract.packed_tets without the CUDA-only parts: same library calls, same IndexError on bad indices."""
    L = _cabi.lib()
    n_tets = tet_fx4.shape[0]
    bad = torch.zeros(1, dtype=torch.int64)
    if tet_fx4.dtype == torch.int32 and tet_fx4.is_contiguous() and tet_fx4.data_ptr() % 16 == 0:
        out = tet_fx4
        _cabi.check(L.d3h_check_tets_i32(out.data_ptr(), n_tets, n_grid, bad.data_ptr(), 0), "d3h_check_tets_i32")
    else:
        src = tet_fx4.contiguous().to(torch.int64)
        out = torch.empty((n_tets, 4), dtype=torch.int32)
        _cabi.check(L.d3h_pack_tets_i64(src.data_ptr(), n_tets, n_grid, out.data_ptr(), bad.data_ptr(), 0), "d3h_pack_tets_i64")
    if int(bad.item()):
        raise IndexError(f"tet_fx4 holds {int(bad.item())} vertex indices outside [0, {n_grid})")
    key = (tet_fx4.data_ptr(), tuple(tet_fx4.shape), tet_fx4.dtype, int(n_grid))
    return _packed_cache.setdefault(key, out)       # a stable address per tet array, like the real cache


_packed_cache = {}


@pytest.fixture(scope="module")
def emu_lib_path():
    return build_emu.build()


@pytest.fixture(params=["sort", "static", "scan", "scan_rows", "scan_csr"])
def edges_mode(request):
    if request.param in ("scan_rows", "scan_csr") and request.node.originalname not in (
            "test_golden", "test_oracle", "test_random_tet_soups", "test_tet_soups_with_repeated_vertices"):
        pytest.skip("the other forms of the static edge list are covered by the golden / oracle / soup tests")
    # the tet stream over the static edge table (D3H_EDGE_SCAN=0) is not a default path any more: on the emulation it
    # keeps the golden / oracle / soup / batch tests (everything runs on it on the GPU); keeps the CPU suite short
    if request.param == "static" and request.node.originalname not in (
            "test_golden", "test_oracle", "test_random_tet_soups", "test_tet_soups_with_repeated_vertices", "test_batches",
            "test_integer_intermediates", "test_regrowth", "test_emulated_library_is_the_real_abi"):
        pytest.skip("static-table tet stream: golden / oracle / soup / batch tests only on the emulation")
    if request.param == "sort" and request.node.originalname == "test_fused_frames_shared_topology_and_regrowth":
        pytest.skip("frames are fused on the run-length path only")
    E.set_scan_rows(request.param != "scan_csr")
    E.set_scan_runs(request.param == "scan")
    yield "scan" if request.param.startswith("scan") else request.param
    E.set_scan_rows(True)
    E.set_scan_runs(True)


@pytest.fixture
def dev(emu_lib_path, edges_mode, monkeypatch):
    """A 'device' for the GPU test functions: CPU tensors + the emulated library behind the real C ABI binding."""
    monkeypatch.setattr(_cabi, "LIB_PATH", emu_lib_path)
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(E, "_check_cuda", lambda t: None)
    monkeypatch.setattr(E, "packed_tets", _packed_tets_cpu)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: _Stream())
    monkeypatch.setattr(torch.cuda, "device", lambda dev=None: contextlib.nullcontext())
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    orig_ensure = E._Plan.ensure

    def ensure(self, lanes, n_edges=0):       # CPU allocations are 64-byte aligned, the ABI wants 256 for the workspace
        orig_ensure(self, lanes, n_edges)
        for i, w in enumerate(self.workspaces):
            if w.data_ptr() % 256:
                big = torch.empty(self.workspace_bytes + 256, dtype=torch.uint8)
                off = (-big.data_ptr()) % 256
                self.workspaces[i] = big[off:off + self.workspace_bytes]
                self.workspace_ptrs[i] = self.workspaces[i].data_ptr()

    monkeypatch.setattr(E._Plan, "ensure", ensure)
    E.reset_plans()
    _packed_cache.clear()
    E.set_static_edges("0" if edges_mode == "sort" else "1")
    E.set_edge_scan(edges_mode == "scan")
    yield torch.device("cpu")
    E.set_static_edges("auto")
    E.set_edge_scan(True)
    E.reset_plans()


def test_emulated_library_is_the_real_abi(dev):
    L = _cabi.lib()
    assert L.d3h_version() == _cabi.VERSION
    for name in _cabi.EXPORTED_SYMBOLS:
        assert hasattr(L, name)


@pytest.mark.parametrize("name", U.golden_cases())
def test_golden(dev, name):
    G.test_cuda_matches_golden(dev, name)


@pytest.mark.parametrize("res,field,cls,typ,wt", [
    (16, "sphere", "GShell_Tets", None, True),
    (24, "capsule", "hmSDF_Tets", "cloth", True),
    (24, "capsule", "hmSDF_Tets", "body", True),
    (12, "adv", "GShell_Tets", None, True),
    (12, "adv", "hmSDF_Tets", "body", True),
    (10, "adv", "GShell_Tets", None, False),
    (10, "adv", "hmSDF_Tets", "body", False),
])
def test_oracle(dev, res, field, cls, typ, wt):
    G.test_cuda_matches_oracle(dev, res, field, cls, typ, wt)


def test_fused_frames_shared_topology_and_regrowth(dev, edges_mode):
    G.test_fused_frames_shared_topology_and_regrowth(dev, edges_mode)


def test_integer_intermediates(dev, edges_mode):
    G.test_integer_intermediates_match_oracle(dev, edges_mode)


def test_smplx_layout(dev):
    G.test_smplx_layout_split_extraction(dev)


def test_regrowth(dev):
    G.test_capacity_regrowth_and_reuse(dev)


def test_validation_and_refusals(dev):
    G.test_input_validation(dev)
    G.test_msdf_boundary_view_carries_gradient(dev)


def test_batches(dev):
    G.test_extract_frames_batch_matches_oracle_per_frame(dev)
    G.test_extract_frames_list_form_and_repeat(dev)


def test_packed_batch(dev):
    G.test_packed_batch_equals_per_frame_results(dev)


def test_compact_gradient_return(dev):
    G.test_compact_gradient_return(dev)


@pytest.mark.parametrize("res,field,typ,vr", [(16, "capsule", "cloth", 3), (12, "adv", "body", 2)])
def test_tet_range_sharding(dev, res, field, typ, vr):
    G.test_tet_range_sharding_virtual_ranks_bit_identical(dev, res, field, typ, vr)


def test_pipelined_groups_and_split(dev):
    Z.test_pipelined_async_groups_equal_single_calls(dev)
    Z.test_split_pair_matches_two_calls(dev)


@pytest.mark.parametrize("seed,n,f", [(0, 9, 60), (1, 40, 400), (2, 25, 3000), (3, 12, 6000), (4, 300, 5000), (5, 6, 2500)])
def test_random_tet_soups(dev, seed, n, f):
    """Non-manifold tet soups (random vertex quadruples): edges shared by hundreds of tets, vertices with hundreds of
    neighbours -- the oversized-group path of the sort, long neighbour lists of the static edge table, dense buckets.
    tests/test_oracle_vs_reference.py shows the oracle tracks the reference on such input."""
    from oracle import gshell_oracle as O
    rng = np.random.default_rng(500 + seed)
    tets = np.stack([rng.permutation(n)[:4] for _ in range(f)]).astype(np.int64)
    pos = rng.standard_normal((n, 3)).astype(np.float32)
    sdf = rng.standard_normal(n).astype(np.float32)
    msdf = rng.standard_normal(n).astype(np.float32)
    sdf[::7] = 0.0
    msdf[::5] = 0.0
    typ = (None, "cloth", "body")[seed % 3]
    cls = "GShell_Tets" if typ is None else "hmSDF_Tets"
    fwd = O.extract_forward(pos, sdf, msdf, tets, -1 if typ == "body" else 1, True)
    rng2 = np.random.default_rng(1)
    grads = dict(g_verts_aug=rng2.standard_normal(fwd["verts_aug"].shape).astype(np.float32),
                 g_msdf=rng2.standard_normal(fwd["msdf"].shape).astype(np.float32),
                 g_msdf_watertight=None, g_vertices_watertight=None)
    out, g = G._run(dev, pos, sdf, msdf, tets, cls, typ, True, grads)
    U.assert_exact("faces_aug", out["faces_aug"], fwd["faces_aug"])
    U.assert_exact("verts_aug", out["verts_aug"], fwd["verts_aug"])
    U.assert_exact("msdf", out["msdf"], fwd["msdf"])
    U.assert_exact("faces_watertight", out["faces_watertight"], fwd["faces_watertight"])
    U.assert_exact("vertices_watertight", out["vertices_watertight"], fwd["vertices_watertight"])
    g_pos, g_sdf, g_msdf = O.extract_backward(fwd, grads["g_verts_aug"], grads["g_msdf"])
    U.assert_close_normwise("grad_pos", g[0], g_pos, 5 * U.GRAD_RTOL)
    U.assert_close_normwise("grad_sdf", g[1], g_sdf, 5 * U.GRAD_RTOL)
    if typ != "body":
        U.assert_close_normwise("grad_msdf", g[2], g_msdf, 5 * U.GRAD_RTOL)


@pytest.mark.parametrize("res,field,wt", [(12, "capsule", True), (10, "adv", True), (8, "adv", False), (6, "sphere", True)])
def test_fused_pair_equals_two_calls(dev, res, field, wt):
    """hmSDF_Tets.split(fused=True): one classification / de-duplication for the cloth / body pair, only the mSDF cut is
    replayed -- bit-identical to the two separate calls, gradients equal to their sum."""
    from d3human_code_b200.geometry.hmsdf_tets_split import hmSDF_Tets
    pos, sdf, msdf, tets = G._inputs(res, field, seed=res)
    hm = hmSDF_Tets()
    tt = torch.tensor(tets)

    def leaves():
        return (torch.tensor(pos, requires_grad=True), torch.tensor(sdf, requires_grad=True),
                torch.tensor(msdf, requires_grad=True))

    def loss(c, b):
        out = c[0].square().sum() + b[0].square().sum() + c[5]["msdf"].sum() - 2.0 * b[5]["msdf"].sum()
        if wt:
            out = out + c[5]["vertices_watertight"].sum() + (b[5]["msdf_watertight"] ** 2).sum()
        return out

    for rep in range(2):      # second round: capacities settled, no re-run
        tp, ts, tm = leaves()
        cloth, body = hm.split(tp, ts, tm, tt, output_watertight_template=wt, fused=True)
        loss(cloth, body).backward()
        tp2, ts2, tm2 = leaves()
        c2 = hm(tp2, ts2, tm2, tt, "cloth", wt)
        b2 = hm(tp2, ts2, tm2, tt, "body", wt)
        loss(c2, b2).backward()
        for a, b in ((cloth, c2), (body, b2)):
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), rep
            assert tuple(a[5].keys()) == tuple(b[5].keys())
            for k in a[5]:
                if torch.is_tensor(a[5][k]) and "tng" not in k:
                    assert torch.equal(a[5][k], b[5][k]), (rep, k)
            U.assert_tangents_close("v_tng_aug", a[4].detach().numpy(), b[4].detach().numpy(), 2.0 if field == "adv" else U.TNG_CUDA_ATOL)
        U.assert_close_normwise("grad_pos", tp.grad.numpy(), tp2.grad.numpy(), U.GRAD_RTOL)
        U.assert_close_normwise("grad_sdf", ts.grad.numpy(), ts2.grad.numpy(), U.GRAD_RTOL)
        U.assert_close_normwise("grad_msdf", tm.grad.numpy(), tm2.grad.numpy(), U.GRAD_RTOL)


@pytest.mark.parametrize("res,field", [(12, "capsule"), (8, "adv")])
def test_gpu_fused_pair_test_body(dev, res, field):
    Z.fused_pair_equals_two_calls(dev, res, field)


def _fuzz_case(case):
    from d3human_code_b200 import grids
    rng = np.random.default_rng(case)
    kind = int(rng.integers(0, 4))
    if kind == 0:      # lattice, smooth field
        res = int(rng.integers(1, 9))
        pos, tets = grids.kuhn_grid(res)
        c, r = rng.standard_normal(3) * 0.3, rng.uniform(0.05, 1.5)
        sdf = (r - np.linalg.norm(pos - c, axis=1)).astype(np.float32)
        msdf = (pos @ rng.standard_normal(3) + rng.normal() * 0.2).astype(np.float32)
    elif kind == 1:    # lattice, adversarial field (exact zeros)
        res = int(rng.integers(1, 7))
        pos, tets = grids.kuhn_grid(res)
        pos, sdf, msdf = grids.adversarial_field(pos, res, seed=case)
    elif kind == 2:    # tet soup
        n, f = int(rng.integers(4, 80)), int(rng.integers(1, 1500))
        tets = np.stack([rng.permutation(n)[:4] for _ in range(f)]).astype(np.int64)
        pos = rng.standard_normal((n, 3)).astype(np.float32)
        sdf, msdf = rng.standard_normal(n).astype(np.float32), rng.standard_normal(n).astype(np.float32)
        sdf[::3] = 0
        msdf[::4] = 0
    else:              # degenerate: constant fields with one flipped vertex
        res = int(rng.integers(1, 4))
        pos, tets = grids.kuhn_grid(res)
        sdf = np.full(pos.shape[0], rng.choice([-1.0, 1.0, 0.0]), np.float32)
        sdf[int(rng.integers(0, pos.shape[0]))] = rng.choice([-1.0, 1.0])
        msdf = np.full(pos.shape[0], rng.choice([-1.0, 1.0, 0.0]), np.float32)
    typ = [None, "cloth", "body"][int(rng.integers(0, 3))]
    wt = bool(rng.integers(0, 4) != 0)
    return pos, sdf, msdf, tets, typ, wt


@pytest.mark.parametrize("seed,n,f,wt", [(0, 10, 400, True), (1, 30, 2500, True), (2, 16, 1500, False)])
def test_tet_soups_with_repeated_vertices(dev, edges_mode, seed, n, f, wt):
    Z.test_tet_soups_with_repeated_vertices(dev, seed, n, f, wt)


def test_mark_rows_variant(dev, edges_mode):
    """Opt-in marking kernel over fixed-width incidence rows (edge_mark_rows_kernel, D3H_MARK_ROWS=1): the owner of a valid
    tet is elected by rule (its first crossing edge), no atomic result is awaited.  Lattices, crowded edges (> 8 tets: the
    CSR fallback) and tets that repeat a vertex."""
    if edges_mode != "scan":
        pytest.skip("variant of the edge-scan path")
    E.set_mark_rows(True)
    E.reset_plans()
    try:
        G.test_cuda_matches_oracle(dev, 12, "adv", "GShell_Tets", None, True)
        G.test_cuda_matches_oracle(dev, 16, "capsule", "hmSDF_Tets", "body", False)
        G.test_extract_frames_batch_matches_oracle_per_frame(dev)
        test_random_tet_soups(dev, 3, 12, 6000)
        Z.test_tet_soups_with_repeated_vertices(dev, 1, 30, 2500, True)
        Z.test_tet_soups_with_repeated_vertices(dev, 2, 16, 1500, False)
        ents = [ent for ent in E._static_cache.values() if ent[1] is not None]
        assert ents and all(ent[1][7] is not None for ent in ents)     # the rows were really built and passed
    finally:
        E.set_mark_rows(False)
        E.reset_plans()


@pytest.mark.parametrize("res,field,cls,typ", [(12, "sphere", "GShell_Tets", None), (12, "capsule", "hmSDF_Tets", "cloth"),
                                               (12, "capsule", "hmSDF_Tets", "body")])
def test_tangent_gradients(dev, edges_mode, res, field, cls, typ):
    G.test_tangent_gradients_match_oracle(dev, res, field, cls, typ)


def test_tangent_gradients_batch(dev, edges_mode):
    G.test_tangent_gradients_in_a_batch_and_three_face_refusal(dev)


def test_fuzz_forward_against_oracle(dev):
    """60 seeded random inputs (lattices, adversarial fields, tet soups, degenerate fields; 1650 such cases were run once
    while writing this): every integer output, position and mSDF value bit-exact against the oracle."""
    from oracle import gshell_oracle as O
    for case in range(60):
        pos, sdf, msdf, tets, typ, wt = _fuzz_case(case)
        if case % 5 == 0:
            E.reset_plans()
            _packed_cache.clear()
        out = E.extract(torch.tensor(pos), torch.tensor(sdf), torch.tensor(msdf), torch.tensor(tets),
                        msdf_negate=(typ == "body"), output_watertight_template=wt)
        fwd = O.extract_forward(pos, sdf, msdf, tets, -1 if typ == "body" else 1, wt)
        U.assert_exact(f"verts_aug[{case}]", out[0].numpy(), fwd["verts_aug"])
        U.assert_exact(f"faces_aug[{case}]", out[1].numpy(), fwd["faces_aug"])
        U.assert_exact(f"msdf[{case}]", out[5]["msdf"].numpy(), fwd["msdf"])
        if wt:
            U.assert_exact(f"faces_watertight[{case}]", out[5]["faces_watertight"].numpy(), fwd["faces_watertight"])
            U.assert_exact(f"vertices_watertight[{case}]", out[5]["vertices_watertight"].numpy(), fwd["vertices_watertight"])


def test_fuzz_backward_against_oracle(dev):
    """The first 40 fuzz cases with seeded upstream gradients on verts_aug and msdf: dense gradients against the oracle's
    float64 adjoint (a 120-case run of both edge paths stayed below 2.3e-6 normwise)."""
    from oracle import gshell_oracle as O
    for case in range(40):
        pos, sdf, msdf, tets, typ, wt = _fuzz_case(case)
        if case % 5 == 0:
            E.reset_plans()
            _packed_cache.clear()
        tp, ts, tm = (torch.tensor(x, requires_grad=True) for x in (pos, sdf, msdf))
        out = E.extract(tp, ts, tm, torch.tensor(tets), msdf_negate=(typ == "body"), output_watertight_template=wt)
        fwd = O.extract_forward(pos, sdf, msdf, tets, -1 if typ == "body" else 1, wt)
        if fwd["verts_aug"].shape[0] == 0:
            continue
        rng = np.random.default_rng(case + 7)
        gv = rng.standard_normal(fwd["verts_aug"].shape).astype(np.float32)
        gm = rng.standard_normal(fwd["msdf"].shape).astype(np.float32)
        torch.autograd.backward([out[0], out[5]["msdf"]], [torch.tensor(gv), torch.tensor(gm)])
        g_pos, g_sdf, g_m = O.extract_backward(fwd, gv, gm)
        U.assert_close_normwise(f"g_pos[{case}]", tp.grad.numpy(), g_pos, U.GRAD_RTOL)
        U.assert_close_normwise(f"g_sdf[{case}]", ts.grad.numpy().reshape(g_sdf.shape), g_sdf, U.GRAD_RTOL)
        if typ != "body":
            U.assert_close_normwise(f"g_msdf[{case}]", tm.grad.numpy(), g_m, U.GRAD_RTOL)
        else:
            assert tm.grad is None


def test_tet_edge_rank_table_variant(dev, edges_mode):
    """EXPERIMENTAL D3H_TET_EDGE_RANKS: the compaction kernel reads the edge ranks of a valid tet from a per-tet table
    instead of bisecting the neighbour lists -- same results."""
    if edges_mode != "static":
        pytest.skip("variant of the static edge table path")
    E.set_tet_edge_ranks(True)
    try:
        G.test_cuda_matches_oracle(dev, 12, "adv", "GShell_Tets", None, True)
        G.test_cuda_matches_oracle(dev, 16, "capsule", "hmSDF_Tets", "body", True)
        G.test_extract_frames_batch_matches_oracle_per_frame(dev)
        test_random_tet_soups(dev, 3, 12, 6000)
        plan_keys = list(E._static_cache.values())
        assert plan_keys and all(ent[1] is None or ent[1][3] is not None for ent in plan_keys)   # the table was really used
    finally:
        E.set_tet_edge_ranks(False)
