"""The run-length extraction path (scan_runs_kernel / runs_expand_kernel, csrc/d3h_scan.cu) on structured tet grids other
than the axis-numbered Kuhn lattice.

extract.build_edge_runs / build_tet_runs compress a grid's tables whenever it averages at least _RUNS_MIN_EDGES edges or
tets per entry, so any grid with some structure in its numbering lands on this path: tets whose vertex lists are rotated
(negative tet-run differences: windows that start below their chunk), tets listed in any order (the ids of an entry spread
over many compaction tiles: the collision fallback of the per-CTA count table), grids cropped to the body (isolated
vertices, partial lane masks), boxes whose vertex count is a multiple of 32 or one more (the last sign word and the spare
word behind it), tets that repeat a vertex (self edges, d = 0 entries), and grids that only get the compressed edge list
(edge runs without tet runs: the marking kernel behind the expansion).  Every family is checked against the numpy oracle
on all edge paths: outputs and integer intermediates bit-exact, gradients normwise; on the "scan" path the table form
the family must produce is asserted, so that a silent fall-back to the rows cannot pass for coverage.
"""
import functools
import itertools

import numpy as np
import pytest
import torch

from oracle import gshell_oracle as O
from d3human_code_b200 import grids
from tests import _util as U
from tests import test_cuda_parity as G

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(autouse=True, params=["sort", "static", "scan", "scan_rows", "scan_csr"])
def edges_mode(request):
    """sort: per-call radix sort; static: tet stream over the static edge table; scan: edge scan, the host picks the table
    form (run-length here); scan_rows: transposed edge rows; scan_csr: CSR walk.  Tables are dropped around every test so
    that the form asserted is the one this test built."""
    from d3human_code_b200 import extract as E
    E.reset_plans()
    E.set_static_edges("0" if request.param == "sort" else "1")
    E.set_edge_scan(request.param.startswith("scan"))
    E.set_scan_rows(request.param != "scan_csr")
    E.set_scan_runs(request.param == "scan")
    yield request.param
    E.set_static_edges("auto")
    E.set_edge_scan(True)
    E.set_scan_rows(True)
    E.set_scan_runs(True)
    E.reset_plans()


# ---------------------------------------------------------------------------------------------- grid families
def box_grid(nx, ny, nz):
    """Anisotropic Kuhn lattice of nx * ny * nz cells on [-1,1]^3: N = (nx+1)(ny+1)(nz+1), vertex id = (z*(ny+1) + y)*(nx+1)
    + x, tets cube-major like grids.kuhn_grid (which is box_grid(res, res, res))."""
    lx, ly, lz = (np.linspace(-1.0, 1.0, k + 1, dtype=np.float64).astype(np.float32) for k in (nx, ny, nz))
    z, y, x = np.meshgrid(lz, ly, lx, indexing="ij")
    pos = np.stack([x, y, z], -1).reshape(-1, 3).astype(np.float32)
    sy, sz = nx + 1, (nx + 1) * (ny + 1)
    cz, cy, cx = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    base = (cz * sz + cy * sy + cx).reshape(-1).astype(np.int64)

    def corner(bits):
        return ((bits >> 2) & 1) * sz + ((bits >> 1) & 1) * sy + (bits & 1)

    shapes = [np.stack([base + corner(b) for b in (0, p[0], p[0] | p[1], 7)], -1) for p in itertools.permutations((1, 2, 4))]
    return pos, np.ascontiguousarray(np.stack(shapes, 1).reshape(-1, 4))


#: vertex-list permutation of each of the 6 Kuhn shapes: identity, odd ones (flipped winding), and ones that move the
#: smallest vertex out of slot 0 (negative tet-run differences)
_ROTATIONS = ((0, 1, 2, 3), (1, 0, 2, 3), (2, 3, 0, 1), (3, 2, 1, 0), (1, 2, 3, 0), (0, 2, 1, 3))


def rotated(res):
    """Edge runs and tet runs; 5 of the 6 tet shapes have a negative difference."""
    pos, tets = grids.kuhn_grid(res)
    t = tets.reshape(-1, 6, 4).copy()
    for s, perm in enumerate(_ROTATIONS):
        t[:, s] = t[:, s][:, list(perm)]
    return pos, t.reshape(-1, 4)


def per_tet_order(res):
    """Edge runs, NO tet runs (a seeded random vertex order per tet: ~24 shapes per chunk, too few tets per entry): the
    expansion marks no tets, edge_mark_kernel finds them behind it."""
    pos, tets = grids.kuhn_grid(res)
    rng = np.random.default_rng(res)
    return pos, np.ascontiguousarray(rng.permuted(tets, axis=1))


def shuffled_tets(res):
    """Edge runs and tet runs: the lattice numbering, the tet rows in seeded random order.  The ids of a tet entry fall
    into random compaction tiles; past 64 tiles (F > 64 * 8192, res >= 45) the per-CTA count table of runs_expand_kernel
    has colliding keys and takes its fallback."""
    pos, tets = grids.kuhn_grid(res)
    return pos, np.ascontiguousarray(tets[np.random.default_rng(res).permutation(tets.shape[0])])


def _crop(res):
    pos, tets = grids.kuhn_grid(res)
    keep = grids.capsule_sdf(pos[tets].astype(np.float64).mean(1), 0.25) > 0
    return pos, np.ascontiguousarray(tets[keep])


def cropped(res):
    """Edge runs and tet runs: the tets whose centroid is inside the dilated capsule body, lattice ids kept (isolated
    vertices, partial lane masks, chunks without any entry)."""
    return _crop(res)


def cropped_compacted(res):
    """The same tets, vertex ids compacted in axis order: the differences of a shape vary from row to row.  Edge runs at
    every size; tet runs from res 12 on (4.5 tets per entry), not at res 9 (too few tets per entry)."""
    pos, tets = _crop(res)
    used = np.unique(tets)
    remap = np.full(pos.shape[0], -1, np.int64)
    remap[used] = np.arange(used.shape[0])
    return np.ascontiguousarray(pos[used]), np.ascontiguousarray(remap[tets])


def box(res):
    """Edge runs and tet runs on anisotropic boxes: res 7 -> 7 x 5 x 19 cells, N = 960 (N % 32 == 0: the last chunk is
    full and its windows reach into the spare word); other res -> 4 x 12 x 32 cells, N = 2145 (N % 32 == 1: a last chunk
    of one vertex)."""
    return box_grid(7, 5, 19) if res == 7 else box_grid(4, 12, 32)


def lattice_plus_degenerate(res):
    """Edge runs and tet runs: a Kuhn lattice plus 40 tets that repeat a vertex (self edges (v, v): d = 0 edge entries,
    tet shapes with a zero difference)."""
    pos, tets = grids.kuhn_grid(res)
    rng = np.random.default_rng(res)
    extra = tets[rng.choice(tets.shape[0], 40, replace=False)].copy()
    src, dst = rng.integers(0, 4, 40), rng.integers(1, 4, 40)
    dst = (src + dst) % 4                                           # another slot of the same tet
    extra[np.arange(40), dst] = extra[np.arange(40), src]
    tets = np.concatenate([tets, extra])
    assert np.unique(tets, axis=0).shape[0] == tets.shape[0]       # no two tets list the same vertices in the same order
    return pos, np.ascontiguousarray(tets)


#: family -> (build(res), expected (edge runs, tet runs) on the scan path)
FAMILIES = {
    "rotated": (rotated, (True, True)),
    "per_tet_order": (per_tet_order, (True, False)),
    "shuffled_tets": (shuffled_tets, (True, True)),
    "cropped": (cropped, (True, True)),
    "cropped_compacted": (cropped_compacted, None),                 # depends on res: expected_form()
    "box": (box, (True, True)),
    "lattice_plus_degenerate": (lattice_plus_degenerate, (True, True)),
}

#: sizes on the B200: shuffled_tets large enough for colliding count keys, cropped_compacted on both sides of the
#: tet-runs threshold, both box sizes
GPU_CASES = [("rotated", 16), ("per_tet_order", 16), ("shuffled_tets", 48), ("cropped", 24), ("cropped_compacted", 9),
             ("cropped_compacted", 24), ("box", 7), ("box", 32), ("lattice_plus_degenerate", 12)]

#: (class, type, output_watertight_template)
CONFIGS = {"gshell": ("GShell_Tets", None, True), "cloth": ("hmSDF_Tets", "cloth", True),
           "body": ("hmSDF_Tets", "body", True), "gshell_open": ("GShell_Tets", None, False)}


def expected_form(family, res):
    if family == "cropped_compacted":
        return {9: (True, False), 12: (True, True), 16: (True, True), 24: (True, True)}[res]
    return FAMILIES[family][1]


@functools.lru_cache(maxsize=None)
def family_grid(family, res):
    pos, tets = FAMILIES[family][0](res)
    pos.flags.writeable = tets.flags.writeable = False
    return pos, tets


def family_field(pos):
    """The capsule body dilated by 0.1 (a surface of a few hundred faces at res 9) and the garment band."""
    _, msdf = grids.capsule_garment_field(pos)
    return grids.capsule_sdf(pos, 0.1).astype(np.float32), msdf


def family_inputs(family, res):
    """family_field on the family's grid, positions jittered by a fraction of a cell (seeded) so that no interpolation
    weight is a round number."""
    pos, tets = family_grid(family, res)
    sdf, msdf = family_field(pos)
    rng = np.random.default_rng(7)
    pos = (pos + (0.2 / res) * rng.standard_normal(pos.shape)).astype(np.float32)
    return pos, sdf, msdf, tets


@functools.lru_cache(maxsize=None)
def _oracle(family, res, config):
    _, typ, wt = CONFIGS[config]
    pos, sdf, msdf, tets = family_inputs(family, res)
    fwd = O.extract_forward(pos, sdf, msdf, tets, -1 if typ == "body" else 1, wt)
    rng = np.random.default_rng(5)
    grads = dict(g_verts_aug=rng.standard_normal(fwd["verts_aug"].shape).astype(np.float32),
                 g_msdf=rng.standard_normal(fwd["msdf"].shape).astype(np.float32),
                 g_msdf_watertight=rng.standard_normal(fwd["msdf_watertight"].shape).astype(np.float32),
                 g_vertices_watertight=(rng.standard_normal(fwd["vertices_watertight"].shape).astype(np.float32) if wt else None))
    want = O.extract_backward(fwd, grads["g_verts_aug"], grads["g_msdf"], grads["g_vertices_watertight"],
                              grads["g_msdf_watertight"])
    return fwd, grads, want


def assert_table_form(tets, n_grid, form):
    """The edge table(s) built for this tet array have the run-length form `form` = (edge runs, tet runs)."""
    from d3human_code_b200 import extract as E
    ents = [ent[1] for ent in E._static_cache.values()
            if ent[1] is not None and tuple(ent[2].shape) == tuple(tets.shape) and ent[1][0].shape[0] == n_grid + 1]
    assert ents, "no static edge table was built"
    for tab in ents:
        assert (tab[10][0] is not None, tab[11][0] is not None) == tuple(form), "table form"


def check_family(dev, edges_mode, family, res, config):
    """One family, one configuration: the drop-in class against the oracle (outputs exact, gradients normwise), then the
    integer intermediates of the library call (counts, crossing edges, corners) exact, then the table form."""
    from d3human_code_b200 import extract as E
    cls, typ, wt = CONFIGS[config]
    pos, sdf, msdf, tets = family_inputs(family, res)
    n = pos.shape[0]
    fwd, grads, (g_pos, g_sdf, g_msdf) = _oracle(family, res, config)
    assert fwd["faces_aug"].shape[0] > 0 and fwd["edge_a"].shape[0] > 0          # the case is not vacuous
    out, g = G._run(dev, pos, sdf, msdf, tets, cls, typ, wt, grads)
    assert out["extra_keys"] == fwd["extra_keys"]
    for k in ("faces_aug", "verts_aug", "msdf", "msdf_watertight", "msdf_boundary"):
        U.assert_exact(k, out[k], fwd[k])
    if wt:
        assert out["n_verts_watertight"] == fwd["n_verts_watertight"]
        U.assert_exact("faces_watertight", out["faces_watertight"], fwd["faces_watertight"])
        U.assert_exact("vertices_watertight", out["vertices_watertight"], fwd["vertices_watertight"])
    U.assert_close_normwise("grad_pos", g[0], g_pos, U.GRAD_RTOL)
    U.assert_close_normwise("grad_sdf", g[1], g_sdf, U.GRAD_RTOL)
    if typ == "body":
        assert g[2] is None
    else:
        U.assert_close_normwise("grad_msdf", g[2], g_msdf, U.GRAD_RTOL)
    # integer intermediates (test_integer_intermediates_match_oracle): classification counts, crossing edges, corners
    tt = E.packed_tets(torch.tensor(tets, device=dev), n)
    static = E.static_edges_for(tt, n)
    assert (static is not None) == (edges_mode != "sort")
    r = E.forward_raw(torch.tensor(pos, device=dev), torch.tensor(sdf, device=dev), torch.tensor(msdf, device=dev), tt,
                      typ == "body", wt, static=static)
    c = r.frames[0].counts
    assert c["n_valid_tets"] == fwd["fv"] and c["n_tri_tets"] == fwd["t1"] and c["n_quad_tets"] == fwd["t2"]
    assert c["n_verts"] == fwd["n_verts_watertight"] and c["n_faces_aug"] == fwd["faces_aug"].shape[0]
    assert c["bucket_polys"] == tuple(int(x // k) for x, k in zip(fwd["bucket_counts"], (1, 2, 1, 2, 3, 4)))
    edges = r.tape_edges(0).cpu().numpy()
    U.assert_exact("edge_a", edges[:, 0].astype(np.int64), fwd["edge_a"])
    U.assert_exact("edge_b", edges[:, 1].astype(np.int64), fwd["edge_b"])
    U.assert_exact("corners", r.tape_corners(0).cpu().numpy().astype(np.int64), fwd["corners"])
    if edges_mode == "scan":
        assert_table_form(tets, n, expected_form(family, res))


_FUSED_TYPES = ("cloth", "cloth", "body", "cloth", "cloth")


@functools.lru_cache(maxsize=None)
def _fused_oracle(family, res):
    B = len(_FUSED_TYPES)
    pos, tets = family_grid(family, res)
    sdf, msdf = family_field(pos)
    pos_b = np.stack([pos + grids.frame_offsets(pos.shape[0], res, f) for f in range(B)]).astype(np.float32)
    fwd = [O.extract_forward(pos_b[i], sdf, msdf, tets, -1 if _FUSED_TYPES[i] == "body" else 1, True) for i in range(B)]
    rng = np.random.default_rng(3)
    ups = [(rng.standard_normal(f["verts_aug"].shape).astype(np.float32), rng.standard_normal(f["msdf"].shape).astype(np.float32))
           for f in fwd]
    want_pos, want_sdf, want_msdf = np.zeros_like(pos_b), np.zeros_like(sdf), np.zeros_like(msdf)
    for i, f in enumerate(fwd):
        w = O.extract_backward(f, ups[i][0], ups[i][1])
        want_pos[i], want_sdf = w[0], want_sdf + w[1]
        if _FUSED_TYPES[i] != "body":
            want_msdf += w[2]
    return pos_b, sdf, msdf, tets, fwd, ups, (want_pos, want_sdf, want_msdf)


def check_fused_batch(dev, edges_mode, family, res, shrink):
    """extract_frames: B = 5 frames with per-frame offsets on shared sdf / msdf, four cloth frames (fused on the
    run-length path, one topology search) and one body frame, on 3 lanes -- every frame exact against the oracle,
    gradients summed over the frames.  shrink: the plan capacities are cut after a first batch, so that every list (the
    item lists of the expansion among them) overflows and the host re-runs with room."""
    from d3human_code_b200 import extract as E
    pos_b, sdf, msdf, tets, fwd, ups, (want_pos, want_sdf, want_msdf) = _fused_oracle(family, res)
    types = list(_FUSED_TYPES)
    tt = torch.tensor(tets, device=dev)
    for rnd in range(2 if shrink else 1):
        if rnd == 1:
            for plan in E._plans.values():
                plan.cap_tets, plan.cap_v, plan.cap_va, plan.cap_fw, plan.cap_fa = 96, 48, 96, 48, 48
        tp = torch.tensor(pos_b, device=dev, requires_grad=True)
        ts = torch.tensor(sdf[:, None], device=dev, requires_grad=True)
        tm = torch.tensor(msdf, device=dev, requires_grad=True)
        outs = E.extract_frames(tp, ts, tm, tt, types=types, lanes=3)
        loss = 0.0
        for i, o in enumerate(outs):
            U.assert_exact(f"faces_aug[{i}]", o[1].cpu().numpy(), fwd[i]["faces_aug"])
            U.assert_exact(f"verts_aug[{i}]", o[0].detach().cpu().numpy(), fwd[i]["verts_aug"])
            U.assert_exact(f"msdf[{i}]", o[5]["msdf"].detach().cpu().numpy(), fwd[i]["msdf"])
            U.assert_exact(f"faces_watertight[{i}]", o[5]["faces_watertight"].cpu().numpy(), fwd[i]["faces_watertight"])
            U.assert_exact(f"vertices_watertight[{i}]", o[5]["vertices_watertight"].detach().cpu().numpy(),
                           fwd[i]["vertices_watertight"])
            loss = loss + (o[0] * torch.tensor(ups[i][0], device=dev)).sum() + (o[5]["msdf"] * torch.tensor(ups[i][1], device=dev)).sum()
        loss.backward()
        U.assert_close_normwise("grad_pos", tp.grad.cpu().numpy(), want_pos, U.GRAD_RTOL)
        U.assert_close_normwise("grad_sdf", ts.grad.cpu().numpy().reshape(-1), want_sdf, 1e-4)
        U.assert_close_normwise("grad_msdf", tm.grad.cpu().numpy(), want_msdf, 1e-4)
    if edges_mode == "scan":
        assert_table_form(tets, pos_b.shape[1], expected_form(family, res))


def check_scrambled_layout_forced_runs(dev, edges_mode, monkeypatch, res):
    """The scrambled SMPL-X layout with the compression forced (_RUNS_MIN_EDGES = 0): about one edge per entry, item lists
    at their longest, differences up to N."""
    from d3human_code_b200 import extract as E
    monkeypatch.setattr(E, "_RUNS_MIN_EDGES", 0)
    g = grids.smplx_layout_grid(res, dilate=0.15, seed=2)
    pos, tets = g["v"], g["f"]
    sdf, msdf = grids.capsule_garment_field(pos)
    for config, (cls, typ, wt) in CONFIGS.items():
        fwd = O.extract_forward(pos, sdf, msdf, tets, -1 if typ == "body" else 1, wt)
        rng = np.random.default_rng(9)
        gv = rng.standard_normal(fwd["verts_aug"].shape).astype(np.float32)
        gm = rng.standard_normal(fwd["msdf"].shape).astype(np.float32)
        out, g = G._run(dev, pos, sdf, msdf, tets, cls, typ, wt, dict(g_verts_aug=gv, g_msdf=gm))
        for k in ("faces_aug", "verts_aug", "msdf", "msdf_watertight"):
            U.assert_exact(f"{k}[{config}]", out[k], fwd[k])
        if wt:
            U.assert_exact(f"faces_watertight[{config}]", out["faces_watertight"], fwd["faces_watertight"])
            U.assert_exact(f"vertices_watertight[{config}]", out["vertices_watertight"], fwd["vertices_watertight"])
        g_pos, g_sdf, g_msdf = O.extract_backward(fwd, gv, gm)
        U.assert_close_normwise("grad_pos", g[0], g_pos, U.GRAD_RTOL)
        U.assert_close_normwise("grad_sdf", g[1], g_sdf, U.GRAD_RTOL)
        if typ != "body":
            U.assert_close_normwise("grad_msdf", g[2], g_msdf, U.GRAD_RTOL)
    if edges_mode == "scan":
        from d3human_code_b200 import extract as E
        tab = [ent[1] for ent in E._static_cache.values() if ent[1] is not None]
        assert tab and all(t[10][0] is not None and t[10][0].shape[0] * 2 > t[2] for t in tab)   # < 2 edges per entry
        assert all(t[11][0] is not None for t in tab)


# ---------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("family,res", GPU_CASES)
def test_family_matches_oracle(dev, edges_mode, family, res, config):
    check_family(dev, edges_mode, family, res, config)


@pytest.mark.parametrize("shrink", [False, True])
@pytest.mark.parametrize("family,res", [("rotated", 16), ("shuffled_tets", 16), ("per_tet_order", 16)])
def test_fused_batch_on_family(dev, edges_mode, family, res, shrink):
    check_fused_batch(dev, edges_mode, family, res, shrink)


def test_scrambled_layout_with_forced_runs(dev, edges_mode, monkeypatch):
    check_scrambled_layout_forced_runs(dev, edges_mode, monkeypatch, 24)
