"""The numpy oracle against the LIVE reference (a checkout of the original project at D3H_REFERENCE_ROOT), and against
the PyTorch ops it restates (everywhere)."""
import numpy as np
import pytest
import torch

from oracle import gshell_oracle as O
from oracle.ref_loader import load_reference_class, reference_available
from d3human_code_b200 import grids
from tests import _util as U


def needs_reference(fn):
    return pytest.mark.reference(pytest.mark.skipif(not reference_available(), reason="needs a checkout of the original "
                                                    "project (D3H_REFERENCE_ROOT)")(fn))


@needs_reference
def test_case_tables_equal_reference():
    ref = load_reference_class("GShell_Tets", "cpu")
    for mine, theirs in ((O.TRIANGLE_TABLE, ref.triangle_table), (O.MESH_EDGE_TABLE, ref.mesh_edge_table),
                         (O.TRIANGLE_TABLE_TRI, ref.triangle_table_tri), (O.TRIANGLE_TABLE_QUAD, ref.triangle_table_quad),
                         (O.NUM_TRIANGLES_TABLE, ref.num_triangles_table), (O.BASE_TET_EDGES, ref.base_tet_edges),
                         (O.NUM_TRIANGLES_TRI_TABLE, ref.num_triangles_tri_table),
                         (O.NUM_TRIANGLES_QUAD_TABLE, ref.num_triangles_quad_table)):
        assert np.array_equal(mine, theirs.numpy())
    ref2 = load_reference_class("hmSDF_Tets", "cpu")
    assert np.array_equal(O.TRIANGLE_TABLE_QUAD, ref2.triangle_table_quad.numpy())


@pytest.mark.parametrize("n", [1, 2, 3, 16, 17, 100, 1254, 3548, 10033])
def test_linspace_restatement(n):
    want = torch.linspace(0, 1 - (1 / n), n, dtype=torch.float32).numpy()
    assert np.array_equal(O.linspace_f32(n), want)


@needs_reference
def test_uv_atlas_indexed_by_vertex_id():
    ref = load_reference_class("GShell_Tets", "cpu")
    for num_tets in (1, 7, 750, 6000):
        uvs, _ = ref.map_uv(torch.zeros(1, dtype=torch.long), num_tets * 2)
        k = np.arange(uvs.shape[0])
        assert np.array_equal(O.vertex_uv(k, num_tets), uvs.numpy())


def test_cross_restatement():
    rng = np.random.default_rng(0)
    a = rng.standard_normal((20000, 3)).astype(np.float32)
    b = (a * np.float32(1.7) + rng.standard_normal((20000, 3)).astype(np.float32) * np.float32(1e-3)).astype(np.float32)
    want = torch.cross(torch.tensor(a), torch.tensor(b), dim=-1).numpy()
    assert np.array_equal(O._cross_f32(a, b, -1), want)


def _run_reference(cls, typ, wt, pos, sdf, msdf, tets):
    obj = load_reference_class(cls, "cpu")
    tp = torch.tensor(pos, requires_grad=True)
    ts = torch.tensor(sdf[:, None], requires_grad=True)
    tm = torch.tensor(msdf, requires_grad=True)
    args = (tp, ts, tm, torch.from_numpy(tets)) + ((typ,) if cls == "hmSDF_Tets" else ()) + (wt,)
    return obj(*args), (tp, ts, tm)


@needs_reference
@pytest.mark.parametrize("res,field,cls,typ,wt", [
    (16, "sphere", "GShell_Tets", None, True),
    (20, "capsule", "hmSDF_Tets", "cloth", True),
    (20, "capsule", "hmSDF_Tets", "body", True),
    (10, "adv", "GShell_Tets", None, True),
    (10, "adv", "hmSDF_Tets", "body", False),
    (9, "adv", "GShell_Tets", None, False),
])
def test_oracle_matches_live_reference(res, field, cls, typ, wt):
    pos, tets = grids.kuhn_grid(res)
    if field == "sphere":
        sdf, msdf = grids.sphere_plane_field(pos)
    elif field == "capsule":
        sdf, msdf = grids.capsule_garment_field(pos)
    else:
        pos, sdf, msdf = grids.adversarial_field(pos, res, seed=res)
    (verts, faces, _, _, v_tng, extra), (tp, ts, tm) = _run_reference(cls, typ, wt, pos, sdf, msdf, tets)
    sign = -1 if typ == "body" else 1
    fwd = O.extract_forward(pos, sdf, msdf, tets, sign, wt)
    U.assert_exact("faces_aug", fwd["faces_aug"], faces.numpy())
    U.assert_exact("verts_aug", fwd["verts_aug"], verts.detach().numpy())
    U.assert_exact("msdf", fwd["msdf"], extra["msdf"].detach().numpy())
    U.assert_tangents_close("v_tng_aug", fwd["v_tng_aug"], v_tng.detach().numpy())
    assert tuple(extra.keys()) == fwd["extra_keys"]
    if wt:
        U.assert_exact("faces_watertight", fwd["faces_watertight"], extra["faces_watertight"].numpy())
        U.assert_exact("vertices_watertight", fwd["vertices_watertight"], extra["vertices_watertight"].detach().numpy())
        assert extra["n_verts_watertight"] == fwd["n_verts_watertight"]
    rng = np.random.default_rng(3)
    gv = rng.standard_normal(fwd["verts_aug"].shape).astype(np.float32)
    gm = rng.standard_normal(fwd["msdf"].shape).astype(np.float32)
    loss = (verts * torch.tensor(gv)).sum() + (extra["msdf"] * torch.tensor(gm)).sum()
    loss.backward()
    g_pos, g_sdf, g_msdf = O.extract_backward(fwd, gv, gm)
    U.assert_close_normwise("grad_pos", g_pos, tp.grad.numpy(), U.GRAD_RTOL)
    U.assert_close_normwise("grad_sdf", g_sdf, ts.grad.numpy()[:, 0], U.GRAD_RTOL)
    if typ == "body":
        assert tm.grad is None and g_msdf is None
    else:
        U.assert_close_normwise("grad_msdf", g_msdf, tm.grad.numpy(), U.GRAD_RTOL)


@needs_reference
@pytest.mark.parametrize("seed", range(18))
def test_oracle_matches_live_reference_on_random_tet_soups(seed):
    """Unstructured input far from a lattice: random vertex quadruples (a non-manifold tet soup, shared edges with
    arbitrary multiplicity), random positions, fields with exact zeros, random class / type / template flag.  The oracle
    must track the reference bit for bit on integers, positions and mSDF, and to tolerance on gradients."""
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(8, 60))
    f = int(rng.integers(1, 400))
    tets = np.stack([rng.permutation(n)[:4] for _ in range(f)]).astype(np.int64)
    if seed >= 12:     # tets drawn with replacement: repeated vertices inside a tet, self-edges, an edge met twice by a tet
        tets = rng.integers(0, n, size=(f, 4)).astype(np.int64)
    pos = rng.standard_normal((n, 3)).astype(np.float32)
    sdf = rng.standard_normal(n).astype(np.float32)
    msdf = rng.standard_normal(n).astype(np.float32)
    sdf[::7] = 0.0
    msdf[::5] = 0.0
    cls = "GShell_Tets" if seed % 2 == 0 else "hmSDF_Tets"
    typ = None if cls == "GShell_Tets" else ("cloth", "body")[(seed // 2) % 2]
    wt = seed % 3 != 0
    (verts, faces, _, _, v_tng, extra), (tp, ts, tm) = _run_reference(cls, typ, wt, pos, sdf, msdf, tets)
    fwd = O.extract_forward(pos, sdf, msdf, tets, -1 if typ == "body" else 1, wt)
    U.assert_exact("faces_aug", fwd["faces_aug"], faces.numpy())
    U.assert_exact("verts_aug", fwd["verts_aug"], verts.detach().numpy())
    U.assert_exact("msdf", fwd["msdf"], extra["msdf"].detach().numpy())
    assert tuple(extra.keys()) == fwd["extra_keys"]
    if wt:
        U.assert_exact("faces_watertight", fwd["faces_watertight"], extra["faces_watertight"].numpy())
        U.assert_exact("vertices_watertight", fwd["vertices_watertight"], extra["vertices_watertight"].detach().numpy())
    if verts.shape[0] == 0 or not verts.requires_grad:
        return
    gv = rng.standard_normal(fwd["verts_aug"].shape).astype(np.float32)
    gm = rng.standard_normal(fwd["msdf"].shape).astype(np.float32)
    ((verts * torch.tensor(gv)).sum() + (extra["msdf"] * torch.tensor(gm)).sum()).backward()
    g_pos, g_sdf, g_msdf = O.extract_backward(fwd, gv, gm)
    U.assert_close_normwise("grad_pos", g_pos, tp.grad.numpy(), U.GRAD_RTOL)
    U.assert_close_normwise("grad_sdf", g_sdf, ts.grad.numpy()[:, 0], 5 * U.GRAD_RTOL)
    if typ != "body":
        U.assert_close_normwise("grad_msdf", g_msdf, tm.grad.numpy(), U.GRAD_RTOL)


# The oracle's adjoint is float64 (the exact gradient of the fp32 forward); the reference back-propagates in fp32 and
# forms gw1/dd - (gw0*w0 + gw1*w1)/dd with gw0 ~ gw1, so ITS gradients carry a cancellation error that grows with the
# grid resolution (|pos| / |edge|).  Measured in this container (live reference, CPU, vs the oracle, normwise):
#   64^3 sphere 1.2e-5 / capsule 2.7e-6, 128^3 sphere 1.6e-5 / capsule 3.6e-5 (g_sdf; g_msdf 1.9e-5), 256^3 5.2e-5.
# So "oracle == reference to 1e-5" only holds at small sizes; at the BASELINE sizes the honest pin is: integers,
# positions and mSDF bit-exact, gradients within the reference's own fp32 noise.  The CUDA kernels are held to 1e-5
# against the ORACLE (tests/test_y_fullsize_parity.py), i.e. they are closer to the exact gradient than the reference.
def reference_gradient_noise_bound(res):
    return 4e-7 * res


@needs_reference
@pytest.mark.parametrize("res,field,cls,typ", [
    (64, "sphere", "GShell_Tets", None),          # BASELINE configs[0]
    (64, "capsule", "hmSDF_Tets", "cloth"),
    (64, "capsule", "hmSDF_Tets", "body"),
    (128, "capsule", "hmSDF_Tets", "cloth"),      # BASELINE configs[1]
])
def test_oracle_matches_live_reference_at_named_sizes(res, field, cls, typ):
    pos, tets = grids.kuhn_grid(res)
    sdf, msdf = (grids.sphere_plane_field if field == "sphere" else grids.capsule_garment_field)(pos)
    (verts, faces, _, _, v_tng, extra), (tp, ts, tm) = _run_reference(cls, typ, True, pos, sdf, msdf, tets)
    fwd = O.extract_forward(pos, sdf, msdf, tets, -1 if typ == "body" else 1, True)
    U.assert_exact("faces_aug", fwd["faces_aug"], faces.numpy())
    U.assert_exact("verts_aug", fwd["verts_aug"], verts.detach().numpy())
    U.assert_exact("msdf", fwd["msdf"], extra["msdf"].detach().numpy())
    U.assert_exact("faces_watertight", fwd["faces_watertight"], extra["faces_watertight"].numpy())
    U.assert_exact("vertices_watertight", fwd["vertices_watertight"], extra["vertices_watertight"].detach().numpy())
    gv = (2.0 * fwd["verts_aug"].astype(np.float64)).astype(np.float32)     # d/dverts of sum(verts^2)
    gm = np.ones_like(fwd["msdf"])
    ((verts * torch.tensor(gv)).sum() + (extra["msdf"] * torch.tensor(gm)).sum()).backward()
    g_pos, g_sdf, g_msdf = O.extract_backward(fwd, gv, gm)
    bound = reference_gradient_noise_bound(res)
    U.assert_close_normwise("grad_pos", g_pos, tp.grad.numpy(), U.GRAD_RTOL)       # no cancellation on this branch
    U.assert_close_normwise("grad_sdf", g_sdf, ts.grad.numpy()[:, 0], bound)
    if typ == "body":
        assert tm.grad is None and g_msdf is None
    else:
        U.assert_close_normwise("grad_msdf", g_msdf, tm.grad.numpy(), bound)


# ---------------------------------------------------------------------------------------------- tangent gradients
def _well_conditioned_tangent_upstream(fwd, rng, kappa_max=15.0):
    """Upstream gradients of v_tng_aug / v_tng_watertight that vanish on ill-conditioned rows (cancelling face normals /
    tangents: the gradient of a unit vector grows like 1 / |sum|, in the reference's autograd as well)."""
    kap = O.tangent_condition(fwd)
    nv = fwd["n_verts_watertight"]
    ok = (kap < kappa_max).astype(np.float32)[:, None]
    g_aug = rng.standard_normal(fwd["v_tng_aug"].shape).astype(np.float32) * ok
    g_wt = rng.standard_normal((nv, 3)).astype(np.float32) * ok[:nv]
    return g_aug, g_wt


@needs_reference
@pytest.mark.parametrize("res,field,cls,typ", [(12, "sphere", "GShell_Tets", None), (16, "capsule", "hmSDF_Tets", "cloth"),
                                               (14, "capsule", "hmSDF_Tets", "body"), (15, "sphere", "GShell_Tets", None)])
def test_oracle_tangent_gradients_match_live_reference(res, field, cls, typ):
    """SURVEY A.5 optional branch: gradients through v_tng (auto_normals, compute_tangents, Gram-Schmidt, the boundary
    interpolation of the tangents) -- the oracle's hand-derived float64 adjoint against the reference's fp32 autograd."""
    pos, tets = grids.kuhn_grid(res)
    sdf, msdf = (grids.sphere_plane_field if field == "sphere" else grids.capsule_garment_field)(pos)
    rng = np.random.default_rng(res)
    pos = (pos + 0.2 / res * rng.standard_normal(pos.shape)).astype(np.float32)      # break the lattice symmetry
    (verts, faces, _, _, v_tng, extra), (tp, ts, tm) = _run_reference(cls, typ, True, pos, sdf, msdf, tets)
    fwd = O.extract_forward(pos, sdf, msdf, tets, -1 if typ == "body" else 1, True)
    g_aug, g_wt = _well_conditioned_tangent_upstream(fwd, rng)
    assert (np.abs(g_aug).sum(-1) > 0).mean() > 0.3          # a good share of the rows takes part
    # 1. the tangent branch alone, 2. together with the position / mSDF outputs
    for with_rest in (False, True):
        tp.grad = ts.grad = tm.grad = None
        loss = (v_tng * torch.tensor(g_aug)).sum() + (extra["v_tng_watertight"] * torch.tensor(g_wt)).sum()
        gv = gm = None
        if with_rest:
            gv = rng.standard_normal(fwd["verts_aug"].shape).astype(np.float32)
            gm = rng.standard_normal(fwd["msdf"].shape).astype(np.float32)
            loss = loss + (verts * torch.tensor(gv)).sum() + (extra["msdf"] * torch.tensor(gm)).sum()
        loss.backward(retain_graph=True)
        g_pos, g_sdf, g_msdf = O.extract_backward(fwd, gv, gm, None, None, g_aug, g_wt)
        U.assert_close_normwise("grad_pos", g_pos, tp.grad.numpy(), 2e-4)
        U.assert_close_normwise("grad_sdf", g_sdf, ts.grad.numpy()[:, 0], 2e-4)
        if typ != "body":
            U.assert_close_normwise("grad_msdf", g_msdf, tm.grad.numpy(), 2e-4)
