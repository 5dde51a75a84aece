"""Per-frame tangents of fused frames that share one topology.

Frames of a batch that share sdf and msdf are extracted in fused launches (grid.y = frame) on ONE topology: the surface
kernels do the integer and mSDF work of a polygon once, in their topology CTAs, and store it into every frame; each frame's
own CTAs compute only what needs its positions (normals, tangents, boundary vertex positions).  This checks every output
of that split per frame against the numpy oracle, with distinct per-frame positions so that a frame reading another
frame's vertices or accumulators shows, on more frames than workspaces so that the later rounds of launches keep the
topology of the first, and through both the per-frame and the packed API."""
import numpy as np
import pytest
import torch

from oracle import gshell_oracle as O
from d3human_code_b200 import grids
from tests import _util as U
from tests.test_cuda_parity import dev, edges_mode  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu


def test_fused_shared_topology_tangents_and_packed(dev, edges_mode):
    """11 frames on 4 workspaces (rounds of 4, 4 and 3 frames; the last two keep the topology of the first) on the shared
    capsule field: v_tng_aug, v_tng_watertight and msdf_boundary of every frame against the oracle, and the packed form of
    the same batch against the per-frame results.  1,122 polygons: four full 256-polygon tiles and a partial one."""
    if edges_mode != "scan":
        pytest.skip("frames are fused on the run-length path only")
    from d3human_code_b200.extract import extract_frames, extract_frames_async
    res, B, lanes = 20, 11, 4
    pos, tets = grids.kuhn_grid(res)
    sdf, msdf = grids.capsule_garment_field(pos)
    pos_b = np.stack([pos + grids.frame_offsets(pos.shape[0], res, f) for f in range(B)]).astype(np.float32)
    assert all(not np.array_equal(pos_b[0], pos_b[i]) for i in range(1, B))
    fwd = [O.extract_forward(pos_b[i], sdf, msdf, tets, 1, True) for i in range(B)]
    npoly = int(fwd[0]["t1"]) + int(fwd[0]["t2"])
    assert npoly > 2 * 256 and npoly % 256 != 0, npoly      # several polygon tiles, the last one partial
    assert B > lanes                                          # more frames than workspaces: later rounds reuse the topology
    tt = torch.tensor(tets, device=dev)

    def leaves():
        return (torch.tensor(pos_b, device=dev), torch.tensor(sdf[:, None], device=dev), torch.tensor(msdf, device=dev))

    outs = extract_frames(*leaves(), tt, types="cloth", lanes=lanes)
    assert len(outs) == B
    for i, (verts, faces, _, _, v_tng, extra) in enumerate(outs):
        f = fwd[i]
        kappa = O.tangent_condition(f)
        nv = int(f["n_verts_watertight"])
        U.assert_exact(f"faces_aug[{i}]", faces.cpu().numpy(), f["faces_aug"])
        U.assert_exact(f"verts_aug[{i}]", verts.cpu().numpy(), f["verts_aug"])
        U.assert_exact(f"msdf[{i}]", extra["msdf"].cpu().numpy(), f["msdf"])
        U.assert_exact(f"msdf_boundary[{i}]", extra["msdf_boundary"].cpu().numpy(), f["msdf_boundary"])
        U.assert_exact(f"faces_watertight[{i}]", extra["faces_watertight"].cpu().numpy(), f["faces_watertight"])
        U.assert_exact(f"vertices_watertight[{i}]", extra["vertices_watertight"].cpu().numpy(), f["vertices_watertight"])
        U.assert_tangents_conditioned(f"v_tng_aug[{i}]", v_tng.cpu().numpy(), f["v_tng_aug"], kappa, max_unchecked_frac=0.01)
        U.assert_tangents_conditioned(f"v_tng_watertight[{i}]", extra["v_tng_watertight"].cpu().numpy(),
                                      f["v_tng_watertight"], kappa[:nv], max_unchecked_frac=0.01)

    pk = extract_frames_async(*leaves(), tt, types="cloth", lanes=lanes).packed()
    assert len(pk) == B
    for i, (verts, faces, _, _, v_tng, extra) in enumerate(outs):
        va, v, fa, fw = (int(pk.n_verts_aug[i]), int(pk.n_verts_watertight[i]), int(pk.n_faces_aug[i]),
                         int(pk.n_faces_watertight[i]))
        assert (va, fa, v, fw) == (verts.shape[0], faces.shape[0], extra["n_verts_watertight"], extra["faces_watertight"].shape[0])
        assert torch.equal(pk.verts_aug[i, :va], verts) and torch.equal(pk.faces_aug[i, :fa], faces)
        assert torch.equal(pk.msdf[i, :va], extra["msdf"])
        assert torch.equal(pk.faces_watertight[i, :fw], extra["faces_watertight"])
        fr = pk.frame(i)
        assert torch.equal(fr[5]["msdf_boundary"], extra["msdf_boundary"])
        # tangents are sums of float atomics: the packed run against the oracle, like the per-frame one
        kappa = O.tangent_condition(fwd[i])
        U.assert_tangents_conditioned(f"packed v_tng_aug[{i}]", pk.v_tng_aug[i, :va].cpu().numpy(), fwd[i]["v_tng_aug"],
                                      kappa, max_unchecked_frac=0.01)
        U.assert_tangents_conditioned(f"packed v_tng_watertight[{i}]", pk.v_tng_watertight[i, :v].cpu().numpy(),
                                      fwd[i]["v_tng_watertight"], kappa[:v], max_unchecked_frac=0.01)
