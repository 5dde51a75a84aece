"""Loader for the LIVE reference extraction classes (test infrastructure only).

Reads `geometry/gshell_tets.py` / `geometry/hmsdf_tets_split.py` from a checkout of the original D3Human-code
project at run time (nothing is copied into this repo), swaps the hard-coded 'cuda' device literals for the requested
device (the reference hard-codes device='cuda' 19 times, e.g. gshell_tets.py:108) and stubs the two imports
of render/util.py:12-13 that the extraction path never uses.  The checkout is not part of this repository: point
D3H_REFERENCE_ROOT at it to run the live-reference tests; without it they skip and the committed goldens (written from
the original by oracle/make_golden*.py) stand in for it.
"""
from __future__ import annotations

import os
import sys
import types

REF_ROOT = os.environ.get("D3H_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "geometry", "gshell_tets.py"))


def load_reference_class(which: str = "GShell_Tets", device: str = "cpu"):
    """which in {"GShell_Tets", "hmSDF_Tets"} -> an instance of the reference class living on `device`."""
    rel = {"GShell_Tets": "geometry/gshell_tets.py", "hmSDF_Tets": "geometry/hmsdf_tets_split.py"}[which]
    for name in ("nvdiffrast", "nvdiffrast.torch", "imageio"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["nvdiffrast"].torch = sys.modules["nvdiffrast.torch"]
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    with open(os.path.join(REF_ROOT, rel)) as fh:
        src = fh.read()
    if device != "cuda":
        src = src.replace("device='cuda'", f"device='{device}'").replace('device="cuda"', f'device="{device}"')
    mod = types.ModuleType("_d3h_ref_" + which)
    exec(compile(src, rel, "exec"), mod.__dict__)
    return getattr(mod, which)()


def load_reference_mesh(device: str = "cpu"):
    """-> the reference's `render/mesh.py` as a module living on `device` (Mesh :139, auto_normals :418).

    `render/mesh.py:14-15` imports `obj` -> `material` -> `mlptexture`, which needs tinycudann (render/mlptexture.py:11);
    none of it is used by Mesh / auto_normals, so the import is stubbed like nvdiffrast above."""
    for name in ("nvdiffrast", "nvdiffrast.torch", "imageio", "tinycudann"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["nvdiffrast"].torch = sys.modules["nvdiffrast.torch"]
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    rel = "render/mesh.py"
    with open(os.path.join(REF_ROOT, rel)) as fh:
        src = fh.read()
    if device != "cuda":
        src = src.replace("device='cuda'", f"device='{device}'").replace('device="cuda"', f'device="{device}"')
    mod = types.ModuleType("_d3h_ref_mesh")
    mod.__package__ = "render"
    exec(compile(src, rel, "exec"), mod.__dict__)
    return mod


def load_reference_mlp():
    """-> the reference's `geometry/mlp.py` as a module (MLP :9-45) next to its `geometry/embedding.py`, without executing
    anything else of the `geometry` package (hmsdf.py needs pysdf / trimesh / nvdiffrast)."""
    import importlib.util
    pkg_name = "_d3h_ref_geometry"
    if pkg_name + ".mlp" in sys.modules:
        return sys.modules[pkg_name + ".mlp"]
    pkg = types.ModuleType(pkg_name)
    pkg.__path__ = [os.path.join(REF_ROOT, "geometry")]
    sys.modules[pkg_name] = pkg
    for sub in ("embedding", "mlp"):
        spec = importlib.util.spec_from_file_location(f"{pkg_name}.{sub}", os.path.join(REF_ROOT, "geometry", sub + ".py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[f"{pkg_name}.{sub}"] = mod
        spec.loader.exec_module(mod)
    return sys.modules[pkg_name + ".mlp"]


def load_reference_lbs_methods():
    """-> (interpolate_weights, apply_lbs_inverse): the two methods of `deform/smplx_exavatar_deformer.py:363-421` as plain
    functions of a duck-typed `self` (attributes vs_template, lbs_weights, k), compiled from the reference source text with
    a brute-force stand-in for `pytorch3d.ops.knn_points` (K nearest by squared distance, ascending; pytorch3d is not
    installed here).  The class itself cannot be built: it loads the SMPL-X model files."""
    import ast
    import torch

    def knn_points(p1, p2, K=1):
        d = ((p1[:, :, None, :] - p2[:, None, :, :]) ** 2).sum(-1)          # (N, P1, P2)
        dist, idx = torch.topk(d, K, dim=2, largest=False, sorted=True)
        return dist, idx, None

    path = os.path.join(REF_ROOT, "deform", "smplx_exavatar_deformer.py")
    with open(path) as fh:
        tree = ast.parse(fh.read())
    cls = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "SMPLX_Deformer"][0]
    wanted = [n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name in ("interpolate_weights", "apply_lbs_inverse")]
    mod = ast.Module(body=wanted, type_ignores=[])
    ns = {"torch": torch, "knn_points": knn_points}
    exec(compile(mod, path, "exec"), ns)
    return ns["interpolate_weights"], ns["apply_lbs_inverse"]
