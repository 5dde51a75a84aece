"""ctypes binding of libd3h_tets.so (C ABI declared in include/d3h_tets.h and include/d3h_mesh.h).

The library is the product: there is no Python / PyTorch fallback.  If it is missing or fails to load, every
entry point raises.  PyTorch is only used by the callers for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libd3h_tets.so")

D3H_OK, D3H_E_BADARG, D3H_E_CUDA, D3H_E_SMALLWS, D3H_E_TIMEOUT = 0, -1, -2, -3, -4
VERSION = 500

#: every symbol include/d3h_tets.h declares (tests/test_cabi.py checks the library exports all of them)
EXPORTED_SYMBOLS = (
    "d3h_version", "d3h_last_error_string", "d3h_workspace_bytes", "d3h_workspace_bytes_static",
    "d3h_backward_workspace_bytes",
    "d3h_pack_tets_i64", "d3h_check_tets_i32", "d3h_extract_forward", "d3h_wait_counts", "d3h_extract_backward",
    "d3h_extract_forward_batch", "d3h_extract_forward_batch_nojoin", "d3h_lanes_join", "d3h_extract_backward_batch", "d3h_tangent_backward", "d3h_gather_rows", "d3h_classify_range", "d3h_extract_from_records",
    "d3h_mesh_edges_workspace_bytes", "d3h_mesh_edges", "d3h_mesh_wait_counts", "d3h_mesh_normals_forward",
    "d3h_mesh_normals_backward",
    "d3h_lbs_blend", "d3h_lbs_blend_backward", "d3h_lbs_nearest_workspace_bytes", "d3h_lbs_nearest", "d3h_lbs_apply",
    "d3h_lbs_apply_backward",
    "d3h_mlp_embed", "d3h_mlp_embed_backward", "d3h_mlp_packed_weight_bytes", "d3h_mlp_pack_weight", "d3h_mlp_linear", "d3h_mlp_wgrad_workspace_bytes", "d3h_mlp_wgrad", "d3h_mlp_head", "d3h_mlp_head_backward",
    "d3h_mlp_embed_tangent", "d3h_mlp_embed_second_backward", "d3h_mlp_linear_tangent", "d3h_mlp_linear_adjoint",
    "d3h_mlp_head_second_backward",
    "d3h_profile_enable", "d3h_profile_kinds", "d3h_profile_kernel_name", "d3h_profile_read", "d3h_profile_timeline", "d3h_profile_scan_kernel", "d3h_trace_enable", "d3h_trace_read", "d3h_debug_table",
)


class Counts(C.Structure):  # d3h_counts
    _fields_ = [("n_valid_tets", C.c_int64), ("n_tri_tets", C.c_int64), ("n_quad_tets", C.c_int64),
                ("n_corners", C.c_int64), ("n_verts", C.c_int64), ("n_faces_aug", C.c_int64),
                ("bucket_polys", C.c_int64 * 6), ("bad_index", C.c_int64), ("overflow", C.c_int64), ("seq", C.c_int64),
                ("reserved", C.c_int64)]


COUNTS_WORDS = C.sizeof(Counts) // 8  # int64 words


class MeshCounts(C.Structure):  # d3h_mesh_counts (include/d3h_mesh.h)
    _fields_ = [("n_edges", C.c_int64), ("bad_index", C.c_int64), ("overflow", C.c_int64), ("seq", C.c_int64)]


class ForwardArgs(C.Structure):  # d3h_forward_args
    _fields_ = [("pos", C.c_void_p), ("sdf", C.c_void_p), ("msdf", C.c_void_p), ("tets", C.c_void_p),
                ("n_grid", C.c_int64), ("n_tets", C.c_int64), ("tet_begin", C.c_int64), ("tet_end", C.c_int64),
                ("msdf_negate", C.c_int32), ("watertight_template", C.c_int32),
                ("cap_valid_tets", C.c_int64), ("cap_verts", C.c_int64), ("cap_verts_aug", C.c_int64),
                ("cap_faces_wt", C.c_int64), ("cap_faces_aug", C.c_int64),
                ("verts_aug", C.c_void_p), ("v_tng_aug", C.c_void_p), ("msdf_aug", C.c_void_p),
                ("faces_aug", C.c_void_p), ("verts_wt", C.c_void_p), ("v_tng_wt", C.c_void_p),
                ("msdf_wt", C.c_void_p), ("faces_wt", C.c_void_p),
                ("tape_edges", C.c_void_p), ("tape_corners", C.c_void_p), ("tape_slots", C.c_void_p),
                ("tape_runs", C.c_void_p),
                ("zero_g_pos", C.c_void_p), ("zero_g_sdf", C.c_void_p), ("zero_g_msdf", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64), ("counts_host", C.c_void_p),
                ("seq", C.c_int64),
                ("edge_off", C.c_void_p), ("edge_ab", C.c_void_p), ("n_edges", C.c_int64), ("vacc", C.c_void_p),
                ("pair_verts_aug", C.c_void_p), ("pair_v_tng_aug", C.c_void_p), ("pair_msdf_aug", C.c_void_p),
                ("pair_faces_aug", C.c_void_p), ("pair_verts_wt", C.c_void_p), ("pair_v_tng_wt", C.c_void_p),
                ("pair_msdf_wt", C.c_void_p), ("pair_faces_wt", C.c_void_p), ("pair_vacc", C.c_void_p),
                ("pair_counts_host", C.c_void_p), ("pair_seq", C.c_int64), ("tet_edge_rank", C.c_void_p),
                ("edge_b", C.c_void_p), ("etet_off", C.c_void_p), ("etets", C.c_void_p), ("etets8", C.c_void_p),
                ("edge_rows", C.c_void_p), ("edge_row_off", C.c_void_p),
                ("edge_runs", C.c_void_p), ("edge_run_chunk", C.c_void_p), ("edge_run_ids", C.c_void_p), ("n_edge_runs", C.c_int64),
                ("tet_runs", C.c_void_p), ("tet_run_chunk", C.c_void_p), ("tet_run_ids", C.c_void_p), ("n_tet_runs", C.c_int64)]


class BackwardArgs(C.Structure):  # d3h_backward_args
    _fields_ = [("pos", C.c_void_p), ("sdf", C.c_void_p), ("msdf", C.c_void_p), ("n_grid", C.c_int64),
                ("msdf_negate", C.c_int32), ("grads_prezeroed", C.c_int32),
                ("tape_edges", C.c_void_p), ("tape_corners", C.c_void_p), ("tape_slots", C.c_void_p),
                ("tape_runs", C.c_void_p), ("verts_wt", C.c_void_p),
                ("msdf_wt", C.c_void_p), ("n_verts", C.c_int64), ("n_tri_tets", C.c_int64),
                ("n_quad_tets", C.c_int64),
                ("g_verts_aug", C.c_void_p), ("g_msdf_aug", C.c_void_p), ("g_verts_wt", C.c_void_p),
                ("g_msdf_wt", C.c_void_p),
                ("g_pos", C.c_void_p), ("g_sdf", C.c_void_p), ("g_msdf", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64), ("g_msdf_boundary", C.c_void_p),
                ("vacc", C.c_void_p), ("g_verts_tng", C.c_void_p), ("g_mvert_tng", C.c_void_p)]


class TangentBackwardArgs(C.Structure):  # d3h_tangent_backward_args
    _fields_ = [("verts_wt", C.c_void_p), ("msdf_wt", C.c_void_p), ("v_tng_wt", C.c_void_p), ("faces_wt", C.c_void_p),
                ("tape_corners", C.c_void_p), ("n_verts", C.c_int64), ("n_tri_tets", C.c_int64), ("n_quad_tets", C.c_int64),
                ("n_tets", C.c_int64), ("g_tng_aug", C.c_void_p), ("g_tng_wt", C.c_void_p), ("g_verts", C.c_void_p),
                ("g_mvert", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64)]


TET_RECORD_BYTES = 32  # sizeof(d3h_tet_record)

_lib = None


def lib() -> C.CDLL:
    """Load the shared library once.  Raises if it has not been built (`python d3human-code_b200/build.py`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA library is the only implementation of this package "
            "(no CPU fallback). Build it with `python d3human-code_b200/build.py` (needs nvcc).")
    L = C.CDLL(LIB_PATH)
    L.d3h_version.restype = C.c_int
    L.d3h_last_error_string.restype = C.c_char_p
    L.d3h_workspace_bytes.restype = C.c_int64
    L.d3h_workspace_bytes.argtypes = [C.c_int64, C.c_int64, C.c_int64]
    L.d3h_workspace_bytes_static.restype = C.c_int64
    L.d3h_workspace_bytes_static.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int64]
    L.d3h_backward_workspace_bytes.restype = C.c_int64
    L.d3h_backward_workspace_bytes.argtypes = [C.c_int64]
    L.d3h_pack_tets_i64.restype = C.c_int
    L.d3h_pack_tets_i64.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.d3h_check_tets_i32.restype = C.c_int
    L.d3h_check_tets_i32.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
    L.d3h_extract_forward.restype = C.c_int
    L.d3h_extract_forward.argtypes = [C.c_void_p, C.c_void_p]
    L.d3h_wait_counts.restype = C.c_int
    L.d3h_wait_counts.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
    L.d3h_extract_backward.restype = C.c_int
    L.d3h_extract_backward.argtypes = [C.c_void_p, C.c_void_p]
    L.d3h_extract_forward_batch.restype = C.c_int
    L.d3h_extract_forward_batch.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    L.d3h_extract_forward_batch_nojoin.restype = C.c_int
    L.d3h_extract_forward_batch_nojoin.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    L.d3h_lanes_join.restype = C.c_int
    L.d3h_lanes_join.argtypes = [C.c_void_p]
    L.d3h_extract_backward_batch.restype = C.c_int
    L.d3h_extract_backward_batch.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    L.d3h_tangent_backward.restype = C.c_int
    L.d3h_tangent_backward.argtypes = [C.c_void_p, C.c_void_p]
    L.d3h_gather_rows.restype = C.c_int
    L.d3h_gather_rows.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
    L.d3h_classify_range.restype = C.c_int
    L.d3h_classify_range.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.d3h_extract_from_records.restype = C.c_int
    L.d3h_extract_from_records.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]
    # include/d3h_mesh.h
    L.d3h_mesh_edges_workspace_bytes.restype = C.c_int64
    L.d3h_mesh_edges_workspace_bytes.argtypes = [C.c_int64, C.c_int64]
    L.d3h_mesh_edges.restype = C.c_int
    L.d3h_mesh_edges.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                 C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.d3h_mesh_wait_counts.restype = C.c_int
    L.d3h_mesh_wait_counts.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
    L.d3h_mesh_normals_forward.restype = C.c_int
    L.d3h_mesh_normals_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p]
    L.d3h_mesh_normals_backward.restype = C.c_int
    L.d3h_mesh_normals_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p]
    # include/d3h_mlp.h (the CPU emulation of tests/emu has no tensor-core stage: its library lacks these symbols; the
    # real library always exports them, tests/test_cabi.py)
    if hasattr(L, "d3h_mlp_linear"):
        vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
        L.d3h_mlp_embed.restype = C.c_int
        L.d3h_mlp_embed.argtypes = [vp, i64, i32, vp, i64, i32, vp]
        L.d3h_mlp_embed_backward.restype = C.c_int
        L.d3h_mlp_embed_backward.argtypes = [vp, i64, i32, vp, i64, vp, i32, vp]
        L.d3h_mlp_linear.restype = C.c_int
        L.d3h_mlp_linear.argtypes = [vp, i64, i64, i32, vp, i32, vp, i32, vp, i64, vp, i64, vp]
        L.d3h_mlp_packed_weight_bytes.restype = C.c_int64
        L.d3h_mlp_packed_weight_bytes.argtypes = [i32, i32]
        L.d3h_mlp_pack_weight.restype = C.c_int
        L.d3h_mlp_pack_weight.argtypes = [vp, i64, i32, i32, i32, i32, i32, i32, i32, vp, vp]
        L.d3h_mlp_wgrad.restype = C.c_int
        L.d3h_mlp_wgrad.argtypes = [vp, i64, vp, i64, i64, i32, i32, vp, i64, vp, vp, i64, vp]
        L.d3h_mlp_wgrad_workspace_bytes.restype = C.c_int64
        L.d3h_mlp_wgrad_workspace_bytes.argtypes = [i64, i32, i32]
        L.d3h_mlp_head.restype = C.c_int
        L.d3h_mlp_head.argtypes = [vp, i64, i64, i32, vp, vp, i32, vp, vp]
        L.d3h_mlp_head_backward.restype = C.c_int
        L.d3h_mlp_head_backward.argtypes = [vp, i64, i64, i32, vp, i32, vp, vp, i64, vp, vp, vp]
        L.d3h_mlp_embed_tangent.restype = C.c_int
        L.d3h_mlp_embed_tangent.argtypes = [vp, vp, i64, i32, vp, i64, i32, vp]
        L.d3h_mlp_embed_second_backward.restype = C.c_int
        L.d3h_mlp_embed_second_backward.argtypes = [vp, vp, i64, i32, vp, i64, vp, i64, vp, vp]
        L.d3h_mlp_linear_tangent.restype = C.c_int
        L.d3h_mlp_linear_tangent.argtypes = [vp, i64, i64, i32, vp, i32, vp, i64, vp, i64, vp, i64, vp]
        L.d3h_mlp_linear_adjoint.restype = C.c_int
        L.d3h_mlp_linear_adjoint.argtypes = [vp, i64, i64, i32, vp, i32, vp, i64, vp, i64, vp, i64, vp, i64, vp]
        L.d3h_mlp_head_second_backward.restype = C.c_int
        L.d3h_mlp_head_second_backward.argtypes = [vp, i64, vp, i64, vp, i64, vp, i64, i64, i32, vp, i32, vp, vp, i64, vp]
    # include/d3h_lbs.h (the CPU emulation of tests/emu has it too)
    if hasattr(L, "d3h_lbs_apply"):
        vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
        L.d3h_lbs_blend.restype = C.c_int
        L.d3h_lbs_blend.argtypes = [vp, vp, i64, i32, i32, vp, vp]
        L.d3h_lbs_blend_backward.restype = C.c_int
        L.d3h_lbs_blend_backward.argtypes = [vp, vp, i64, i32, vp, vp]
        L.d3h_lbs_nearest_workspace_bytes.restype = C.c_int64
        L.d3h_lbs_nearest_workspace_bytes.argtypes = [i64]
        L.d3h_lbs_nearest.restype = C.c_int
        L.d3h_lbs_nearest.argtypes = [vp, i64, vp, i64, vp, vp, i64, vp]
        L.d3h_lbs_apply.restype = C.c_int
        L.d3h_lbs_apply.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, vp]
        L.d3h_lbs_apply_backward.restype = C.c_int
        L.d3h_lbs_apply_backward.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.d3h_profile_enable.restype = C.c_int
    L.d3h_profile_enable.argtypes = [C.c_int]
    L.d3h_profile_kinds.restype = C.c_int
    L.d3h_profile_kernel_name.restype = C.c_char_p
    L.d3h_profile_kernel_name.argtypes = [C.c_int]
    L.d3h_profile_read.restype = C.c_int
    L.d3h_profile_read.argtypes = [C.c_void_p, C.c_void_p]
    L.d3h_profile_timeline.restype = C.c_int
    L.d3h_profile_timeline.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.d3h_profile_scan_kernel.restype = C.c_int
    L.d3h_profile_scan_kernel.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.d3h_trace_enable.restype = C.c_int
    L.d3h_trace_enable.argtypes = [C.c_int]
    L.d3h_trace_read.restype = C.c_int
    L.d3h_trace_read.argtypes = [C.c_void_p]
    L.d3h_debug_table.restype = C.c_int
    L.d3h_debug_table.argtypes = [C.c_int, C.c_void_p, C.c_int]
    if L.d3h_version() != VERSION:
        raise RuntimeError(f"libd3h_tets.so version {L.d3h_version()} does not match this package ({VERSION}); rebuild")
    _lib = L
    return L


def profile_enable(on: bool) -> None:
    lib().d3h_profile_enable(int(bool(on)))


def profile_read():
    """-> {kernel name: (total ms, launches)} since the last read; synchronises the recorded events."""
    L = lib()
    n = L.d3h_profile_kinds()
    ms = (C.c_float * n)()
    cnt = (C.c_int * n)()
    check(L.d3h_profile_read(ms, cnt), "d3h_profile_read")
    return {L.d3h_profile_kernel_name(k).decode(): (float(ms[k]), int(cnt[k])) for k in range(n) if cnt[k]}


def profile_timeline(cap: int = 4096):
    """-> [(start_ms, end_ms, kernel name, stream ordinal)] of every launch since the last read."""
    L = lib()
    a, b = (C.c_float * cap)(), (C.c_float * cap)()
    k, sid = (C.c_int * cap)(), (C.c_int * cap)()
    n = L.d3h_profile_timeline(a, b, k, sid, cap)
    if n < 0:
        check(n, "d3h_profile_timeline")
    return [(a[i], b[i], L.d3h_profile_kernel_name(k[i]).decode(), sid[i]) for i in range(n)]


def trace_enable(on: bool) -> None:
    check(lib().d3h_trace_enable(int(bool(on))), "d3h_trace_enable")


def trace_read():
    """-> {seq % 64: {kernel name: (start_ns, end_ns)}} of the forward kernels run since the last read."""
    import numpy as np
    L = lib()
    t = np.zeros((64, 24, 2), dtype=np.uint64)
    check(L.d3h_trace_read(t.ctypes.data), "d3h_trace_read")
    out = {}
    for f in range(64):
        row = {L.d3h_profile_kernel_name(k).decode(): (int(t[f, k, 0]), int(t[f, k, 1]))
               for k in range(min(24, L.d3h_profile_kinds())) if t[f, k, 0]}
        if row:
            out[f] = row
    return out


def check(rc: int, what: str) -> None:
    """Mirror of the reference plugins' TORCH_CHECK behaviour (torch_bindings.cpp:25-31): errors become RuntimeError."""
    if rc != 0:
        msg = lib().d3h_last_error_string().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")
