"""tests/test_zzzzzzz_lbs_edges.py on the functional emulation of the kernels (tests/emu): the same case bodies, the C ABI
driven with 16-byte aligned CPU buffers; the module cases with CPU tensors that claim to be CUDA tensors.  The
benchmark-shape case is GPU only.  Test infrastructure only."""
import contextlib

import pytest
import torch

from d3human_code_b200 import _cabi
from tests import test_zzzzzzz_lbs_edges as T
from tests.test_emu_parity import _Stream, build_emu


@pytest.fixture(scope="module")
def emu_lib_path():
    return build_emu.build()


@pytest.fixture
def dev(emu_lib_path, monkeypatch):
    monkeypatch.setattr(_cabi, "LIB_PATH", emu_lib_path)
    monkeypatch.setattr(_cabi, "_lib", None)
    return torch.device("cpu")


@pytest.fixture
def module_dev(dev, monkeypatch):
    """deform/lbs.py refuses CPU tensors and asks torch.cuda for the stream: both answered for the emulation"""
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: _Stream())
    monkeypatch.setattr(torch.cuda, "device", lambda dev=None: contextlib.nullcontext())
    return dev


@pytest.mark.parametrize("n_zero", [0, 300])
@pytest.mark.parametrize("n_live", [255, 256, 257])
def test_live_row_counts_at_the_cta_edge(dev, n_live, n_zero):
    T.live_count_case(dev, n_live, n_zero)


@pytest.mark.parametrize("vt", [1, 1023, 1024, 1025, 2500])
def test_template_sizes_at_the_tile_edge(dev, vt):
    T.template_size_case(dev, vt)


def test_ties_go_to_the_lowest_index(dev):
    T.ties_case(dev)


@pytest.mark.parametrize("which", ["all_zero", "no_zero", "neg_zero"])
def test_zero_rows(dev, which):
    T.zero_rows_case(dev, which)


def test_sparse_weights(dev):
    T.sparse_weights_case(dev)


def test_inverse_swaps_rows(dev):
    T.pivot_case(dev)


def test_one_joint_is_rigid(dev):
    T.one_joint_case(dev)


def test_max_joints(dev):
    T.max_joints_case(dev)


def test_joint_counts_outside_the_table_are_refused(dev):
    T.joint_count_refused_case(dev)


@pytest.mark.parametrize("with_trans", [True, False])
def test_trans(dev, with_trans):
    T.trans_case(dev, with_trans)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_forward_inverse(dev, seed):
    T.forward_inverse_case(dev, seed)


@pytest.mark.parametrize("use_pts", [True, False])
def test_zero_rows_across_cta_boundaries(dev, use_pts):
    T.cta_boundaries_case(dev, use_pts)


def test_pts_null_gives_the_same_gradients(dev):
    T.pts_null_matches_case(dev)


def test_zero_upstream_gradient(dev):
    T.zero_upstream_case(dev)


@pytest.mark.parametrize("use_pts", [True, False])
def test_zero_rows_with_different_idx(dev, use_pts):
    T.mixed_zero_idx_case(dev, use_pts)


def test_no_points(dev):
    T.empty_case(dev)


@pytest.mark.parametrize("which", ["no_trans", "a_no_grad", "batched", "view_f64"])
def test_module(module_dev, which):
    T.module_case(module_dev, which)


def test_module_no_points(module_dev):
    T.module_empty_case(module_dev)


def test_module_interpolate_weights_of_two_frames(module_dev):
    T.module_weights_case(module_dev)
