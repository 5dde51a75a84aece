"""tests/test_zero_in_backward.py on the functional emulation of the kernels (tests/emu, fixtures of
tests/test_emu_parity.py), at res 12.  CPU memory is not recycled the way the caching allocator recycles device memory,
so here every torch.empty / torch.empty_like result is filled with NaN instead: the gradient buffers the forward call
allocates are dirty whatever the allocator does."""
import pytest
import torch

from tests import test_zero_in_backward as Z
from tests import test_fused_batch_shapes as T
from tests.test_emu_parity import dev, edges_mode, emu_lib_path  # noqa: F401  (fixtures)


def _nan_filled(fn):
    def wrapper(*args, **kwargs):
        t = fn(*args, **kwargs)
        if t.is_floating_point():
            t.fill_(float("nan"))
        return t
    return wrapper


@pytest.fixture
def dirty(dev, monkeypatch):
    monkeypatch.setattr(torch, "empty", _nan_filled(torch.empty))
    monkeypatch.setattr(torch, "empty_like", _nan_filled(torch.empty_like))
    return lambda *shapes: None


@pytest.mark.parametrize("B", [8, 17])
def test_dirty_memory(dev, edges_mode, dirty, B):
    T._skip_unless_scan(edges_mode)
    Z.dirty_case(dev, dirty, 12, B, skip=(11,) if B == 17 else ())


def test_dirty_memory_empty_frames(dev, edges_mode, dirty):
    T._skip_unless_scan(edges_mode)
    Z.dirty_case(dev, dirty, 12, 17, empty_first=8)


def test_zero_fill_path(dev, edges_mode, dirty, monkeypatch):
    T._skip_unless_scan(edges_mode)
    Z.path_case(dev, dirty, monkeypatch, 12)


@pytest.mark.parametrize("api", ["frames", "packed"])
def test_shared_gradient_over_two_backward_calls(dev, edges_mode, dirty, api):
    T._skip_unless_scan(edges_mode)
    Z.shared_gradient_case(dev, dirty, 12, api)
