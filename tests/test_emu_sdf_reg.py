"""tests/test_zzzzzzzzzz_sdf_reg.py on the functional emulation of the kernels (tests/emu): the same case bodies at small
sizes, with CPU tensors that claim to be CUDA tensors; once more under AddressSanitizer + UBSan and under
ThreadSanitizer (tests/emu/san_runner.py, as tests/test_emu_sanitize.py and tests/test_emu_racecheck.py start it), and on a
shuffled schedule with poisoned fresh allocations (as tests/test_emu_shuffle.py).  The benchmark-shape case is GPU only.
Test infrastructure only."""
import contextlib
import ctypes
import os
import subprocess
import sys

import pytest
import torch

from d3human_code_b200 import _cabi
from tests import test_zzzzzzzzzz_sdf_reg as T
from tests.test_emu_parity import _Stream, build_emu
from tests.test_emu_racecheck import _libtsan
from tests.test_emu_sanitize import _libasan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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
    """geometry/sdf_reg.py refuses CPU tensors and asks torch.cuda for the stream and the device: answered for the emulation"""
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: _Stream())
    monkeypatch.setattr(torch.cuda, "device", lambda dev=None: contextlib.nullcontext())
    return dev


@pytest.mark.parametrize("field", ["capsule", "random"])
@pytest.mark.parametrize("res,n", [(12, 2175), (12, 2176), (12, 2177), (3, None)])   # 32k - 1, 32k, 32k + 1; 64
def test_kuhn_vertex_counts_around_32(module_dev, res, n, field):
    T.kuhn_case(module_dev, res, n, field)


def test_single_tet(module_dev):
    T.single_tet_case(module_dev)


@pytest.mark.parametrize("n_chunks,diffs", [(255, (1,)), (256, (1,)), (257, (1,)), (129, (1, 33))])
def test_entry_counts_around_the_cta(module_dev, n_chunks, diffs):
    T.entries_case(module_dev, n_chunks, diffs)


def test_smplx_layout_takes_the_rows(module_dev):
    T.smplx_case(module_dev, 12)


@pytest.mark.parametrize("which", ["positive", "negative", "zero", "no_edges"])
def test_no_edge_selected(module_dev, which):
    T.m_zero_case(module_dev, which)


def test_one_edge_selected(module_dev):
    T.m_one_case(module_dev)


def test_nan(module_dev):
    T.nan_case(module_dev)


def test_shapes(module_dev):
    T.shapes_case(module_dev)


def test_float64(module_dev):
    T.f64_case(module_dev)


def test_row_order(module_dev):
    T.swapped_rows_case(module_dev)


def test_inplace_edit(module_dev):
    T.inplace_case(module_dev)


@pytest.mark.parametrize("g", [3.5, -0.25])
def test_upstream_gradient(module_dev, g):
    T.upstream_case(module_dev, g)


def test_extraction_edge_table(module_dev):
    T.extraction_table_case(module_dev)


def test_double_backward_raises(module_dev):
    T.double_backward_case(module_dev)


def test_bad_arguments_are_refused(dev):
    """the C ABI: both table forms, neither, a short workspace"""
    L = _cabi.lib()
    runs = torch.zeros(2, dtype=torch.int64)
    ws = torch.zeros(L.d3h_sdf_reg_workspace_bytes(64, 1) // 8 + 2, dtype=torch.int64)
    sdf, loss = torch.zeros(64), torch.zeros(1)
    assert L.d3h_sdf_reg_forward(sdf.data_ptr(), 64, runs.data_ptr(), runs.data_ptr(), 1, runs.data_ptr(), runs.data_ptr(),
                                 ws.data_ptr(), ws.numel() * 8, loss.data_ptr(), None) == _cabi.D3H_E_BADARG
    assert L.d3h_sdf_reg_forward(sdf.data_ptr(), 64, None, None, 0, None, None, ws.data_ptr(), ws.numel() * 8, loss.data_ptr(),
                                 None) == _cabi.D3H_E_BADARG
    assert L.d3h_sdf_reg_forward(sdf.data_ptr(), 64, runs.data_ptr(), runs.data_ptr(), 1, None, None, ws.data_ptr(), 64,
                                 loss.data_ptr(), None) == _cabi.D3H_E_BADARG
    assert b"d3h_sdf_reg_forward" in L.d3h_last_error_string()


# ---------------------------------------------------------------------------------------------- schedules and sanitizers
@pytest.fixture(params=[11, 12])
def shuffled(request, emu_lib_path, monkeypatch):
    from tests.test_emu_shuffle import _poisoned
    lib = ctypes.CDLL(emu_lib_path)
    lib.d3h_emu_set_shuffle.argtypes = [ctypes.c_ulonglong]
    lib.d3h_emu_set_shuffle(request.param)
    if request.param == 12:
        monkeypatch.setattr(torch, "empty", _poisoned(torch.empty))
        monkeypatch.setattr(torch, "empty_like", _poisoned(torch.empty_like))
    yield request.param
    lib.d3h_emu_set_shuffle(0)


def test_shuffled_schedule(shuffled, module_dev):
    T.kuhn_case(module_dev, 12, 2177, "random")
    T.entries_case(module_dev, 257, (1,))
    T.smplx_case(module_dev, 10)
    T.m_zero_case(module_dev, "zero")


# the cases that raise through torch's C++ autograd engine are left out under ASan (tests/test_emu_sanitize.py)
_SAN_SELECTION = ["tests/test_emu_sdf_reg.py", "-k", "not double_backward and not sanitize and not shuffled"]


def test_sanitize_asan():
    asan = _libasan()
    if asan is None:
        pytest.skip("gcc's libasan.so not found")
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0",
               UBSAN_OPTIONS="print_stacktrace=1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "san_runner.py")] + _SAN_SELECTION, cwd=ROOT,
                         env=env, capture_output=True, text=True, timeout=1500)
    tail = (res.stdout + res.stderr)[-4000:]
    assert res.returncode == 0 and " passed" in res.stdout, tail


def test_sanitize_threadsan():
    tsan = _libtsan()
    if tsan is None:
        pytest.skip("gcc's libtsan.so not found")
    env = dict(os.environ, LD_PRELOAD=tsan, D3H_EMU_VARIANT="tsan", OMP_NUM_THREADS="1",
               TSAN_OPTIONS="halt_on_error=0:report_signal_unsafe=0:exitcode=0")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "san_runner.py")] + _SAN_SELECTION + ["-s"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=2400)
    out = res.stdout + res.stderr
    reports = [l for l in out.splitlines() if l.startswith("SUMMARY: ThreadSanitizer") and "/csrc/" in l]
    assert not reports, "\n".join(sorted(set(reports))[:20])
    assert res.returncode == 0 and " passed" in out, out[-3000:]
