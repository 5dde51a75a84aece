"""tests/test_zzzzzzzzz_mlp_edges.py on the functional emulation of the kernels (tests/emu): the same case bodies at small
sizes, the C ABI driven with 16-byte aligned CPU buffers; the module cases with CPU tensors that claim to be CUDA tensors.
The emulation runs the tensor-core pipeline as the PTX ISA defines it -- mbarrier phases, bulk copies, the 128-byte
swizzle of the shared-memory descriptors, TF32 operands, tensor-memory lane quarters -- and aborts on a protocol error.
Test infrastructure only."""
import contextlib

import pytest
import torch

from d3human_code_b200 import _cabi
from tests import test_zzzzzzzzz_mlp_edges as T
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
    """geometry/mlp.py refuses CPU tensors and asks torch.cuda for the stream and the device: answered for the emulation"""
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: _Stream())
    monkeypatch.setattr(torch.cuda, "device", lambda dev=None: contextlib.nullcontext())
    return dev


# every M, N and K of the GPU grid at least once, every epilogue on each shape
LINEAR_SHAPES = [(1, 64, 32), (127, 192, 96), (128, 256, 288), (129, 128, 384), (255, 192, 64), (257, 64, 288)]


@pytest.mark.parametrize("epi", T.EPILOGUES)
@pytest.mark.parametrize("m,n,k", LINEAR_SHAPES)
def test_linear_epilogues_at_the_edges(dev, m, n, k, epi):
    T.linear_case(dev, m, n, k, epi)


@pytest.mark.parametrize("case", T.PACK_CASES, ids=lambda c: "t%d_n%d_k%d_np%d_kp%d" % c[:5])
def test_packed_weight_offsets_transpose_and_zero_fill(dev, case):
    T.pack_case(dev, *case)


WGRAD_CASES = [(1, 128, 64, True), (31, 256, 128, False), (33, 128, 192, True), (511, 256, 256, False),
               (512, 128, 128, True), (513, 256, 192, False), (513, 128, 64, True), (2000, 128, 256, True)]


@pytest.mark.parametrize("m,n,k,with_db", WGRAD_CASES)
def test_wgrad_point_ranges_and_bias(dev, m, n, k, with_db):
    T.wgrad_case(dev, m, n, k, with_db)


@pytest.mark.parametrize("d_out", range(1, 9))
@pytest.mark.parametrize("k", T.HEAD_K)
def test_output_layer_every_width(dev, d_out, k):
    T.head_case(dev, d_out, k, T.HEAD_M[(d_out + T.HEAD_K.index(k)) % len(T.HEAD_M)])


@pytest.mark.parametrize("layout", T.ENC_LAYOUTS)
@pytest.mark.parametrize("n_freq", T.ENC_FREQ)
def test_encoding_paths_and_frequencies(dev, n_freq, layout):
    T.encoding_case(dev, n_freq, layout, m=37)


@pytest.mark.parametrize("eikonal", [False, True], ids=["first_order", "eikonal"])
@pytest.mark.parametrize("m", [1, 128, 129])
@pytest.mark.parametrize("name", list(T.MODULE_CFGS))
def test_module_configurations(module_dev, name, m, eikonal):
    T.module_case(module_dev, name, m, eikonal)


def test_launch_above_48kb_without_the_attribute_fails():
    """the emulated runtime refuses a launch over 48 KB of dynamic shared memory unless the kernel's attribute allows it,
    as the CUDA runtime does (the GEMM kernels set it before their first launch)"""
    import ctypes
    lib = ctypes.CDLL(build_emu.build())
    lib.d3h_emu_launch_probe.argtypes = [ctypes.c_ulonglong]
    assert lib.d3h_emu_launch_probe(48 * 1024) == 0
    assert lib.d3h_emu_launch_probe(48 * 1024 + 16) == 1
