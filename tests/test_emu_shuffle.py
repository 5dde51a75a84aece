"""The emulated kernels under a SHUFFLED schedule: blocks run in a random order and every scheduler sweep of a block
starts at a random thread in a random direction (tests/emu/emu_core.cpp, `d3h_emu_set_shuffle`).  On the GPU both orders
are arbitrary, so results must not depend on them: a shared variable read without the barrier that orders it after its
writer, a counter consumed before every block has added to it, or a test that expects float atomics to be reproducible
fails under some seed.  The second seed also POISONS every `torch.empty` / `torch.empty_like` result (0xCB bytes): on the
GPU fresh allocations and reused workspaces hold arbitrary data, so nothing may rely on zero-filled scratch or outputs.
A selection of the emulated parity tests, two seeds each.  Test infrastructure only."""
import contextlib
import ctypes

import pytest
import torch

from tests import test_emu_mesh as EM
from tests import test_emu_mlp as EMLP
from tests import test_emu_parity as EP
from tests import test_zz_mesh as ZM

emu_lib_path = EP.emu_lib_path          # module-scoped fixture: builds tests/emu/_build/libd3h_tets_emu.so


def _poisoned(fn):
    def wrapper(*args, **kwargs):
        t = fn(*args, **kwargs)
        if t.numel() and t.is_contiguous():
            t.view(torch.uint8).fill_(0xCB)
        return t
    return wrapper


@pytest.fixture(params=[11, 12])
def shuffled(request, emu_lib_path, monkeypatch):
    lib = ctypes.CDLL(emu_lib_path)
    lib.d3h_emu_set_shuffle.argtypes = [ctypes.c_ulonglong]
    lib.d3h_emu_set_shuffle(request.param)
    if request.param == 12:
        monkeypatch.setattr(torch, "empty", _poisoned(torch.empty))
        monkeypatch.setattr(torch, "empty_like", _poisoned(torch.empty_like))
    yield request.param
    lib.d3h_emu_set_shuffle(0)


@pytest.fixture(params=["sort", "static"])
def edges_mode(request):
    return request.param


dev = EP.dev                            # extraction: CPU tensors + the emulated library behind the real C ABI
mesh_dev = EM.dev


@pytest.mark.parametrize("name", ["capsule12_cloth", "adv6_body", "adv5_open", "three_faces"])
def test_extraction_golden(shuffled, dev, name):
    EP.G.test_cuda_matches_golden(dev, name)


def test_extraction_oracle(shuffled, dev):
    EP.G.test_cuda_matches_oracle(dev, 12, "adv", "hmSDF_Tets", "body", True)


@pytest.mark.parametrize("res,field", [(12, "adv")])
def test_fused_pair(shuffled, dev, edges_mode, res, field):
    if edges_mode != "static":
        pytest.skip("the fused pair runs on the static edge path")
    EP.Z.fused_pair_equals_two_calls(dev, res, field)


@pytest.mark.parametrize("name", ["mesh_extracted", "mesh_soup", "mesh_three", "mesh_fan"])
def test_mesh_golden(shuffled, mesh_dev, name):
    ZM.test_mesh_matches_golden(mesh_dev, name)


def test_mesh_oracle_hub_and_memo(shuffled, mesh_dev):
    ZM.test_mesh_matches_oracle(mesh_dev, 80, 2)
    ZM.test_hub_vertex_with_many_neighbours(mesh_dev)
    ZM.test_repeated_auto_normals_share_one_result(mesh_dev)


def test_mesh_soups(shuffled, mesh_dev):
    for seed in (0, 6):
        ZM.test_random_triangle_soups(mesh_dev, seed)
    for seed in (0, 5, 15):
        ZM.test_degenerate_soups(mesh_dev, seed)


mlp_dev = EMLP.dev                      # SDF network: the C ABI of the emulated library with CPU buffers


@pytest.fixture
def mlp_module_dev(mlp_dev, monkeypatch):
    """geometry/mlp.py on CPU tensors that pass as CUDA tensors (as test_emu_mlp.module_dev)"""
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: EP._Stream())
    monkeypatch.setattr(torch.cuda, "device", lambda dev=None: contextlib.nullcontext())
    return mlp_dev


@pytest.mark.parametrize("m,n,k", [(129, 192, 96), (257, 256, 288)])
def test_mlp_linear(shuffled, mlp_dev, m, n, k):
    for epi in ("mode1", "adjoint"):
        EMLP.T.linear_case(mlp_dev, m, n, k, epi)


def test_mlp_wgrad_and_head(shuffled, mlp_dev):
    EMLP.T.wgrad_case(mlp_dev, 2000, 128, 192, True)
    EMLP.T.head_case(mlp_dev, 3, 252, 513)


def test_mlp_module(shuffled, mlp_module_dev):
    EMLP.T.module_case(mlp_module_dev, "f11_d256_o8_skip_last", 129, True)
