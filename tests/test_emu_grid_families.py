"""tests/test_grid_families.py on the CPU: the host tables of every grid family restate its tets and have the form the
family must produce, and the same test bodies run against the functional emulation of the kernels (tests/emu, fixture
of tests/test_emu_parity.py) at sizes the emulation finishes in seconds, on the run-length path ("scan") and the
per-call sort path.  The emulation checks the kernels' logic on these grids; races and memory ordering are left to the
GPU run of tests/test_grid_families.py."""
import numpy as np
import pytest
import torch

from d3human_code_b200 import extract as E
from tests import test_grid_families as F
from tests.test_emu_parity import dev, edges_mode, emu_lib_path  # noqa: F401  (fixtures)
from tests.test_host_layout import _check_edge_runs, _check_tet_runs

#: sizes on the emulation (res <= 16); shuffled_tets has no colliding count keys at this size (the B200 run has)
EMU_CASES = [("rotated", 9), ("per_tet_order", 9), ("shuffled_tets", 16), ("cropped", 16), ("cropped_compacted", 9),
             ("cropped_compacted", 12), ("box", 7), ("box", 32), ("lattice_plus_degenerate", 9)]


@pytest.mark.parametrize("family,res", list(dict.fromkeys(EMU_CASES + F.GPU_CASES)))
def test_family_tables_restate_the_tets(family, res):
    """The run-length tables built for every family: the edge entries restate the sorted edge list, the tet entries (where
    the family gets them) the tet array row for row, and the form is the one the family's comment names."""
    pos, tets = F.family_grid(family, res)
    n = pos.shape[0]
    off, ab, u, *_, (runs, run_chunk, run_ids), (truns, trun_chunk, trun_ids) = E.build_edge_table(
        torch.tensor(tets, dtype=torch.int32), n)
    assert (runs is not None, truns is not None) == F.expected_form(family, res)
    if (family, res) not in EMU_CASES:      # (the B200 sizes: the form only; restating them takes minutes in Python)
        return
    _check_edge_runs(ab, runs, run_chunk, run_ids, n)
    if truns is not None:
        _check_tet_runs(tets, truns, trun_chunk, trun_ids, n)
    else:                                   # forced: what the kernels would get below the threshold restates the tets too
        truns, trun_chunk, trun_ids = E.build_tet_runs(torch.tensor(tets, dtype=torch.int32), n, min_tets_per_entry=0)
        _check_tet_runs(tets, truns, trun_chunk, trun_ids, n)
    r = runs.numpy()
    if family in ("rotated", "lattice_plus_degenerate"):
        assert (truns.numpy()[:, :3] < 0).any()                    # windows below their chunk
    if family == "lattice_plus_degenerate":
        assert (r[:, 0] == 0).any() and (truns.numpy()[:, :3] == 0).any()   # self edges, shapes with a zero difference
    if family == "box":
        assert n % 32 == (0 if res == 7 else 1)
    if family == "cropped":
        assert np.unique(tets).shape[0] < n                         # isolated vertices


@pytest.mark.parametrize("config", list(F.CONFIGS))
@pytest.mark.parametrize("family,res", EMU_CASES)
def test_emu_family_matches_oracle(dev, edges_mode, family, res, config):
    if edges_mode == "sort" and config != "gshell":
        pytest.skip("the sort path does not read the run-length tables: one configuration per family")
    F.check_family(dev, edges_mode, family, res, config)


@pytest.mark.parametrize("family,res", [("shuffled_tets", 9), ("per_tet_order", 9)])
def test_emu_fused_batch_on_family(dev, edges_mode, family, res):
    if edges_mode != "scan":
        pytest.skip("frames are fused on the run-length path only")
    F.check_fused_batch(dev, edges_mode, family, res, shrink=True)


def test_emu_scrambled_layout_with_forced_runs(dev, edges_mode, monkeypatch):
    if edges_mode != "scan":
        pytest.skip("forced run-length tables: the scan path")
    F.check_scrambled_layout_forced_runs(dev, edges_mode, monkeypatch, 12)
