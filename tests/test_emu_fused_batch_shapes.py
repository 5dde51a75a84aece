"""tests/test_fused_batch_shapes.py on the functional emulation of the kernels (tests/emu, fixtures of
tests/test_emu_parity.py): the same case bodies on smaller grids (res 12 and 15); the 128^3 case is GPU only."""
import pytest

from tests import test_fused_batch_shapes as T
from tests.test_emu_parity import dev, edges_mode, emu_lib_path  # noqa: F401  (fixtures)


@pytest.mark.parametrize("typ", ["cloth", "body"])
@pytest.mark.parametrize("B", [8, 9, 17])
def test_eight_rows_per_launch(dev, edges_mode, B, typ):
    T._skip_unless_scan(edges_mode)
    T.eight_rows_case(dev, 12, B, typ, skip=(11,) if B == 17 else ())


def test_thirty_three_frames_three_adjoint_launches(dev, edges_mode):
    T._skip_unless_scan(edges_mode)
    T.eight_rows_case(dev, 12, 33, "cloth")


@pytest.mark.parametrize("which", ["empty", "small", "tiles", "tiles_plus_one"])
def test_polygon_counts_at_tile_edges(dev, edges_mode, which):
    T._skip_unless_scan(edges_mode)
    T.tile_edge_case(dev, 12, which)


def test_empty_frames_with_gradients_in_an_adjoint_batch(dev, edges_mode):
    T._skip_unless_scan(edges_mode)
    T.empty_frames_in_adjoint_batch_case(dev, 12)


@pytest.mark.parametrize("vary", ["sdf", "msdf"])
def test_alternating_fields_never_reuse_the_launch_before(dev, edges_mode, vary):
    T._skip_unless_scan(edges_mode)
    T.alternating_fields_case(dev, 12, vary)


def test_stacked_equal_rows_do_not_share(dev, edges_mode):
    T._skip_unless_scan(edges_mode)
    T.stacked_equal_rows_case(dev, 15)


def test_mixed_types_in_one_launch_do_not_share(dev, edges_mode):
    T._skip_unless_scan(edges_mode)
    T.mixed_types_case(dev, 12)


def test_regrowth_on_eight_lanes(dev, edges_mode):
    T._skip_unless_scan(edges_mode)
    T.regrowth_case(dev, 12)
