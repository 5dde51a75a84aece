"""tests/test_fused_shared_tangents.py on the functional emulation of the kernels (tests/emu, fixtures of
tests/test_emu_parity.py): the same body, the same sizes."""
from tests import test_fused_shared_tangents as T
from tests.test_emu_parity import dev, edges_mode, emu_lib_path  # noqa: F401  (fixtures)


def test_fused_shared_topology_tangents_and_packed(dev, edges_mode):
    T.test_fused_shared_topology_tangents_and_packed(dev, edges_mode)
