"""The emulated kernels under AddressSanitizer + UBSan (alignment, bounds): the product .cu files are compiled a second
time with -fsanitize=address,alignment,bounds and a selection of the emulated parity tests runs against that library in
a child process that preloads libasan.  Every torch buffer the kernels touch (inputs, outputs, tapes, workspaces) is a
heap allocation with red zones, so an out-of-bounds load / store by any emulated CUDA thread, a misaligned 8 / 16-byte
vector access or an out-of-range local-array index aborts the child with the .cu file and line -- the offline stand-in
for `compute-sanitizer --tool memcheck`.  (Regions carved out of ONE workspace allocation are not separated from each
other.)  Test infrastructure only."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# Tests that raise through torch's C++ autograd engine are left out: with libasan preloaded into a non-instrumented
# python its __cxa_throw interceptor cannot find the real one and aborts (a limitation of the preload, not a finding).
SELECTION = [                             # ~40 s: every golden case on the three edge paths + the newest kernels
    "tests/test_emu_parity.py::test_golden",
    "tests/test_emu_parity.py::test_regrowth",
    "tests/test_emu_parity.py::test_tangent_gradients",
    "tests/test_emu_parity.py::test_fused_frames_shared_topology_and_regrowth",   # fused frames, shared / kept topology
    "tests/test_emu_parity.py::test_compact_gradient_return",
    "tests/test_emu_lbs.py",                                                      # the skinning kernels at their edges (+50 s)
    "tests/test_emu_mlp.py",                                                      # the SDF network at its edges
]
FULL = SELECTION + [                      # D3H_SAN_FULL=1: another four minutes (clean at the end of round 2)
    "tests/test_emu_mesh.py",
    "tests/test_emu_parity.py::test_fused_pair_equals_two_calls",
    "tests/test_emu_parity.py::test_tet_edge_rank_table_variant",
    "tests/test_emu_parity.py::test_mark_rows_variant",
    "tests/test_emu_parity.py::test_integer_intermediates",
    "tests/test_emu_parity.py::test_batches",
    "tests/test_emu_parity.py::test_tet_range_sharding",
    "tests/test_emu_parity.py::test_random_tet_soups",
    "tests/test_emu_parity.py::test_tet_soups_with_repeated_vertices",
    "tests/test_emu_parity.py::test_pipelined_groups_and_split",
    "tests/test_emu_parity.py::test_fuzz_forward_against_oracle",
]


def _libasan():
    try:
        path = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        return None
    return path if os.path.isabs(path) and os.path.exists(path) else None


def test_emulated_kernels_are_clean_under_asan_and_ubsan():
    asan = _libasan()
    if asan is None:
        pytest.skip("gcc's libasan.so not found")
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0",
               UBSAN_OPTIONS="print_stacktrace=1")
    tests = FULL if os.environ.get("D3H_SAN_FULL") == "1" else SELECTION
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "san_runner.py")] + tests, cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=1500)
    tail = (res.stdout + res.stderr)[-4000:]
    assert res.returncode == 0, tail
    assert " passed" in res.stdout, tail
