"""The emulated kernels under ThreadSanitizer: the product .cu files compiled with -fsanitize=thread, every emulated CUDA
thread a TSan fibre (tests/emu/emu_core.cpp, EMU_TSAN).  Fibre switches carry no synchronisation; happens-before edges
exist exactly where CUDA gives them -- __syncthreads, __syncwarp, device atomics, block / kernel boundaries -- so two
threads of a block touching the same shared or global address without one of those in between is reported with the .cu
file and line: the offline stand-in for `compute-sanitizer --tool racecheck` (consecutive blocks are ordered, see
emu_core.cpp, so races BETWEEN blocks are not seen).  A deliberately racy probe kernel checks that the detector works.
Runs in child processes with libtsan preloaded.  Test infrastructure only."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu")
SELECTION = [                              # ~40 s: every golden case on the three edge paths + the newest kernels
    "tests/test_emu_parity.py::test_golden",
    "tests/test_emu_parity.py::test_regrowth",
    "tests/test_emu_parity.py::test_tangent_gradients",
    "tests/test_emu_parity.py::test_fused_frames_shared_topology_and_regrowth",   # fused frames, shared / kept topology
    "tests/test_emu_lbs.py",                                                      # the skinning kernels at their edges (+30 s)
    "tests/test_emu_mlp.py",                                                      # the SDF network: mbarrier pipeline, tcgen05
]
FULL = SELECTION + [                       # D3H_RACECHECK_FULL=1: another four minutes (clean at the end of round 2)
    "tests/test_emu_mesh.py",
    "tests/test_emu_parity.py::test_batches",
    "tests/test_emu_parity.py::test_fused_pair_equals_two_calls",
    "tests/test_emu_parity.py::test_tet_edge_rank_table_variant",
    "tests/test_emu_parity.py::test_mark_rows_variant",
    "tests/test_emu_parity.py::test_integer_intermediates",
    "tests/test_emu_parity.py::test_tet_range_sharding",
    "tests/test_emu_parity.py::test_random_tet_soups",
    "tests/test_emu_parity.py::test_tet_soups_with_repeated_vertices",
    "tests/test_emu_parity.py::test_pipelined_groups_and_split",
]

PROBE = r"""
#include <cuda_runtime.h>
#include <stdio.h>
__global__ void probe(int* out, int with_barrier) {
  __shared__ int s_x;
  if (threadIdx.x == 0) s_x = 42;
  if (with_barrier) __syncthreads();
  out[threadIdx.x] = s_x;
}
int main(int argc, char** argv) {
  int* out = (int*)malloc(64 * sizeof(int));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2);
  cfg.blockDim = dim3(64);
  cudaLaunchKernelEx(&cfg, probe, out, (int)(argc > 1));
  printf("out=%d\n", out[5]);
  return 0;
}
"""


def _libtsan():
    try:
        path = subprocess.run(["gcc", "-print-file-name=libtsan.so"], capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        return None
    return path if os.path.isabs(path) and os.path.exists(path) else None


def test_detector_sees_a_missing_syncthreads(tmp_path):
    if _libtsan() is None:
        pytest.skip("gcc's libtsan.so not found")
    src = tmp_path / "probe.cu"
    src.write_text(PROBE)
    core = tmp_path / "core.o"
    exe = tmp_path / "probe"
    common = ["g++", "-O1", "-g", "-std=c++17", "-w", "-DD3H_CPU_EMU=1", "-DEMU_TSAN=1", "-I", EMU]
    subprocess.run(common + ["-fPIC", "-c", os.path.join(EMU, "emu_core.cpp"), "-o", str(core)], check=True)
    subprocess.run(common + ["-fsanitize=thread", "-x", "c++", str(src), "-x", "none", str(core), "-o", str(exe)], check=True)
    racy = subprocess.run([str(exe)], capture_output=True, text=True)
    clean = subprocess.run([str(exe), "barrier"], capture_output=True, text=True)
    assert "ThreadSanitizer: data race" in racy.stderr and "in probe(int*, int)" in racy.stderr, racy.stderr[-2000:]
    assert "ThreadSanitizer" not in clean.stderr and "out=42" in clean.stdout, clean.stderr[-2000:]


def test_emulated_kernels_have_no_intra_block_races():
    tsan = _libtsan()
    if tsan is None:
        pytest.skip("gcc's libtsan.so not found")
    # one OpenMP thread: libgomp is not instrumented, its barriers are invisible to TSan and torch's own parallel loops
    # would be reported; reports are filtered to the product's sources anyway (exitcode=0: the filter decides)
    env = dict(os.environ, LD_PRELOAD=tsan, D3H_EMU_VARIANT="tsan", OMP_NUM_THREADS="1",
               TSAN_OPTIONS="halt_on_error=0:report_signal_unsafe=0:exitcode=0")
    tests = FULL if os.environ.get("D3H_RACECHECK_FULL") == "1" else SELECTION
    res = subprocess.run([sys.executable, os.path.join(EMU, "san_runner.py")] + tests + ["-s"], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=2400)
    out = res.stdout + res.stderr
    reports = [l for l in out.splitlines() if l.startswith("SUMMARY: ThreadSanitizer") and "/csrc/" in l]
    assert not reports, "\n".join(sorted(set(reports))[:20])
    assert res.returncode == 0 and " passed" in out, out[-3000:]
