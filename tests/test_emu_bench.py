"""Control-flow dry run of bench.py on CPU: two gloo ranks, CPU tensors, the emulated kernels (tests/emu), tiny grid.
Round 1 lost 120 GPU-minutes to a collective that only rank 0 entered; this test runs the same script, same argument
parsing, same step / timing / diagnostics / end-to-end legs on two ranks and fails fast if a rank is left waiting.  The
numbers it prints mean nothing."""
import contextlib
import io
import json
import os
import socket
import sys
import time

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _Event:
    def __init__(self, enable_timing=False):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return (other.t - self.t) * 1e3


class _Stream:
    cuda_stream = 0

    def synchronize(self):
        pass

    def wait_stream(self, other):
        pass

    def wait_event(self, ev):
        pass


def _worker(rank, world, port, out_dir, argv):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port), D3H_BENCH_DEVICE="cpu")
    sys.path.insert(0, ROOT)
    from tests.test_emu_multirank import _patch_for_cpu
    _patch_for_cpu()
    from d3human_code_b200.render import mesh as M
    M._check_cuda = lambda t: None
    torch.cuda.current_stream = lambda dev=None: _Stream()
    torch.cuda.Event = _Event
    torch.cuda.Stream = _Stream
    torch.cuda.stream = lambda s: contextlib.nullcontext()
    torch.cuda.synchronize = lambda dev=None: None
    import bench
    sys.argv = ["bench.py"] + argv
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.main()
    with open(os.path.join(out_dir, f"out_{rank}.txt"), "w") as fh:
        fh.write(buf.getvalue())


@pytest.mark.parametrize("world", [1, 2])
def test_bench_control_flow(tmp_path, world):
    import torch.multiprocessing as mp
    argv = ["--gpus", str(world), "--steps", "2", "--warmup", "1", "--res", "6", "--frames-per-rank", "16", "--groups", "2",
            "--lanes", "2", "--profile-steps", "1", "--e2e-chunk", "8", "--dump-outputs", str(tmp_path / "dump")]
    if world > 1:
        argv.append("--no-cpu-baseline")     # N = 1 runs the CPU baseline leg as well (tiny grid: a fraction of a second)
    ctx = mp.start_processes(_worker, args=(world, _free_port(), str(tmp_path), argv), nprocs=world, join=False,
                             start_method="spawn")
    deadline = time.time() + 240
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for p in ctx.processes:
                p.terminate()
            pytest.fail("bench.py did not finish: a rank is waiting in a collective the others never entered")
    line = [l for l in open(tmp_path / "out_0.txt") if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["n_gpus"] == world and d["steps"] == 2 and d["unit"] == "tets/s" and d["higher_is_better"] is True
    assert d["config"]["frames_per_step"] == 16 * world and d["config"]["groups"] == 2
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] > 0
    assert d["e2e"] is not None and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["device_trace"] is not None and "error" not in d["device_trace"]
    if world == 1:                               # the mesh-stage leg ran (on the emulated kernels) and agrees with torch
        ms = d["mesh_stage"]
        assert "error" not in ms, ms
        for name in ("open", "watertight"):
            assert ms[name]["edges_equal_torch"] is True and ms[name]["E"] > 0 and ms[name]["normals_fwd_us"] > 0
        assert ms["gpu_launches"] > 0
        assert d["single_call"]["fwd_ms_median"] > 0 and d["single_call"]["bwd_ms_median"] > 0
        cb = d["cpu_baseline"]
        assert cb["kind"] == "port" and cb["value"] > 0 and "error" not in cb["torch_port"] and cb["torch_port"]["value"] > 0
        tb = d["torch_gpu_baseline"]             # the plain-PyTorch port ran (on CPU here) and produced a number
        assert "error" not in tb and tb["value"] > 0 and tb["kind"] == "port", tb
    else:
        assert d["mesh_stage"] is None and d["torch_gpu_baseline"] is None
    for r in range(1, world):                    # only rank 0 prints
        assert not [l for l in open(tmp_path / f"out_{r}.txt") if l.startswith("{")]
    assert len(d["ms_per_step_blocks"]) == 2 and d["config"]["mode"] == "weak"       # --steps 2: two blocks of one step
    _check_dump(tmp_path / "dump", world)
    rk = d["ranks"]
    assert len(rk["local_step_ms"]) == world and rk["frames"] == [16] * world and all(t > 0 for t in rk["local_step_ms"])
    assert (world == 1) == (sum(rk["allreduce_ms"]) == 0)
    if world == 1:
        assert "error" not in d["cold"] and d["cold"]["ms_per_frame"] > 0, d["cold"]
        sp = d["split_pair"]
        assert "error" not in sp and sp["two_calls_ms"] > 0 and sp["split_ms"] > 0 and sp["split_fused_ms"] > 0, sp
        # the compact gradient return: far fewer bytes back than the dense (N,3) gradients it replaces
        assert d["e2e"]["d2h_bytes_per_step"] < d["e2e"]["h2d_bytes_per_step"] * 4


def _check_dump(out_dir, world):
    """--dump-outputs of test_bench_control_flow (res 6, 16 frames on rank 0, nothing sampled at this size): the surfaces
    of every frame are the oracle's; on one rank the gradients are the oracle's adjoint of bench.py's upstream gradients."""
    import numpy as np
    from oracle import gshell_oracle as O
    from d3human_code_b200 import grids
    from tests import _util as U
    sys.path.insert(0, ROOT)
    import bench
    got = {n: np.load(out_dir / f"{n}.npy") for n in bench.SURFACE_OUTPUTS + ("counts", "grad_pos", "grad_sdf", "grad_msdf")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    pos, sdf, msdf, tets = bench.make_inputs(6, "capsule")
    N = pos.shape[0]
    want = {n: [] for n in got}
    gen = torch.Generator(device="cpu").manual_seed(1234)
    fwds = [O.extract_forward(pos + grids.frame_offsets(N, 6, f), sdf, msdf, tets, 1, True) for f in range(16)]
    ups_v = [torch.randn(fw["verts_aug"].shape, generator=gen).numpy() for fw in fwds]
    ups_m = [torch.randn(fw["msdf"].shape, generator=gen).numpy() for fw in fwds]
    want["grad_sdf"], want["grad_msdf"] = np.zeros(N), np.zeros(N)
    for fw, gv, gm in zip(fwds, ups_v, ups_m):
        for n in bench.SURFACE_OUTPUTS:
            want[n].append(fw[n])
        want["counts"].append([len(fw["verts_aug"]), len(fw["faces_aug"]), len(fw["vertices_watertight"]),
                               len(fw["faces_watertight"])])
        g_pos, g_sdf, g_msdf = O.extract_backward(fw, gv, gm)
        want["grad_pos"].append(g_pos)
        want["grad_sdf"] += g_sdf
        want["grad_msdf"] += g_msdf
    for n in bench.SURFACE_OUTPUTS:
        w = np.concatenate(want[n])
        if n.startswith("v_tng"):          # sums of float atomics in any order, as everywhere against the oracle
            U.assert_tangents_close(n, got[n], w, U.TNG_CUDA_ATOL)
        else:
            assert got[n].shape == w.shape and np.array_equal(got[n], w), n
    assert np.array_equal(got["counts"], np.array(want["counts"]))
    assert got["grad_pos"].shape == (16 * N, 3) and got["grad_sdf"].shape == got["grad_msdf"].shape == (N,)
    if world == 1:
        for n in ("grad_pos", "grad_sdf", "grad_msdf"):
            w = np.concatenate(want[n]) if n == "grad_pos" else want[n]
            assert np.abs(got[n] - w).max() <= 1e-4 * np.abs(w).max(), n


def test_dump_outputs_keeps_a_fixed_sample_of_large_arrays(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    big = np.random.default_rng(0).standard_normal((5000, 3)).astype(np.float32)
    arrays = {"small": np.arange(12, dtype=np.int32).reshape(4, 3), "big": big}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit=64 << 10)
    small, kept = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "big.npy")
    assert small.dtype == np.float64 and np.array_equal(small, arrays["small"])
    assert kept.dtype == np.float32 and 1000 < kept.shape[0] and kept.nbytes <= (64 << 10) // 2
    assert np.array_equal(kept, np.load(tmp_path / "b" / "big.npy"))        # the same rows every run
    rows = [int(np.flatnonzero((big == r).all(1))[0]) for r in kept]
    assert rows == sorted(set(rows))                                          # rows of the array, in order


def _run(tmp_path, world, argv, timeout=240):
    import torch.multiprocessing as mp
    ctx = mp.start_processes(_worker, args=(world, _free_port(), str(tmp_path), argv), nprocs=world, join=False,
                             start_method="spawn")
    deadline = time.time() + timeout
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for p in ctx.processes:
                p.terminate()
            pytest.fail("bench.py did not finish: a rank is waiting in a collective the others never entered")
    lines = [l for l in open(tmp_path / "out_0.txt") if l.startswith("{")]
    for r in range(1, world):
        assert not [l for l in open(tmp_path / f"out_{r}.txt") if l.startswith("{")]
    return json.loads(lines[-1])


def test_bench_strong_mode_two_ranks(tmp_path):
    """--mode strong (BASELINE configs[3] as written): a fixed batch of frames sharded over the ranks."""
    d = _run(tmp_path, 2, ["--gpus", "2", "--steps", "2", "--warmup", "1", "--res", "6", "--mode", "strong", "--frames-total",
                           "5", "--groups", "2", "--lanes", "2", "--profile-steps", "1", "--no-cpu-baseline", "--blocks", "2"])
    assert d["scaling"] == "strong" and d["config"]["frames_per_step"] == 5 and d["ranks"]["frames"] == [3, 2]
    assert d["value"] > 0 and d["config"]["mode"] == "strong"


@pytest.mark.parametrize("world", [1, 2])
def test_bench_tets_mode(tmp_path, world):
    """--mode tets (BASELINE configs[4]): tet-range shards + all-gather of the records; every rank ends with the same mesh."""
    d = _run(tmp_path, world, ["--gpus", str(world), "--steps", "2", "--warmup", "1", "--res", "8", "--mode", "tets", "--blocks", "2"])
    assert d["scaling"] == "strong" and d["ranks_hold_same_mesh"] is True and d["comm_nranks_ok"] is True
    assert d["config"]["mode"] == "tets" and d["config"]["F"] == 6 * 8 ** 3 and d["value"] > 0 and d["gpu_launches"] > 0


def test_reference_arm_prints_the_same_config(tmp_path):
    """--impl reference: same metric / unit / config / steps / warm-up as the GPU arm (the driver compares them)."""
    argv = ["--gpus", "1", "--steps", "2", "--warmup", "1", "--res", "6", "--frames-per-rank", "16", "--groups", "2", "--lanes", "2",
            "--profile-steps", "1", "--no-cpu-baseline", "--no-e2e", "--no-mesh-stage", "--no-torch-baseline", "--no-cold",
            "--no-split-pair"]
    ours = _run(tmp_path, 1, argv)
    import subprocess
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"] + argv, capture_output=True,
                         text=True, timeout=200)
    ref = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert ref["impl"] == "reference" and ref["config"] == ours["config"], (ref["config"], ours["config"])
    for k in ("metric", "unit", "steps", "warmup", "higher_is_better", "scaling", "n_gpus"):
        assert ref[k] == ours[k], k
    assert ref["cpu_baseline"]["kind"] == "port" and ref["e2e"]["h2d_bytes_per_step"] == 0
