#!/usr/bin/env python
"""Headline benchmark: tets/s of fwd+bwd G-Shell / mSDF extraction (BASELINE.json metric) + HBM roofline fraction.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): 128^3 Kuhn tet grid (F=12,582,912, N=2,146,689), analytic capsule-union SDF +
garment mSDF, hmSDF_Tets(type="cloth") forward + backward with upstream gradients on verts_aug and extra['msdf'].
Each rank runs `--frames-per-rank` frames per step (default 32 = two configs[3] batches); a frame is one full extraction
with its own per-frame tet-vertex offsets (seed = global frame index); the frames of a step go through `--groups`
extract_frames_async() calls of 8 frames (one autograd node and one library call per direction each, frames spread over
concurrent lanes), all launched up front so that the host work of one group overlaps the GPU work of the next.
sdf/msdf are shared, so their gradients accumulate over the rank's frames (atomics) and are all-reduced (NCCL) when
N > 1.  Weak scaling: per-GPU work is fixed.  value = N * frames_per_rank * F / (max-over-ranks device time per step).
`single_call` reports the same frames through the drop-in class one call at a time (the reference's calling pattern).

One JSON line on stdout (rank 0).  See DESIGN.md, "Measurement: keys of the bench.py JSON line".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "tets/s fwd+bwd G-Shell extraction"
UNIT = "tets/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--res", type=int, default=128, help="Kuhn grid resolution (128 = BASELINE configs[1])")
    ap.add_argument("--frames-per-rank", type=int, default=32,
                    help="frames per rank per step (BASELINE configs[3]: batches of 16 video frames; default = 2 batches)")
    ap.add_argument("--lanes", type=int, default=8, help="concurrent lanes the frames of a batch are spread over")
    ap.add_argument("--groups", type=int, default=2,
                    help="the frames of a step are issued as this many extract_frames_async batches (host / GPU pipelining; "
                         "a batch runs its frames fused, 8 per launch: with 2 groups a 32-frame step is 4 rounds of launches "
                         "and 2 host round trips -- 1.32 ms against 1.57 ms with 4 groups, r02ag)")
    ap.add_argument("--field", default="capsule", choices=["capsule", "sphere"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-mesh-stage", action="store_true", help="skip the Mesh / auto_normals leg (SURVEY 8f row 2)")
    ap.add_argument("--no-torch-baseline", action="store_true", help="skip the plain-PyTorch-on-this-GPU leg (SURVEY 8d)")
    ap.add_argument("--profile-steps", type=int, default=20)
    ap.add_argument("--e2e-chunk", type=int, default=4, help="frames per pipelined chunk of the end-to-end leg")
    ap.add_argument("--e2e-pos", choices=["copy", "mapped", "both"], default="both",
                    help="end-to-end leg: per-frame positions copied to the device every step (copy), or read by the "
                         "kernels straight from the pinned, device-mapped host buffer (mapped: extract.mapped_view, only "
                         "the rows of crossing-edge end points cross PCIe); both = mapped as `e2e`, copy next to it")
    ap.add_argument("--e2e-chunk-mapped", type=int, default=8, help="frames per chunk of the mapped end-to-end leg")
    ap.add_argument("--mode", default="weak", choices=["weak", "strong", "tets"],
                    help="weak: --frames-per-rank frames on every rank (default); strong: BASELINE configs[3] as written, "
                         "--frames-total frames sharded over the ranks; tets: configs[4], one 256^3 extraction whose tet "
                         "ranges are sharded over the ranks + NCCL all-gather of the valid-tet records")
    ap.add_argument("--frames-total", type=int, default=16, help="--mode strong: frames per step over ALL ranks")
    ap.add_argument("--blocks", type=int, default=5,
                    help="the --steps timed steps are split into this many blocks run back to back; value = median block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0's frames: surfaces, counts, "
                         "gradients) as DIR/<name>.npy, float32 / float64, at most 64 MB in all")
    ap.add_argument("--api", default="packed", choices=["packed", "frames"],
                    help="batch results as padded (B,cap,..) tensors (O(1) host work per batch) or as per-frame tuples")
    ap.add_argument("--no-cold", action="store_true", help="skip the L2-flushed single-call leg")
    ap.add_argument("--no-split-pair", action="store_true", help="skip the configs[2] cloth/body pair leg")
    ap.add_argument("--no-sdf-query", action="store_true", help="skip the SDF-network leg (SURVEY 8f row 3)")
    ap.add_argument("--no-lbs-stage", action="store_true", help="skip the skinning leg (SURVEY 8f row 4)")
    return ap.parse_args()


def make_inputs(res, field):
    from d3human_code_b200 import grids
    pos, tets = grids.kuhn_grid(res)
    sdf, msdf = (grids.capsule_garment_field if field == "capsule" else grids.sphere_plane_field)(pos)
    return pos, sdf, msdf, tets


def workload_name(args):
    field = 'capsule-union SDF + garment mSDF' if args.field == 'capsule' else 'sphere SDF + plane mSDF'
    if args.mode == "strong":
        return (f"configs[3]: {args.res}^3 Kuhn grid, {field}, hmSDF_Tets(cloth) semantics fwd+bwd, a batch of "
                f"{args.frames_total} frames/step with per-frame offsets sharded over the ranks (strong scaling)")
    return (f"configs[1]: {args.res}^3 Kuhn grid, {field}"
            f", hmSDF_Tets(cloth) semantics fwd+bwd, {args.frames_per_rank} frame(s)/rank/step with per-frame offsets "
            f"(configs[3] batch) through extract_frames ({args.lanes} workspaces: the frames of a batch run fused, up to 8 per "
            f"launch, and share one topology since they share sdf / msdf)")


def frames_of_rank(args, world, rank):
    """Global frame indices this rank extracts every step."""
    if args.mode == "strong":
        from d3human_code_b200 import sharding
        return list(sharding.frame_slice(args.frames_total, world, rank))
    return [rank * args.frames_per_rank + i for i in range(args.frames_per_rank)]


def make_config(args, world, F, N, counts0, ngroups, frames_per_step):
    """The `config` object of the JSON line: identical for the GPU arm and the --impl reference arm."""
    return {"workload": workload_name(args), "F": int(F), "N": int(N), "frames_per_step": int(frames_per_step),
            "counts_frame0": counts0,
            "l2": "per step every frame writes 26 MB of position gradients (zero-filled, then scattered into) next to its "
                  "surface buffers (%d MB per rank and step > 126 MB L2); the static run-length tables (14 MB at 128^3) are "
                  "re-read by every batch as in training, where the tet grid is static; no explicit flush in the headline, "
                  "`cold` = L2-flushed single call"
                  % (34 * max(1, frames_per_step // max(world, 1))),
            "lanes": args.lanes, "groups": ngroups, "mode": args.mode,
            "parallelism": (("frames x%d" % world) if args.mode != "tets" else ("tet ranges x%d" % world)) if world > 1 else "single GPU"}


def block_sizes(steps, blocks):
    """Exactly `steps` timed steps, split into up to `blocks` blocks that run back to back."""
    n = max(1, min(blocks, steps))
    return [(b + 1) * steps // n - b * steps // n for b in range(n)]


def group_bounds(n, groups):
    # at least 8 frames per group: a group is one library call on up to 8 lanes, smaller ones cannot fill them and the
    # host cost per group (launch, size read, backward) stops being hidden
    g = max(1, min(groups, n // 8))
    return [(n * k // g, n * (k + 1) // g) for k in range(g)]


# ------------------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while a region runs."""

    def __init__(self, index, period=0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.stop_flag, self.max_mhz = [], set(), False, None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:  # pragma: no cover
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # pragma: no cover
                pass
            time.sleep(self.period)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------- --dump-outputs
DUMP_LIMIT = 64 << 20
#: the gradients on the grid are almost all zero; they are kept on the grid vertices nearest the surface (smallest
#: |sdf|), where the rows the extraction touches lie
DUMP_GRID_ROWS = 1 << 16
SURFACE_OUTPUTS = ("verts_aug", "faces_aug", "v_tng_aug", "msdf", "vertices_watertight", "faces_watertight",
                   "v_tng_watertight", "msdf_watertight")


def step_outputs(groups, flat_grad, rows):
    """What a caller of the timed step holds afterwards, as numpy.  `groups`: (results, gradient of the positions) of
    every extract_frames_async call of the step, results packed or per frame.  Per frame, concatenated over the frames
    in order: the reference's outputs and `counts` (rows of verts_aug, faces_aug, vertices_watertight and
    faces_watertight).  The gradients of pos (frame-major), sdf and msdf on the grid vertices `rows`."""
    per, counts, g_pos = {k: [] for k in SURFACE_OUTPUTS}, [], []
    for res, g in groups:
        frames = [res.frame(i) for i in range(len(res))] if hasattr(res, "frame") else res
        for verts, faces, _, _, v_tng, extra in frames:
            vals = (verts, faces, v_tng, extra["msdf"], extra["vertices_watertight"], extra["faces_watertight"],
                    extra["v_tng_watertight"], extra["msdf_watertight"])
            for k, t in zip(SURFACE_OUTPUTS, vals):
                per[k].append(t.detach().cpu().numpy())
            counts.append([vals[i].shape[0] for i in (0, 1, 4, 5)])
        g_pos.append(g[:, rows].reshape(-1, 3).cpu().numpy())
    n = flat_grad.shape[0] // 2
    out = {k: np.concatenate(v) for k, v in per.items()}
    out.update(counts=np.array(counts), grad_pos=np.concatenate(g_pos), grad_sdf=flat_grad[:n][rows].cpu().numpy(),
               grad_msdf=flat_grad[n:][rows].cpu().numpy())
    return out


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """Writes every array as out_dir/<name>.npy: float32 stays float32, anything else becomes float64 (exact for the
    integer outputs).  An array larger than an equal share of `limit` keeps a sample of its rows, drawn with a seed of
    its own and sorted, so that two runs with the same row count keep the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    share = (limit - 4096 * len(arrays)) // len(arrays)      # 4096: room for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64, copy=False)
        if a.nbytes > share:
            keep = np.random.default_rng(zlib.crc32(name.encode())).choice(a.shape[0], share // (a.nbytes // a.shape[0]),
                                                                            replace=False)
            a = a[np.sort(keep)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """The reference's CPU implementation of the path, timed on this box's host cores: the numpy port in oracle/
    (the reference itself is PyTorch code that does not travel to the GPU box).  Same config / metric / unit / steps /
    warm-up as the GPU arm; a step is a BOUNDED SAMPLE of the workload: one frame (fwd+bwd) of the step's frames."""
    if rank != 0:
        return
    from oracle import gshell_oracle as O
    cores = os.cpu_count() or 1
    if args.mode == "tets":
        res = args.res if args.res != 128 else 256
        args.res, args.field = res, "sphere"
    pos, sdf, msdf, tets = make_inputs(args.res, args.field)
    F, N = tets.shape[0], pos.shape[0]
    from d3human_code_b200 import grids
    if args.mode != "tets":
        pos = pos + grids.frame_offsets(pos.shape[0], args.res, 0)
    state = {}

    def step():
        fwd = O.extract_forward(pos, sdf, msdf, tets, 1, True, n_threads=cores)
        gv = np.ones_like(fwd["verts_aug"])
        gm = np.ones_like(fwd["msdf"])
        O.extract_backward(fwd, gv, gm)
        state["fwd"] = fwd

    step()
    t0 = time.perf_counter(); step(); one = time.perf_counter() - t0
    fwd = state["fwd"]
    t1, t2 = int(fwd["t1"]), int(fwd["t2"])
    v, va = int(fwd["vertices_watertight"].shape[0]), int(fwd["verts_aug"].shape[0])
    counts0 = dict(n_valid_tets=int(fwd["fv"]), n_tri_tets=t1, n_quad_tets=t2, n_corners=3 * t1 + 4 * t2, n_verts=v,
                   n_verts_aug=va, n_faces_watertight=t1 + 2 * t2, n_faces_aug=int(fwd["faces_aug"].shape[0]),
                   bucket_polys=[int(c) // k for c, k in zip(fwd["bucket_counts"], (1, 2, 1, 2, 3, 4))])
    warm = max(args.warmup, 3)
    steps = args.steps
    note = ""
    if (steps + warm) * one > 240.0:      # keep the whole run within a few minutes on a slow host
        steps = max(1, int(240.0 / one) - warm)
        note = f" (--steps {args.steps} cut to {steps} to bound the run)"
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    value = F / dt
    if args.mode == "tets":
        fps, ngroups = 1, 1
    else:
        nf = len(frames_of_rank(args, world, 0))
        fps = args.frames_total if args.mode == "strong" else world * args.frames_per_rank
        ngroups = len(group_bounds(nf, args.groups))
    sample = (f"{steps} step(s), each ONE frame (a full fwd+bwd extraction) of the step's {fps} frames on the host CPU, "
              f"numpy port with the O(F) stage on {cores} threads{note}")
    config = make_config(args, world, F, N, counts0, ngroups, fps) if args.mode != "tets" else tets_config(args, world, F, N, counts0)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak" if args.mode == "weak" else "strong",
            "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference", "config": config,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def tets_config(args, world, F, N, counts0):
    return {"workload": f"configs[4]: {args.res}^3 Kuhn grid, sphere SDF + plane mSDF, ONE extraction fwd+bwd per step, "
                        f"tet ranges sharded over the ranks, NCCL all-gather of the compact valid-tet records, surface "
                        f"stages replicated (bit-identical to one GPU)",
            "F": int(F), "N": int(N), "frames_per_step": 1, "counts_frame0": counts0,
            "l2": "the tet stream of a rank is 16*F/ranks bytes (1.6 GB on one GPU) > 126 MB L2", "lanes": 1, "groups": 1,
            "mode": "tets", "parallelism": ("tet ranges x%d" % world) if world > 1 else "single GPU"}


# ------------------------------------------------------------------------------------------------- configs[4]
def run_tets(args, rank, local_rank, world, dev, dev_type):
    """--mode tets: BASELINE configs[4].  One 256^3 extraction (sphere + plane) per step whose only O(F) stage, the
    classification stream over the tet array, is split in `world` contiguous tet ranges (sharding.extract_tet_sharded):
    every rank classifies its range, the compact 32-byte valid-tet records are all-gathered (NCCL; rank order = global tet
    order) and the O(surface) stages run replicated, so every rank ends with the whole mesh, bit-identical to one GPU.
    value = F / (max-over-ranks device time of fwd+bwd).  Strong scaling."""
    import torch
    import torch.distributed as dist
    from d3human_code_b200 import extract as E, grids, sharding
    res = args.res if args.res != 128 else 256
    args.res = res
    pos_np, tets_np = grids.kuhn_grid(res)
    sdf_np, msdf_np = grids.sphere_plane_field(pos_np)
    F, N = int(tets_np.shape[0]), int(pos_np.shape[0])
    tets = torch.from_numpy(tets_np).to(dev)
    del tets_np
    pos = torch.from_numpy(pos_np).to(dev).requires_grad_(True)
    sdf = torch.from_numpy(sdf_np[:, None].copy()).to(dev).requires_grad_(True)
    msdf = torch.from_numpy(msdf_np).to(dev).requires_grad_(True)
    E.set_static_edges("0")      # the sharded path exchanges records and sorts their edges; no static table at 256^3

    def fwd():
        return sharding.extract_tet_sharded(pos, sdf, msdf, tets, msdf_negate=False, group=None,
                                            virtual_ranks=1 if world == 1 else None)

    verts, faces, _, _, _, extra = fwd()
    c0 = dict(E.last_counts())
    c0["bucket_polys"] = list(c0["bucket_polys"])
    g = torch.Generator(device=dev).manual_seed(1234)
    gv = torch.randn(verts.shape, device=dev, generator=g)
    gm = torch.randn(extra["msdf"].shape, device=dev, generator=g)
    checksum = int(faces.sum().item()) ^ int(verts.shape[0])

    def step():
        pos.grad = sdf.grad = msdf.grad = None
        v, f, _, _, _, ex = fwd()
        torch.autograd.backward([v, ex["msdf"]], [gv, gm])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = E.launch_counter()
    blocks = [timed(n) for n in block_sizes(args.steps, args.blocks)]
    launches = E.launch_counter() - l0
    sampler.stop_flag = True
    sampler.join(timeout=2)
    ms = float(np.median(blocks))
    # every rank must hold the same mesh
    cs = torch.tensor([checksum], dtype=torch.int64, device=dev)
    same = True
    if world > 1:
        allc = [torch.zeros_like(cs) for _ in range(world)]
        dist.all_gather(allc, cs)
        same = all(int(c.item()) == checksum for c in allc)
    if rank == 0:
        peak, peak_src = FALLBACK_HBM_GBS, "fallback"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                peak, peak_src = float(json.load(fh)["hbm_gbs"]), "measured"
        except Exception:
            pass
        balg = grids.surface_counts_bytes(F, N, c0["n_verts"], c0["n_verts_aug"], c0["n_faces_watertight"], c0["n_faces_aug"])
        line = {"metric": METRIC, "value": F / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": tets_config(args, world, F, N, c0),
                "ms_per_step_blocks": [round(b, 5) for b in blocks],
                "path_roofline": {"algorithmic_bytes_per_frame": int(balg), "achieved_GBps_step": balg / (ms * 1e-3) / 1e9,
                                  "frac_step": balg / (ms * 1e-3) / 1e9 / peak, "peak": peak, "peak_source": peak_src},
                "ranks_hold_same_mesh": bool(same), "comm_nranks_ok": bool(world == 1 or dist.get_world_size() == world),
                "gpu_launches": int(launches), "clocks": sampler.result()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------- our arm
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl == "reference" or args.mode == "tets"):
        raise SystemExit("--dump-outputs: only the batched extraction (--impl ours, --mode weak / strong) keeps its outputs")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    # D3H_BENCH_DEVICE=cpu is a TEST hook (tests/test_emu_bench.py): a control-flow dry run of this script on CPU tensors,
    # gloo and the emulated kernels of tests/emu -- it exists to catch collective mismatches between ranks without a GPU;
    # the product has no CPU path and the numbers of such a run mean nothing.
    dev_type = os.environ.get("D3H_BENCH_DEVICE", "cuda")
    if dev_type == "cuda":
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU path)")
        torch.cuda.set_device(local_rank)
    dev = torch.device(dev_type, local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a mismatched collective should fail within minutes, not hold the box for the default 10
        if dev_type == "cuda":
            dist.init_process_group(backend="nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))
        else:
            dist.init_process_group(backend="gloo", timeout=datetime.timedelta(seconds=120))
    from d3human_code_b200 import _cabi, grids
    from d3human_code_b200 import extract as E
    from d3human_code_b200.geometry.hmsdf_tets_split import hmSDF_Tets

    if args.mode == "tets":
        run_tets(args, rank, local_rank, world, dev, dev_type)
        return
    pos_np, sdf_np, msdf_np, tets_np = make_inputs(args.res, args.field)
    F, N = int(tets_np.shape[0]), int(pos_np.shape[0])
    frames = frames_of_rank(args, world, rank)
    fpr = len(frames)
    fps = args.frames_total if args.mode == "strong" else world * fpr      # frames per step over all ranks
    if fpr == 0:
        raise SystemExit("--mode strong needs --frames-total >= number of ranks")
    hm = hmSDF_Tets()
    tets = torch.from_numpy(tets_np).to(dev)                      # int64 like hmsdf.py:207-212; packed once (static)
    # sdf (N,1) like the SDF MLP output, msdf (N,).  Their gradients accumulate over the rank's frames and are summed over
    # the ranks: both .grad tensors are views of ONE flat buffer, so the exchange is one all-reduce of 8N bytes
    sdf = torch.from_numpy(sdf_np[:, None].copy()).to(dev).requires_grad_(True)
    msdf = torch.from_numpy(msdf_np).to(dev).requires_grad_(True)
    flat_grad = torch.zeros(2 * N, dtype=torch.float32, device=dev)
    # per-frame deformed grid vertices as ONE (B,N,3) tensor: one autograd leaf, one gradient buffer for the batch
    host_pos = torch.from_numpy(np.stack([pos_np + grids.frame_offsets(N, args.res, f) for f in frames])).pin_memory()
    host_sdf = torch.from_numpy(sdf_np[:, None].copy()).pin_memory()
    host_msdf = torch.from_numpy(msdf_np).pin_memory()
    pos = host_pos.to(dev).requires_grad_(True)
    # the frames of a step go through `--groups` extract_frames_async calls that are all launched up front: while the GPU
    # extracts group k+1 the host reads the sizes of group k, wraps its outputs and runs its backward pass
    gb = group_bounds(fpr, args.groups)
    ngroups = len(gb)
    pos_groups = [pos.detach()[lo:hi].clone().requires_grad_(True) for lo, hi in gb]   # one (b,N,3) leaf per group

    # dry run: shapes of the upstream gradients (constant across steps: inputs are fixed)
    outs = E.extract_frames(pos, sdf, msdf, tets, types="cloth", lanes=args.lanes)
    counts = [dict(c) for c in E.last_counts_frames()]
    g = torch.Generator(device=dev).manual_seed(1234)
    ups_v = [torch.randn(o[0].shape, device=dev, generator=g) for o in outs]
    ups_m = [torch.randn(o[5]["msdf"].shape, device=dev, generator=g) for o in outs]
    c0 = counts[0]
    c0["bucket_polys"] = list(c0["bucket_polys"])
    balg = sum(grids.surface_counts_bytes(F, N, c["n_verts"], c["n_verts_aug"], c["n_faces_watertight"], c["n_faces_aug"])
               for c in counts) / len(counts)
    del outs
    # padded upstream gradients for the packed API: rows beyond a frame's Va are never read, so one generous buffer per
    # group serves whatever capacity the plan settles on
    va_max = max(c["n_verts_aug"] for c in counts)
    pad_rows = 2 * va_max + 4096
    pups_v = [torch.zeros((hi - lo, pad_rows, 3), device=dev) for lo, hi in gb]
    pups_m = [torch.zeros((hi - lo, pad_rows), device=dev) for lo, hi in gb]
    for k, (lo, hi) in enumerate(gb):
        for i in range(lo, hi):
            pups_v[k][i - lo, :ups_v[i].shape[0]] = ups_v[i]
            pups_m[k][i - lo, :ups_m[i].shape[0]] = ups_m[i]
    last_step = []      # --dump-outputs: (results, gradient of the positions) of every group of the latest step

    def local_step():
        """This rank's share of a step, no collective: every group of frames is one extract_frames_async call (one
        library call, concurrent lanes) and one backward call; gradients of the shared sdf / msdf are summed over the
        frames by the kernels and over the groups by autograd (in place, into the flat buffer)."""
        flat_grad.zero_()
        sdf.grad, msdf.grad = flat_grad[:N].view(N, 1), flat_grad[N:]
        for pg in pos_groups:
            pg.grad = None
        last_step.clear()
        futs = [E.extract_frames_async(pg, sdf, msdf, tets, types="cloth", lanes=args.lanes) for pg in pos_groups]
        for k, (fut, (lo, hi)) in enumerate(zip(futs, gb)):
            if args.api == "packed":
                res = pk = fut.packed()
                cva = pk.verts_aug.shape[1]
                if cva > pad_rows:
                    raise RuntimeError("bench: padded upstream gradients too small for the plan's capacity")
                torch.autograd.backward([pk.verts_aug, pk.msdf], [pups_v[k][:, :cva], pups_m[k][:, :cva]])
            else:
                res = outs = fut.result()
                torch.autograd.backward([o[0] for o in outs] + [o[5]["msdf"] for o in outs], ups_v[lo:hi] + ups_m[lo:hi])
            if args.dump_outputs:
                last_step.append((res, pos_groups[k].grad))

    def step():
        """One training-step's worth of extraction: local_step() + the sum of the shared gradients over the ranks (ONE
        NCCL all-reduce of the flat sdf|msdf gradient buffer).  Every rank must call it the same number of times."""
        local_step()
        if world > 1:
            dist.all_reduce(flat_grad)

    pos_single = [pos.detach()[i].clone().requires_grad_(True) for i in range(min(fpr, 4))]   # separate (N,3) leaves

    def single_call_step():
        """The reference's own calling pattern: one drop-in call + backward per frame (hmsdf.py:548)."""
        sdf.grad = msdf.grad = None
        for p, gv, gm in zip(pos_single, ups_v, ups_m):
            p.grad = None
            verts, faces, _, _, v_tng, extra = hm(p, sdf, msdf, tets, "cloth")
            torch.autograd.backward([verts, extra["msdf"]], [gv, gm])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        tmax = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        return float(tmax.item()) / steps

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    # exactly --steps timed steps in up to --blocks blocks run back to back (each between two barriers, CUDA events, max
    # over ranks); the reported time is the MEDIAN block (one block is tens of ms: a single one is at the mercy of a clock
    # ramp or a host hiccup)
    launches0 = E.launch_counter()
    block_ms = [timed(step, n) for n in block_sizes(args.steps, args.blocks)]
    launches_timed = E.launch_counter() - launches0      # library kernels enqueued by this rank in the timed steps
    ms_step = float(np.median(block_ms))
    value = fps * F / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        rows = torch.from_numpy(np.sort(np.argsort(np.abs(sdf_np), kind="stable")[:DUMP_GRID_ROWS])).to(dev)
        dump_outputs(args.dump_outputs, step_outputs(last_step, flat_grad, rows))
    last_step.clear()

    # ---- where a step's time goes on every rank: the local part (no collective) and the exchange alone ----
    ranks_info = None
    k_br = max(3, min(args.steps, 30))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    e0.record()
    for _ in range(k_br):
        local_step()
    e1.record()
    t_host = (time.perf_counter() - t_host0) / k_br * 1e3      # host time to ISSUE a step (the GPU may lag behind)
    torch.cuda.synchronize()
    loc_ms = e0.elapsed_time(e1) / k_br
    ar_ms = 0.0
    if world > 1:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k_br):
            dist.all_reduce(flat_grad)
        e1.record()
        torch.cuda.synchronize()
        ar_ms = e0.elapsed_time(e1) / k_br
    mine = torch.tensor([loc_ms, ar_ms, t_host, float(fpr)], device=dev)
    allr = [torch.zeros_like(mine) for _ in range(world)]
    if world > 1:
        dist.all_gather(allr, mine)
    else:
        allr = [mine]
    ranks_info = {"local_step_ms": [round(float(t[0]), 4) for t in allr], "allreduce_ms": [round(float(t[1]), 4) for t in allr],
                  "host_issue_ms": [round(float(t[2]), 4) for t in allr], "frames": [int(t[3]) for t in allr],
                  "allreduce_bytes": int(flat_grad.numel() * 4), "steps": k_br,
                  "note": "per rank: device time of a step without the collective, of the collective alone (one all-reduce "
                          "of the flat sdf|msdf gradient), and the host time to issue a step"}

    # ---- the same frames through the drop-in class, one call + backward per frame (no batching, no lanes) ----
    single = None
    if world == 1:
        k_single = max(3, min(args.steps, 50))
        for _ in range(3):
            single_call_step()
        ms_single = timed(single_call_step, k_single) / len(pos_single)
        single = {"ms_per_frame": ms_single, "value": F / (ms_single * 1e-3), "unit": UNIT, "steps": k_single,
                  "note": "hmSDF_Tets()(...) + backward per frame, strictly serial on the host (the reference's calling pattern)"}
        # forward and backward separately (SURVEY 8d): CUDA events around each half of one drop-in call, median
        try:
            f_ms, b_ms = [], []
            p1, gv1, gm1 = pos_single[0], ups_v[0], ups_m[0]
            for _ in range(min(max(k_single, 10), 100)):
                sdf.grad = msdf.grad = p1.grad = None
                ea, eb_, ec = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                ea.record()
                verts, faces, _, _, v_tng, extra = hm(p1, sdf, msdf, tets, "cloth")
                eb_.record()
                torch.autograd.backward([verts, extra["msdf"]], [gv1, gm1])
                ec.record()
                barrier()
                f_ms.append(ea.elapsed_time(eb_))
                b_ms.append(eb_.elapsed_time(ec))
            single["fwd_ms_median"], single["bwd_ms_median"] = float(np.median(f_ms)), float(np.median(b_ms))
        except Exception as exc:  # noqa: BLE001
            single["fwd_bwd_split_error"] = f"{type(exc).__name__}: {exc}"[:200]

    # ---- the dominant kernel timed alone: back-to-back launches of edge_scan_kernel on the state the last single call left
    # in its workspace, CUDA events around the whole run on the launching stream (d3h_profile_scan_kernel) ----
    scan_alone_us = scan_warm_us = None
    if rank == 0 and dev_type == "cuda":
        try:
            from d3human_code_b200 import single as S1
            with torch.no_grad():
                hm(pos_single[0].detach(), sdf.detach(), msdf.detach(), tets, "cloth")
            flush_buf = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)
            scan_alone_us = S1.profile_scan_kernel(tets, N, reps=50, flush=flush_buf)
            scan_warm_us = S1.profile_scan_kernel(tets, N, reps=50, flush=None)
            del flush_buf
            E._ExtractFn.total_launches += 102 if scan_alone_us else 0
        except Exception as exc:  # noqa: BLE001
            scan_alone_us = None
            sys.stderr.write(f"profile_scan_kernel: {type(exc).__name__}: {exc}\n")

    # ---- cold figure (SURVEY 8d): the same single call with L2 flushed before every call (a 256 MB fill) ----
    cold = None
    if world == 1 and not args.no_cold:
        try:
            flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
            f_ms, b_ms = [], []
            p1, gv1, gm1 = pos_single[0], ups_v[0], ups_m[0]
            for rep in range(min(max(args.steps, 10), 50)):
                sdf.grad = msdf.grad = p1.grad = None
                flush.fill_(rep & 255)
                ea, eb_, ec = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                ea.record()
                verts, faces, _, _, v_tng, extra = hm(p1, sdf, msdf, tets, "cloth")
                eb_.record()
                torch.autograd.backward([verts, extra["msdf"]], [gv1, gm1])
                ec.record()
                barrier()
                f_ms.append(ea.elapsed_time(eb_))
                b_ms.append(eb_.elapsed_time(ec))
            tot = float(np.median(f_ms)) + float(np.median(b_ms))
            cold = {"fwd_ms_median": float(np.median(f_ms)), "bwd_ms_median": float(np.median(b_ms)), "ms_per_frame": tot,
                    "value": F / (tot * 1e-3), "unit": UNIT,
                    "note": "single drop-in call + backward with L2 flushed (256 MB device fill) before every call"}
            del flush
        except Exception as exc:  # noqa: BLE001
            cold = {"error": f"{type(exc).__name__}: {exc}"[:200]}

    # ---- per-kernel device time (CUDA events on the launching stream, recorded by the library; one frame at a time so
    # that every kernel is timed alone) ----
    prof = {}
    if rank == 0:
        _cabi.profile_enable(True)
        nprof = max(1, min(args.profile_steps, 128 // len(pos_single)))
        for _ in range(nprof):
            single_call_step()
        torch.cuda.synchronize()
        prof = _cabi.profile_read()
        _cabi.profile_enable(False)
    # ---- device-side stamps (globaltimer written by the kernels themselves) of one batched step inside the cached
    # graphs: duration of every kernel as it runs in the timed region, overlapped with the other lanes ----
    dev_trace = None
    if rank == 0:
        try:
            _cabi.trace_enable(True)
            plan = E._plan_for(pos.device, F, N)
            seq0 = plan.seq
            local_step()          # rank 0 only: must not contain a collective
            torch.cuda.synchronize()
            tr = _cabi.trace_read()
            _cabi.trace_enable(False)
            durs = {}
            t_lo, t_hi = None, None
            for i in range(fpr):
                for name, (a, b) in tr.get((seq0 + 1 + i) % 64, {}).items():
                    durs.setdefault(name, []).append((b - a) / 1e3)
                    t_lo = a if t_lo is None else min(t_lo, a)
                    t_hi = b if t_hi is None else max(t_hi, b)
            if durs:
                dev_trace = {"us_mean": {k: round(float(np.mean(v)), 2) for k, v in durs.items()},
                             "forward_span_us": round((t_hi - t_lo) / 1e3, 1), "frames": fpr}
        except Exception as exc:  # pragma: no cover
            dev_trace = {"error": str(exc)}
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- end to end through the public API with HOST buffers ----
    e2e = None
    def e2e_leg(mapped):
        # The batch is cut into chunks of `--e2e-chunk` frames that flow through three streams: H2D copies of chunk
        # k+1 and D2H copies of chunk k-1 run under the extraction of chunk k (PCIe is full duplex, ~55 GB/s each way).
        # Results copied back per frame: verts_aug, faces_aug, msdf, and the pos gradient in COMPACT form -- the ids of
        # the grid vertices the frame touched (its crossing edges, FramesFuture.tape_edges) and their gradient rows
        # (extract.gather_touched): the dense (N,3) gradient is > 99 % zeros.  The sdf | msdf gradients of the step (one
        # flat buffer) follow the last chunk.
        chunk = max(1, min(args.e2e_chunk_mapped if mapped else args.e2e_chunk, fpr))
        bounds = [(i, min(i + chunk, fpr)) for i in range(0, fpr, chunk)]
        d_sdf = torch.empty_like(sdf)
        d_msdf = torch.empty_like(msdf)
        d_flat = torch.zeros_like(flat_grad)
        diag = os.environ.get("D3H_E2E_DIAG", "")   # diagnostics only: "resident" = positions already on the device,
        no_d2h = "nod2h" in diag                     # "nod2h" = results stay on the device
        if "resident" in diag:
            mapped = True
            d_pos = [host_pos[lo:hi].to(dev) for lo, hi in bounds]
        elif mapped:
            # CUDA tensors that ALIAS the pinned host buffer (unified addressing: pinned allocations are device-mapped at
            # the same address): the kernels fetch the rows they need over PCIe, nothing is copied up front
            d_pos = [E.mapped_view(host_pos[lo:hi], dev) for lo, hi in bounds]
        else:
            d_pos = [torch.empty_like(pos[lo:hi]) for lo, hi in bounds]
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        outs_host = None
        k_e2e = max(3, min(args.steps, 20))

        def e2e_step():
            nonlocal outs_host
            h2d = d2h = 0
            cur = torch.cuda.current_stream()
            s_in.wait_stream(cur)
            ev_in = []
            with torch.cuda.stream(s_in):
                for dst, src in ((d_sdf, host_sdf), (d_msdf, host_msdf)):
                    dst.requires_grad_(False)
                    dst.copy_(src, non_blocking=True)
                    dst.requires_grad_(True)
                h2d += host_sdf.numel() * 4 + host_msdf.numel() * 4
                for dp, (lo, hi) in zip(d_pos, bounds):
                    dp.requires_grad_(False)
                    if not mapped:
                        dp.copy_(host_pos[lo:hi], non_blocking=True)
                        h2d += dp.numel() * 4
                    dp.requires_grad_(True)
                    dp.grad = None
                    ev = torch.cuda.Event()
                    ev.record(s_in)
                    ev_in.append(ev)
            d_flat.zero_()
            d_sdf.grad, d_msdf.grad = d_flat[:N].view(N, 1), d_flat[N:]
            keep, res_all = [], []
            futs = None
            if mapped:
                # nothing to wait for but sdf / msdf: every chunk is launched up front (as in the device-resident step), the
                # host reads the sizes of chunk k while the GPU extracts chunk k + 1
                cur.wait_stream(s_in)
                futs = [E.extract_frames_async(dp, d_sdf, d_msdf, tets, types="cloth", lanes=args.lanes) for dp in d_pos]
            for k, (dp, (lo, hi)) in enumerate(zip(d_pos, bounds)):
                if futs is None:
                    cur.wait_event(ev_in[k])
                    fut = E.extract_frames_async(dp, d_sdf, d_msdf, tets, types="cloth", lanes=args.lanes)
                else:
                    fut = futs[k]
                outs = fut.result()
                torch.autograd.backward([o[0] for o in outs] + [o[5]["msdf"] for o in outs],
                                        ups_v[lo:hi] + ups_m[lo:hi])
                res = []
                for i, o in enumerate(outs):
                    edges = fut.tape_edges(i)
                    res += [o[0].detach(), o[1], o[5]["msdf"].detach(), edges, E.gather_touched(dp.grad[i], edges)]
                    if mapped:      # rows of `pos` the kernels read in place: both end points of every crossing edge,
                        h2d += 2 * edges.numel() * 12   # once by the vertex interpolation and once by its adjoint
                if k == len(bounds) - 1:
                    res.append(d_flat)
                ev_out = torch.cuda.Event()      # (an event, not the stream: later chunks are already queued behind this one)
                ev_out.record(cur)
                s_out.wait_event(ev_out)
                res_all.append(res)
                if outs_host is not None and not no_d2h:
                    with torch.cuda.stream(s_out):
                        for h, t in zip(outs_host[k], res):
                            h.copy_(t, non_blocking=True)
                            d2h += t.numel() * t.element_size()
                keep.append((outs, fut))
            if outs_host is None:   # first call: allocate the pinned result buffers, copy without overlap
                outs_host = [[torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in res] for res in res_all]
                for hs, res in zip(outs_host, res_all):
                    for h, t in zip(hs, res):
                        h.copy_(t, non_blocking=True)
                        d2h += t.numel() * t.element_size()
            torch.cuda.synchronize()
            return h2d, d2h

        for _ in range(3):
            h2d_b, d2h_b = e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            e2e_step()
        barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / k_e2e], device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        # the PCIe floor of this step: its H2D bytes alone, copied from the same pinned buffers with nothing else running
        barrier()
        t0 = time.perf_counter()
        floor_dst = [torch.empty_like(pos[lo:hi]) for lo, hi in bounds] if mapped else d_pos
        for _ in range(3):
            for dp, (lo, hi) in zip(floor_dst, bounds):
                dp.detach().copy_(host_pos[lo:hi], non_blocking=True)
        torch.cuda.synchronize()
        h2d_only = (time.perf_counter() - t0) / 3
        return {"value": fps * F / float(dt.item()), "unit": UNIT, "h2d_bytes_per_step": int(h2d_b),
               "d2h_bytes_per_step": int(d2h_b), "steps": k_e2e, "ms_per_step": float(dt.item()) * 1e3,
               "chunk_frames": chunk, "h2d_only_ms_per_step": h2d_only * 1e3, "pos": "mapped" if mapped else "copy",
               "h2d_GBps": (4 * host_pos.numel()) / h2d_only / 1e9,
               "positions": ("read in place from pinned host memory (extract.mapped_view): h2d_bytes_per_step counts the rows "
                             "the kernels fetch (end points of the crossing edges, forward and backward, 12 B each; PCIe "
                             "sector granularity not included) + sdf + msdf") if mapped else "copied to the device every step",
               "note": "extract_frames_async() with inputs copied from pinned host memory each step (pos per frame, sdf, "
                       "msdf); per frame verts_aug, faces_aug, msdf and the COMPACT pos gradient (touched vertex ids + "
                       "their rows), plus the flat sdf|msdf gradient, copied back to pinned host memory; static tet "
                       "indices stay resident; chunks of frames pipelined over H2D / compute / D2H streams.  "
                       "h2d_only_ms_per_step: the same per-frame positions copied alone = the PCIe floor of the step"}
    if not args.no_e2e:
        if args.e2e_pos == "copy" or dev_type != "cuda":      # (the CPU dry run of the tests has no mapped memory)
            e2e = e2e_leg(False)
        else:
            # headline: the positions stay in pinned host memory and the kernels read the rows they need (mapped_view);
            # the same leg with the positions copied to the device first is reported next to it
            e2e = e2e_leg(True)
            if args.e2e_pos == "both":
                e2e["positions_copied_first"] = e2e_leg(False)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ----
    # Since the run-length tables (round 2) no kernel of the path streams an O(F) or O(U) array any more: the kernels that
    # are left work on the surface (a few MB per frame) and are bound by dependent look-ups and instruction issue, not by
    # HBM.  The kernel reported is the one with the largest share of a frame's device time (single-frame pass, CUDA events
    # around each launch), against the bytes it has to move (formulas below and in DESIGN.md); `path_roofline` keeps the
    # SURVEY's B_alg for the whole call.
    peak, peak_src = FALLBACK_HBM_GBS, "fallback"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peak, peak_src = float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        pass
    roofline = None
    kern = {}
    if prof:
        kern = {k: {"ms_total": round(v[0], 4), "launches": v[1], "us_avg": round(1e3 * v[0] / v[1], 3)} for k, v in prof.items()}
        st = E.static_edges_for(E.packed_tets(tets, N), N) if "edge_scan" in prof else None
        V_, Va_, Fw_, Fa_ = c0["n_verts"], c0["n_verts_aug"], c0["n_faces_watertight"], c0["n_faces_aug"]
        Fv_ = c0["n_valid_tets"]
        alg = {"classify": 16.0 * F,
               # sdf read, sign bitmap written, scan state cleared (two tet bitmaps, edge bitmap)
               "prepare": 4.0 * N + N / 8.0 + F / 4.0 + (st[2] / 8.0 if st else 0.0),
               # vertex: edge id + end points (8) + sdf / msdf / pos of both ends (40) in, 44 + 32 + 20 out (SURVEY: 44 B per
               # vertex out); valid tet: queue entry (8) + tet (16) + edge ranks (32) in, record (32) + corners (16) out
               "edge_emit": V_ * (4 + 8 + 40 + 96.0) + Fv_ * (8 + 16 + 32 + 32 + 16.0),
               # record (32) + corner ids (16) + 3.5 vertex rows (16 B) in per valid tet, 24 B per watertight face out, normals
               "poly_faces": Fv_ * (32 + 16 + 56.0) + 24.0 * Fw_ + 32.0 * V_,
               # record + corners per valid tet in, 28 B per augmented vertex (verts_aug, v_tng_aug, msdf) + 24 B per face out
               "poly_cut": Fv_ * (32 + 16.0) + 48.0 * V_ + 28.0 * Va_ + 24.0 * Fa_,
               "zero": 20.0 * N}
        if st is not None:
            scan_bytes = 4.0 * st[2] + 4.0 * (N + 1) + N / 8.0            # CSR walk: 4 B per edge + offsets + sign bitmap
            if len(st) > 9 and st[8] is not None:                          # transposed rows
                scan_bytes = 4.0 * st[2] + 4.0 * ((N + 31) // 32 + 1) + N / 8.0
            if len(st) > 11 and st[10][0] is not None:
                # run-length tables (scan_runs_kernel): 12 B per edge entry (difference, mask, chunk), 20 B per tet entry
                # (three differences, mask, chunk), the sign bitmap once (the windows come from L1 / L2)
                scan_bytes = 12.0 * st[10][0].shape[0] + N / 8.0 + (20.0 * st[11][0].shape[0] if st[11][0] is not None else 0.0)
            alg["edge_scan"] = scan_bytes
        cand = {k: prof[k][0] / prof[k][1] for k in alg if k in prof and prof[k][1] and prof[k][0] > 0 and k != "zero"}
        if cand:
            dom = max(cand, key=cand.get)
            ms, n = prof[dom]
            dom_bytes = alg[dom]
            t_events = ms / n * 1e-3      # one launch at a time between two events: includes the ~3 us launch / event gap
            t = scan_alone_us * 1e-6 if (dom == "edge_scan" and scan_alone_us) else t_events
            achieved = dom_bytes / t / 1e9
            traffic = None
            try:
                with open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")) as fh:
                    tj = json.load(fh).get(dom, {})
                    if int(tj.get("F", 0)) == F:
                        traffic = tj.get("dram_bytes_per_launch")
            except Exception:
                pass
            names = {"edge_scan": "scan_runs_kernel" if (st and len(st) > 11 and st[10][0] is not None) else "edge_scan_kernel",
                     "edge_emit": "scan_emit_kernel"}
            roofline = {"kernel": names.get(dom, dom + "_kernel"), "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": int(dom_bytes), "us_per_launch": t * 1e6,
                        "timing": "CUDA events recorded around each launch on its stream, one frame at a time "
                                  "(includes the ~3 us launch / event gap of a lone launch)",
                        "note": "largest share of a frame's device time; latency- and issue-bound on O(surface) data, no "
                                "O(F) / O(U) stream is left on the path (DESIGN.md section 4)",
                        "share_of_frame_kernel_time": cand[dom] / sum(cand.values()),
                        "all_kernels": {k: {"us_per_launch": round(cand[k] * 1e3, 2), "algorithmic_bytes": int(alg[k]),
                                            "frac": alg[k] / (cand[k] * 1e-3) / 1e9 / peak} for k in cand}}
            if scan_alone_us and "edge_scan" in alg:
                roofline["scan_kernel_alone"] = {"us_per_launch_l2_flushed": scan_alone_us, "us_per_launch_warm": scan_warm_us,
                                                 "algorithmic_bytes": int(alg["edge_scan"]),
                                                 "frac": alg["edge_scan"] / (scan_alone_us * 1e-6) / 1e9 / peak,
                                                 "timing": "d3h_profile_scan_kernel: 50 launches, each between its own pair of "
                                                           "CUDA events, L2 evicted by reading 256 MB before every launch"}
    dev_ms_frame = sum(v[0] for v in prof.values()) / max(nprof * len(pos_single), 1) if prof else None
    # Bytes THIS design has to move per frame: the dense gradients (zero-filled, then scattered into: 20 N), the surface
    # outputs and tapes (44 Va + 28 V + 24 Fa + 24 Fw, as in the SURVEY's B_alg) and the frame's share of the topology inputs
    # (sdf 4 N, sign bitmap N/8, run-length tables) which a batch reads once when its frames share sdf / msdf.  The SURVEY's
    # B_alg (16 F + 40 N + ...) assumes the tet array and all of pos / sdf / msdf are streamed per frame; the path no longer
    # does that, so speed measured against B_alg can exceed the HBM roofline.
    surf_bytes = balg - 16.0 * F - 40.0 * N
    table_bytes = 0.0
    try:
        st_ = E.static_edges_for(E.packed_tets(tets, N), N)
        if st_ is not None and len(st_) > 11 and st_[10][0] is not None:
            table_bytes = 12.0 * st_[10][0].shape[0] + (20.0 * st_[11][0].shape[0] if st_[11][0] is not None else 0.0)
    except Exception:  # noqa: BLE001
        pass
    frames_per_topology = max(1, min(8, fpr // max(ngroups, 1)))     # frames of one fused launch share the topology
    design_bytes = 20.0 * N + surf_bytes + (4.0 * N + N / 8.0 + table_bytes) / frames_per_topology
    path_roofline = {"algorithmic_bytes_per_frame": int(balg),
                     "bytes_this_design_per_frame": int(design_bytes),
                     "achieved_GBps_step": design_bytes * fpr / (ms_step * 1e-3) / 1e9,
                     "frac_step": design_bytes * fpr / (ms_step * 1e-3) / 1e9 / peak,
                     "frac_step_survey_b_alg": balg * fpr / (ms_step * 1e-3) / 1e9 / peak,
                     "kernel_ms_per_frame": dev_ms_frame,
                     "frac_kernels_only": (design_bytes / (dev_ms_frame * 1e-3) / 1e9 / peak) if dev_ms_frame else None,
                     "frac_single_call": (design_bytes / (single["ms_per_frame"] * 1e-3) / 1e9 / peak) if single else None,
                     "note": "frac_step = bytes_this_design_per_frame x frames / step time / peak: 20N (dense gradients) + "
                             "44Va + 28V + 24Fa + 24Fw (surface outputs, tapes) + the frame's share of sdf, sign bitmap and "
                             "run-length tables (read once per fused launch of frames that share sdf / msdf).  "
                             "frac_step_survey_b_alg uses the SURVEY's B_alg = 16F + 40N + ... (tet array and all inputs "
                             "streamed per frame): the path no longer moves those bytes, so that figure is a speed against "
                             "the contract, not a bandwidth, and may exceed 1"}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import gshell_oracle as O
        cores = os.cpu_count() or 1
        p0 = host_pos[0].numpy()

        def cpu_step():
            fwd = O.extract_forward(p0, sdf_np, msdf_np, tets_np, 1, True, n_threads=cores)
            O.extract_backward(fwd, np.ones_like(fwd["verts_aug"]), np.ones_like(fwd["msdf"]))

        cpu_step()
        reps, best, t_all = 0, 1e9, time.perf_counter()
        while reps < 20 and time.perf_counter() - t_all < 15.0:
            t0 = time.perf_counter(); cpu_step(); best = min(best, time.perf_counter() - t0); reps += 1
        cpu_baseline = {"value": F / best, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"best of {reps} full fwd+bwd extractions of one frame of the same workload, numpy oracle "
                                  f"with the O(F) stage on {cores} threads",
                        "ms_per_frame": best * 1e3}
        try:  # the same path as plain PyTorch ops on the host cores: how the reference itself behaves on a CPU
            from oracle import gshell_torch as GT
            cp = torch.from_numpy(p0.copy()).requires_grad_(True)
            cs, cm = torch.from_numpy(sdf_np[:, None].copy()).requires_grad_(True), torch.from_numpy(msdf_np.copy()).requires_grad_(True)
            ct = torch.from_numpy(tets_np)
            tbest = 1e9
            for _ in range(2):
                cp.grad = cs.grad = cm.grad = None
                t0 = time.perf_counter()
                v, _f, _, _, _, ex = GT.extract(cp, cs, cm, ct, 1, True)
                torch.autograd.backward([v, ex["msdf"]], [torch.ones_like(v), torch.ones_like(ex["msdf"])])
                tbest = min(tbest, time.perf_counter() - t0)
            cpu_baseline["torch_port"] = {"value": F / tbest, "unit": UNIT, "ms_per_frame": tbest * 1e3,
                                          "threads": torch.get_num_threads(),
                                          "note": "oracle/gshell_torch.py on CPU tensors, best of 2: the reference's op "
                                                  "sequence on the host (the numpy figure above is the faster, conservative one)"}
        except Exception as exc:  # noqa: BLE001
            cpu_baseline["torch_port"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}

    # ---- the stage right behind the extraction (SURVEY 8f row 2): Mesh.edges + auto_normals fwd / bwd of this package on
    # frame 0's surfaces against the same PyTorch ops on the device.  Last leg, never fatal: the headline is complete.
    mesh_stage = None
    if world == 1 and not args.no_mesh_stage:
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("_mesh_bench", os.path.join(ROOT, "profiles", "mesh_bench.py"))
            mb = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mb)
            with torch.no_grad():
                verts, faces, _, _, _, extra = hm(pos_single[0].detach(), sdf.detach(), msdf.detach(), tets, "cloth")
            l0 = mb.mesh.launch_counter()
            mesh_stage = mb.measure([("open", verts.detach(), faces),
                                     ("watertight", extra["vertices_watertight"].detach(), extra["faces_watertight"])],
                                    max(3, min(args.steps, 100)), sync=None if dev_type == "cuda" else "cpu")
            mesh_stage["gpu_launches"] = mb.mesh.launch_counter() - l0
            mesh_stage["unit"] = "us per call (median, CUDA events; edges include the host's size read)"
        except Exception as exc:  # noqa: BLE001
            mesh_stage = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- BASELINE configs[2]: body + garment split extraction on a grid in the script/get_tet_smpl.py layout (unstructured,
    # scrambled vertex labels and tet order) at the f3c.json resolution: the cloth / body pair of one training iteration
    # (train.py:1040-1047) as two drop-in calls, as one split() batch, and as the fused pair.  Never fatal.
    split_pair = None
    if world == 1 and not args.no_split_pair:
        try:
            sg = grids.smplx_layout_grid(args.res)
            sv, sf = sg["v"], sg["f"]
            ssdf, smsdf = grids.capsule_garment_field(sv)
            qp = torch.from_numpy(sv).to(dev).requires_grad_(True)
            qs = torch.from_numpy(ssdf[:, None].copy()).to(dev).requires_grad_(True)
            qm = torch.from_numpy(smsdf).to(dev).requires_grad_(True)
            qt = torch.from_numpy(sf).to(dev)

            def pair_two():
                return hm(qp, qs, qm, qt, "cloth"), hm(qp, qs, qm, qt, "body")

            variants = {"two_calls": pair_two, "split": lambda: hm.split(qp, qs, qm, qt),
                        "split_fused": lambda: hm.split(qp, qs, qm, qt, fused=True)}
            split_pair = {"workload": f"configs[2]: SMPL-X-layout grid from the {args.res}^3 lattice, cloth + body pair fwd+bwd",
                          "F": int(sf.shape[0]), "N": int(sv.shape[0]), "unit": "ms per pair (median, CUDA events)"}
            cb_ = pair_two()
            gq = torch.Generator(device=dev).manual_seed(7)
            gvs = [torch.randn(o[0].shape, device=dev, generator=gq) for o in cb_]
            gms = [torch.randn(o[5]["msdf"].shape, device=dev, generator=gq) for o in cb_]
            split_pair["counts"] = {"cloth_faces": int(cb_[0][1].shape[0]), "body_faces": int(cb_[1][1].shape[0]),
                                    "verts_aug": int(cb_[0][0].shape[0])}
            for name, fn in variants.items():
                ts_ = []
                for rep in range(8 + min(max(args.steps, 10), 60)):
                    qp.grad = qs.grad = qm.grad = None
                    ea, eb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    ea.record()
                    c_, b_ = fn()
                    torch.autograd.backward([c_[0], c_[5]["msdf"], b_[0], b_[5]["msdf"]], [gvs[0], gms[0], gvs[1], gms[1]])
                    eb_.record()
                    barrier()
                    if rep >= 8:
                        ts_.append(ea.elapsed_time(eb_))
                split_pair[name + "_ms"] = float(np.median(ts_))
            split_pair["value"] = 2 * int(sf.shape[0]) / (min(split_pair[k + "_ms"] for k in variants) * 1e-3)
        except Exception as exc:  # noqa: BLE001
            split_pair = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- the stage in FRONT of the extraction (SURVEY 8f row 3): the SDF network on all N grid vertices in batches of 100000
    # (hmsdf.py:187, 434-444), tcgen05 / 3xTF32 kernels of this package against the same module in plain PyTorch fp32.
    # Never fatal.
    sdf_query = None
    if world == 1 and not args.no_sdf_query and dev_type == "cuda":
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("_mlp_bench", os.path.join(ROOT, "profiles", "mlp_bench.py"))
            mq = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mq)
            sdf_query = mq.measure(points=N, reps=3, dev=dev, tf32_leg=False)
        except Exception as exc:  # noqa: BLE001
            sdf_query = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- the stage BEHIND the extraction and the mesh wrapper (SURVEY 8f row 4): skinning of the extracted vertices, this
    # package against the reference's op sequence in PyTorch on the same device.  Never fatal.
    lbs_stage = None
    if world == 1 and not args.no_lbs_stage and dev_type == "cuda" and args.res == 128:
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("_lbs_bench", os.path.join(ROOT, "profiles", "lbs_bench.py"))
            lb = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(lb)
            lbs_stage = lb.measure(reps=5, dev=dev)
        except Exception as exc:  # noqa: BLE001
            lbs_stage = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- the reference's way on the same GPU: the path as plain PyTorch ops + autograd (oracle/gshell_torch.py, a port
    # pinned against the reference's golden vectors; the reference tree itself is not on this box).  SURVEY 8(d).  Never fatal.
    torch_baseline = None
    if world == 1 and not args.no_torch_baseline:
        try:
            from oracle import gshell_torch as GT
            tp = pos_single[0].detach().clone().requires_grad_(True)
            ts_, tm_ = sdf.detach().clone().requires_grad_(True), msdf.detach().clone().requires_grad_(True)

            def torch_step():
                tp.grad = ts_.grad = tm_.grad = None
                v, f_, _, _, _, ex = GT.extract(tp, ts_, tm_, tets, 1, True)
                torch.autograd.backward([v, ex["msdf"]], [ups_v[0], ups_m[0]])

            for _ in range(2):
                torch_step()
            reps, t_all = 0, time.perf_counter()
            barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            while reps < 20 and time.perf_counter() - t_all < 10.0:
                torch_step()
                reps += 1
            ev1.record()
            barrier()
            ms = ev0.elapsed_time(ev1) / max(reps, 1)
            torch_baseline = {"value": F / (ms * 1e-3), "unit": UNIT, "ms_per_frame": ms, "kind": "port", "reps": reps,
                              "note": "the same extraction fwd+bwd of one frame as plain PyTorch ops + autograd on this GPU "
                                      "(boolean-mask compactions, torch.unique(dim=0), scatter_add, the full UV table), "
                                      "the way the reference runs it; oracle/gshell_torch.py"}
        except Exception as exc:  # noqa: BLE001
            torch_baseline = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak" if args.mode == "weak" else "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args, world, F, N, c0, ngroups, fps),
            "ms_per_step_blocks": [round(b, 5) for b in block_ms],
            "roofline": roofline, "path_roofline": path_roofline, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "ranks": ranks_info, "device_trace": dev_trace, "single_call": single, "cold": cold,
            "gpu_launches": int(launches_timed), "kernels": kern, "split_pair": split_pair,
            "mesh_stage": mesh_stage, "sdf_query": sdf_query, "lbs_stage": lbs_stage, "torch_gpu_baseline": torch_baseline, "clocks": sampler.result()}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
