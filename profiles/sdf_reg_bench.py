#!/usr/bin/env python
"""The SDF sign-change regulariser: the reference's PyTorch form (geometry/hmsdf.py:162-170) against
geometry/sdf_reg.compute_sdf_reg_loss on the same GPU, at the benchmark's two grids -- the 128^3 Kuhn lattice with the
capsule body field (run-length table) and smplx_layout_grid(128) with the same field (transposed rows).  Prints one JSON
line; writes nothing.

    python profiles/sdf_reg_bench.py [--reps 200] [--warmup 20]

Per workload: E, N, the table form and its bytes; forward and forward + backward times (CUDA events, median of --reps
single-call timings) for both forms, with warm caches and with a 256 MB buffer written between reps (L2 is 126 MB);
the bytes the native op needs (table + sign bitmaps + 4 bytes per vertex read for the bitmaps + 8 bytes per selected edge
read and, with the backward pass, 8 bytes per selected edge scattered) and the achieved GB/s; the largest difference to
the PyTorch result; and whether forward + backward of the native op ran under torch.cuda.set_sync_debug_mode("error").
The card name and power limit are read in the same run.

In the L2-flushed timings the flush kernel is queued before the first event, so the host work of the timed call (Python,
ctypes, the autograd node) overlaps it and the window holds device time; in the warm timings the device waits for that
host work, which is why the native op's warm times are the larger ones.  profiles/sdf_reg_bench_b200.json: one run on a
B200."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from d3human_code_b200 import grids  # noqa: E402
from d3human_code_b200.geometry import sdf_reg as R  # noqa: E402


def torch_form(sdf, all_edges):
    """the reference's compute_sdf_reg_loss (hmsdf.py:162-170)"""
    sdf_f1x6x2 = sdf[all_edges.reshape(-1)].reshape(-1, 2)
    mask = torch.sign(sdf_f1x6x2[..., 0]) != torch.sign(sdf_f1x6x2[..., 1])
    sdf_f1x6x2 = sdf_f1x6x2[mask]
    return F.binary_cross_entropy_with_logits(sdf_f1x6x2[..., 0], (sdf_f1x6x2[..., 1] > 0).float()) + \
        F.binary_cross_entropy_with_logits(sdf_f1x6x2[..., 1], (sdf_f1x6x2[..., 0] > 0).float())


def all_edges_of(tets, n):
    """generate_edges (hmsdf.py:381-388): the distinct (min, max) tet edges, ascending, int64"""
    sel = torch.tensor([0, 1, 0, 2, 0, 3, 1, 2, 1, 3, 2, 3], device=tets.device)
    e = tets[:, sel].reshape(-1, 2)
    key = torch.unique(torch.minimum(e[:, 0], e[:, 1]) * n + torch.maximum(e[:, 0], e[:, 1]))
    a = torch.div(key, n, rounding_mode="floor")
    return torch.stack([a, key - a * n], 1)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:   # noqa: BLE001
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unavailable ({exc})"}


def timed(fn, reps, warmup, flush):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        if flush is not None:
            flush.add_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times)), float(np.min(times))


def workload(name, sdf_np, tets_np, reps, warmup, flush):
    dev = torch.device("cuda")
    n = sdf_np.shape[0]
    edges = all_edges_of(torch.from_numpy(tets_np).to(dev), n)
    tab = R.tables_for(edges, n)
    s = torch.from_numpy(sdf_np).to(dev).reshape(-1, 1).requires_grad_()

    def fwd_t():
        torch_form(s.detach(), edges)

    def fb_t():
        s.grad = None
        torch_form(s, edges).backward()

    def fwd_n():
        R.compute_sdf_reg_loss(s.detach(), edges)

    def fb_n():
        s.grad = None
        R.compute_sdf_reg_loss(s, edges).backward()

    # results
    s.grad = None
    lt = torch_form(s, edges)
    lt.backward()
    gt = s.grad.clone()
    s.grad = None
    ln = R.compute_sdf_reg_loss(s, edges)
    ln.backward()
    gn = s.grad.clone()
    torch.cuda.synchronize()
    m = int((torch.sign(s.detach().reshape(-1)[edges[:, 0]]) != torch.sign(s.detach().reshape(-1)[edges[:, 1]])).sum())
    sync_free = True
    torch.cuda.set_sync_debug_mode("error")
    try:
        fb_n()
    except RuntimeError:
        sync_free = False
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    out = {"workload": name, "E": int(edges.shape[0]), "N": n, "M": m, "form": tab.form, "table_bytes": tab.nbytes,
           "loss_torch": lt.item(), "loss_native": ln.item(),
           "loss_rel_diff": abs(ln.item() - lt.item()) / abs(lt.item()),
           "grad_max_diff_over_max": float((gn - gt).abs().max() / gt.abs().max()),
           "native_fwd_bwd_without_host_sync": sync_free}
    words = (n + 31) // 32 + 1
    need_fwd = tab.nbytes + 4 * n + 2 * 4 * words * 2 + 8 * m          # table, sdf for the bitmaps, bitmaps written+read, end points
    need_bwd = tab.nbytes + 2 * 4 * words + 8 * m + 8 * m + 4 * n      # the scan again, atomics, g_sdf zero fill
    out["bytes_fwd"], out["bytes_fwd_bwd"] = need_fwd, need_fwd + need_bwd
    for cache, fl in (("warm", None), ("l2_flushed", flush)):
        for label, fn in (("torch_fwd", fwd_t), ("torch_fwd_bwd", fb_t), ("native_fwd", fwd_n), ("native_fwd_bwd", fb_n)):
            med, mn = timed(fn, reps, warmup, fl)
            out[f"{label}_ms_{cache}"] = med
            out[f"{label}_ms_{cache}_min"] = mn
        out[f"speedup_fwd_{cache}"] = out[f"torch_fwd_ms_{cache}"] / out[f"native_fwd_ms_{cache}"]
        out[f"speedup_fwd_bwd_{cache}"] = out[f"torch_fwd_bwd_ms_{cache}"] / out[f"native_fwd_bwd_ms_{cache}"]
        out[f"native_fwd_GBps_{cache}"] = need_fwd / out[f"native_fwd_ms_{cache}"] / 1e6
        out[f"native_fwd_bwd_GBps_{cache}"] = (need_fwd + need_bwd) / out[f"native_fwd_bwd_ms_{cache}"] / 1e6
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--res", type=int, default=128)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    flush = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device="cuda")   # 256 MB > L2
    pos, tets = grids.kuhn_grid(args.res)
    res = [workload(f"kuhn{args.res}_capsule", grids.capsule_garment_field(pos)[0], tets, args.reps, args.warmup, flush)]
    g = grids.smplx_layout_grid(args.res)
    res.append(workload(f"smplx_layout{args.res}_capsule", grids.capsule_garment_field(g["v"])[0], g["f"], args.reps, args.warmup,
                        flush))
    print(json.dumps({"card": card(), "reps": args.reps, "warmup": args.warmup, "workloads": res}))


if __name__ == "__main__":
    main()
