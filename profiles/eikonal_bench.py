#!/usr/bin/env python
"""The eikonal step of D3-Human's training loop (hmsdf.py:856-880) on one GPU: the SDF network (n_freq 6, 256 wide, 6 hidden
layers, skip_in [3]; train.py:1622-1625) on P points in batches of 100000 (hmsdf.py:187), timed as
    sdf = net(x);  gx = autograd.grad(sdf, x, ones, create_graph=True);  ((|gx| - 1)^2).mean().backward()
for this package (tcgen05, 3xTF32; the double backward in geometry/mlp.py) against the same layers in plain torch fp32
(TF32 off, how the reference runs).  CUDA events, median of --reps after one warm-up pass.  Prints one JSON line with the
FLOPs counted from the shapes, the largest differences between the two arms, and the card's name and power limit.
    python profiles/eikonal_bench.py [--points 100000] [--batch 100000] [--reps 10]"""
import argparse, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)
import numpy as np, torch

from mlp_bench import CFG, TorchMLP


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def measure(points=100000, batch=100000, reps=10):
    from d3human_code_b200.geometry import mlp as M
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(0)
    ours = M.MLP(**CFG).to(dev)
    ref = TorchMLP(ours)
    params = list(ours.parameters())
    pts = torch.rand(points, 3, device=dev) * 2 - 1
    # forward: Linear(39,256) + 5 Linear(256,256) + Linear(295,256) + Linear(256,1).  The eikonal step is ~7 of those:
    # forward, first backward (input and weight gradients), tangent pass, adjoint pass, two weight-gradient contractions.
    flops_fwd = 2.0 * (39 * 256 + 5 * 256 * 256 + 295 * 256 + 256) * points
    flops = 7.0 * flops_fwd

    def run(net):
        for p in params:
            p.grad = None
        gxs, xgs = [], []
        for i in range(0, points, batch):
            x = pts[i:i + batch].clone().requires_grad_(True)
            sdf = net(x)
            gx, = torch.autograd.grad(sdf, x, torch.ones_like(sdf), create_graph=True)
            ((gx.norm(dim=-1) - 1.0) ** 2).mean().backward()
            gxs.append(gx.detach())
            xgs.append(x.grad)
        return torch.cat(gxs), torch.cat(xgs), [p.grad.clone() if p.grad is not None else None for p in params]

    def timed(net):
        run(net)
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); run(net); b.record(); b.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts)), float(min(ts)), float(max(ts))

    res = {"gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "points": points, "batch": batch,
           "network": CFG, "flops_eikonal_step": flops, "flops_forward": flops_fwd,
           "unit": "ms for all points, forward + autograd.grad(create_graph=True) + eikonal backward (median of %d, CUDA events)" % reps}
    g0, x0, p0 = run(ours)
    g1, x1, p1 = run(ref)
    res["max_abs_diff_gx"] = float((g0 - g1).abs().max())
    res["max_abs_gx"] = float(g1.abs().max())
    res["normwise_diff_x_grad"] = float((x0 - x1).norm() / x1.norm())
    res["max_normwise_diff_param_grads"] = max(float((a - b).norm() / b.norm()) for a, b in zip(p0, p1) if b is not None)
    res["output_bias_grad_ours_is_none"] = p0[-1] is None
    for name, net in (("ours", ours), ("torch_fp32", ref)):
        med, lo, hi = timed(net)
        res[name + "_ms"], res[name + "_ms_min"], res[name + "_ms_max"] = med, lo, hi
        res[name + "_tflops"] = flops / (med * 1e-3) / 1e12
    res["speedup_vs_torch_fp32"] = res["torch_fp32_ms"] / res["ours_ms"]
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=100000)
    ap.add_argument("--batch", type=int, default=100000)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    print(json.dumps(measure(a.points, a.batch, a.reps)))
