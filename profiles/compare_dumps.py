#!/usr/bin/env python
"""Compares what two builds computed for the same bench step: the .npy files that `bench.py --dump-outputs DIR` writes.

    python profiles/compare_dumps.py BASE NEW [BASE2]

BASE and NEW are the dumps of the old and the new build.  BASE2, a second dump of the old build, gives the run-to-run
spread of the outputs that are sums of float atomics.
- counts and the integer / interpolated outputs (faces_aug, faces_watertight, verts_aug, msdf, vertices_watertight,
  msdf_watertight) must be bit-identical;
- the tangents (v_tng_aug, v_tng_watertight) are sums of float atomics: the largest difference NEW - BASE must stay
  within twice the largest difference BASE2 - BASE (exact equality when no BASE2 is given);
- the gradients (grad_pos, grad_sdf, grad_msdf) must agree normwise: |NEW - BASE| / |BASE| <= 1e-5.
Prints one line per file and exits with 1 if any check fails."""
import os
import sys

import numpy as np

EXACT = ("counts", "faces_aug", "faces_watertight", "verts_aug", "msdf", "vertices_watertight", "msdf_watertight")
ATOMIC_SUMS = ("v_tng_aug", "v_tng_watertight")
GRADIENTS = ("grad_pos", "grad_sdf", "grad_msdf")
GRAD_RTOL = 1e-5


def load(d, name):
    return np.load(os.path.join(d, name + ".npy"))


def max_abs_diff(a, b):
    if a.shape != b.shape:
        return float("inf")
    d = np.abs(a.astype(np.float64) - b.astype(np.float64))
    both_nan = np.isnan(a) & np.isnan(b)
    d[both_nan] = 0.0
    return float(np.nan_to_num(d, nan=np.inf).max()) if d.size else 0.0


def main(argv):
    if len(argv) not in (3, 4):
        raise SystemExit(__doc__)
    base, new = argv[1], argv[2]
    base2 = argv[3] if len(argv) == 4 else None
    ok = True
    for name in EXACT:
        a, b = load(base, name), load(new, name)
        same = a.shape == b.shape and np.array_equal(a, b, equal_nan=True)
        print(f"{name:20s} {'identical' if same else 'DIFFERS'}  shape {b.shape}")
        ok = ok and same
    for name in ATOMIC_SUMS:
        a, b = load(base, name), load(new, name)
        d = max_abs_diff(a, b)
        spread = max_abs_diff(a, load(base2, name)) if base2 else 0.0
        good = d <= 2.0 * spread if base2 else d == 0.0
        print(f"{name:20s} max |new - base| {d:.3e}  run-to-run max |base2 - base| {spread:.3e}  {'ok' if good else 'FAIL'}")
        ok = ok and good
    for name in GRADIENTS:
        a, b = load(base, name).astype(np.float64), load(new, name).astype(np.float64)
        if a.shape != b.shape:
            print(f"{name:20s} shape {a.shape} != {b.shape}  FAIL")
            ok = False
            continue
        err = float(np.linalg.norm(b - a) / max(np.linalg.norm(a), 1e-30))
        print(f"{name:20s} normwise {err:.3e}  {'ok' if err <= GRAD_RTOL else 'FAIL'}")
        ok = ok and err <= GRAD_RTOL
    print("PASS" if ok else "FAIL")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv))
