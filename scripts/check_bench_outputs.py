#!/usr/bin/env python
"""Check what the benchmark computed against the blockwise fp64 reference.

    python bench.py --gpus 1 --steps 20 --warmup 5 --dump-outputs DIR
    python scripts/check_bench_outputs.py DIR

Rebuilds the seeded BASELINE configs[2] scene with bench.py's own constants (6 cameras x 50,000 frames,
0.5 px noise, 20 % missing views, seed 0; lambda 1e-3, soft_l1), evaluates oracle/blockwise.py at x0 (about
15 s on one host core) and compares every file bench.py wrote: S, b, g_cam, cost and the gradient
[g_cam | g_pose].  An output bench.py had to sample comes with `<name>_index.npy` (flat indices); only those
entries are compared.  Tolerances are those of tests/test_scale_parity.py.  Exits non-zero on disagreement.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (constants only: bench.py runs nothing on import)
from multicam_calibration_b200.synthetic import make_scene  # noqa: E402
from oracle import blockwise  # noqa: E402


def load(path, name):
    a = np.load(os.path.join(path, name + ".npy"))
    ix = os.path.join(path, name + "_index.npy")
    return a, (np.load(ix).astype(np.int64) if os.path.exists(ix) else None)


def main(path):
    cfg = bench.CONFIGS[2]
    sc = make_scene(cfg["cams"], cfg["frames"], sigma=bench.SIGMA, p_missing_view=bench.P_MISSING, seed=0)
    ev = blockwise.BlockwiseEvaluation(sc.x0(), sc.uvs, sc.objpoints, lam=bench.LAMBDA, loss=bench.LOSS)
    nc = 12 * ev.C
    grad = np.r_[ev.g_cam, ev.g_pose.ravel()]
    gmax = np.abs(grad).max()
    # name -> (reference, per-entry tolerance)
    checks = {
        "S": (ev.S, np.full(ev.S.size, 1e-9 * np.abs(ev.S).max())),
        "b": (ev.b, np.full(nc, 1e-9 * np.abs(ev.b).max())),
        "g_cam": (ev.g_cam, np.full(nc, 1e-10 * np.abs(ev.g_cam).max())),
        "cost": (np.array([ev.cost]), np.array([1e-12 * ev.cost])),
        "gradient": (grad, np.r_[np.full(nc, 1e-10 * np.abs(ev.g_cam).max()),
                                 np.repeat(1e-9 * np.abs(ev.g_pose).max(1) + 1e-12 * gmax, 6)]),
    }
    report, ok = {}, True
    for name, (ref, tol) in checks.items():
        if not os.path.exists(os.path.join(path, name + ".npy")):
            report[name] = "missing"
            ok = False
            continue
        got, idx = load(path, name)
        ref, tol = ref.ravel(), tol.ravel()
        if idx is not None:
            ref, tol = ref[idx], tol[idx]
        if got.size != ref.size:
            report[name] = f"size {got.size}, expected {ref.size}"
            ok = False
            continue
        err = np.abs(got.ravel() - ref)
        good = bool((err <= tol).all())
        report[name] = {"entries": int(got.size), "max_abs_err": float(err.max()),
                        "worst_err_over_tol": float((err / tol).max()), "ok": good}
        ok &= good
    if os.path.exists(os.path.join(path, "gradient.npy")):
        got, idx = load(path, "gradient")
        full = np.arange(grad.size) if idx is None else idx
        empty = np.nonzero(np.repeat(ev.empty, 6))[0] + nc
        hit = np.isin(full, empty)
        good = bool((got.ravel()[hit] == 0.0).all())
        report["empty_frames"] = {"frames": int(ev.empty.sum()), "gradient_exactly_zero": good}
        ok &= good
    print(json.dumps({"agree": ok, "outputs": report}, indent=1))
    return 0 if ok else 1


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1]))
