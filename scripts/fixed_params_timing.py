"""LM solve time with camera parameters held (``BAProblem.solve(fixed=...)``) against the unmasked solve, at the
benchmark scene (BASELINE configs[2]: 6 cameras x 50,000 frames) and at one 16 x 25,000 shard of configs[3].

Masks: none, intrinsics held, camera 0 pinned (its six extrinsics), pose-only (every camera parameter held).  Every
solve uses the library defaults (ftol 1e-4) and starts from the same x0; the masks are run alternately, ``--reps``
rounds, and the medians are reported: the whole solve (CUDA events inside ``mcba_lm_run``), the evaluations it
needed and the time per evaluation.  The mask is 12C bytes read by kernels that already run, so a masked
evaluation should cost what an unmasked one does.  The card's name and power limit are read in the same run.

    python scripts/fixed_params_timing.py [--reps 10] [--out profiles/fixed_params_timing.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_identity():
    import torch
    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except (OSError, subprocess.TimeoutExpired):
        out["power_limit_and_max_sm_clock"] = None
    return out


def masks(C):
    out = {"none": None}
    m = np.zeros((C, 12), dtype=bool)
    m[:, :6] = True
    out["intrinsics"] = m
    m = np.zeros((C, 12), dtype=bool)
    m[0, 6:] = True
    out["camera0_pinned"] = m
    out["pose_only"] = np.ones((C, 12), dtype=bool)
    return out


def time_scene(name, C, F, reps, seed=0):
    import multicam_calibration_b200 as mcc
    from multicam_calibration_b200.synthetic import make_scene
    sc = make_scene(C, F, sigma=0.5, p_missing_view=0.2, seed=seed)
    x0 = sc.x0()
    prob = mcc.BAProblem(sc.uvs, sc.objpoints)
    ms = masks(C)
    for fixed in ms.values():                       # warm-up: module loads, allocations of every path
        prob.solve(x0, fixed=fixed, verbose=0)
    rows = {k: [] for k in ms}
    for _ in range(reps):
        for k, fixed in ms.items():
            _, res = prob.solve(x0, fixed=fixed, verbose=0)
            rows[k].append((res.solve_ms, res.nfev, res.iterations, res.kernel_launches, res.cost))
    prob.close()
    out = dict(scene=name, cameras=C, frames=F, reps=reps, masks={})
    for k, r in rows.items():
        a = np.array(r)
        out["masks"][k] = dict(solve_ms_median=float(np.median(a[:, 0])), solve_ms_min=float(a[:, 0].min()),
                               solve_ms_max=float(a[:, 0].max()), nfev=int(a[0, 1]), iterations=int(a[0, 2]),
                               kernel_launches=int(a[0, 3]), cost=float(a[0, 4]),
                               ms_per_evaluation=float(np.median(a[:, 0] / a[:, 1])))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="profiles/fixed_params_timing.json")
    args = ap.parse_args()
    from multicam_calibration_b200 import _native
    _native.require_cuda()
    result = dict(gpu=gpu_identity(),
                  scenes=[time_scene("configs[2] 6 x 50,000", 6, 50000, args.reps),
                          time_scene("configs[3] shard 16 x 25,000", 16, 25000, args.reps, seed=3)])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
