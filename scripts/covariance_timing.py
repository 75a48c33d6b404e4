"""Device time of the calibration covariance (``BAProblem.covariance`` / ``mcba_covariance``) at the benchmark
scene (BASELINE configs[2]: 6 cameras x 50,000 frames) and at one 16 x 25,000 shard of configs[3], split into
evaluation (+ frame check), camera inverse (including its two host read-backs) and the pose kernel (CUDA events
inside the call), with the pose kernel set against its byte and FP64 floors.  The card's name, power limit and
measured FP64 FMA rate are read in the same run.

    python scripts/covariance_timing.py [--reps 20] [--out profiles/covariance_timing.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


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


def pose_kernel_floors(prob, fma_per_s):
    """Bytes and FP64 FMAs the pose kernel needs: the live (tile, camera) units of Z, L^-1 and the output;
    sum over tiles of 32 frames x (live cameras)^2 x 12 x 12 x 6 FMAs for Sigma_raw Z plus 12 x 21 per live camera."""
    plan = prob.plan_info()
    units = int(sum(plan["units"]))
    tiles = plan["tiles"]
    nbytes = units * 12 * 6 * 32 * 8 + tiles * 21 * 32 * 8 + prob.F * 36 * 8
    live = units / tiles                                  # average live cameras per tile
    fma = tiles * 32 * (live ** 2 * 864 + live * 12 * 21)
    return dict(bytes=nbytes, fma=fma, byte_floor_ms=1e3 * nbytes / HBM_BYTES_PER_S,
                fp64_floor_ms=1e3 * fma / fma_per_s, live_units=units, tiles=tiles)


def time_scene(name, C, F, reps, fma_per_s, shard=0, seed=0):
    import torch
    import multicam_calibration_b200 as mcc
    from multicam_calibration_b200.synthetic import make_scene
    sc = make_scene(C, F, sigma=0.5, p_missing_view=0.2, seed=seed, shard=shard)
    x = sc.x0()
    prob = mcc.BAProblem(sc.uvs, sc.objpoints)
    for _ in range(3):
        prob.covariance(x)
    rows = []
    for _ in range(reps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(prob.stream)
        _, _, info = prob.covariance(x)
        b.record(prob.stream)
        b.synchronize()
        rows.append([info["eval_ms"], info["camera_ms"], info["pose_ms"], a.elapsed_time(b)])
    med = np.median(np.array(rows), axis=0)
    floors = pose_kernel_floors(prob, fma_per_s)
    prob.close()
    return dict(scene=name, cameras=C, frames=F, reps=reps,
                median_ms=dict(evaluation_and_frame_check=med[0], camera_inverse=med[1], pose_kernel=med[2],
                               whole_call_incl_host=med[3]),
                pose_kernel=dict(floors, share_of_byte_floor=floors["byte_floor_ms"] / med[2],
                                 share_of_fp64_floor=floors["fp64_floor_ms"] / med[2]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="profiles/covariance_timing.json")
    args = ap.parse_args()
    from multicam_calibration_b200 import _native
    _native.require_cuda()
    lib = _native.load()
    fma = ctypes.c_double()
    _native.check(lib.mcba_measure_fp64_peak(0, ctypes.byref(fma)))
    result = dict(gpu=gpu_identity(), fp64_fma_per_s_measured=fma.value, hbm_bytes_per_s_datasheet=HBM_BYTES_PER_S,
                  scenes=[time_scene("configs[2] 6 x 50,000", 6, 50000, args.reps, fma.value),
                          time_scene("configs[3] shard 16 x 25,000", 16, 25000, args.reps, fma.value, seed=3)])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
