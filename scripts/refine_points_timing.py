"""Device time of ``refine_points`` (``mcba_refine_points``) at configs[4]: 1 M keypoints x 6 cameras, sigma 0.3 px,
20 % missing views, for each of the five losses.  Per loss: the median of 20 calls by CUDA events around the C ABI
call on device buffers (start given, so the time is the refinement kernel alone; and with the triangulation in the
call), mean / maximum iterations, achieved FP64 FMAs against ``mcba_measure_fp64_peak`` and bytes against a
device-to-device copy rate, both measured in the same run, and the time of the public numpy call.  The card's
name and power limit are read in the same run.

FMA count per seen view, from the kernel's source (k9_refine.cu), counting a multiply or add as one FMA slot:
the "seen" undistortion 75, a projection with its Jacobian and two accumulated scalars 80, a projection for a
trial cost 25.  A point that takes k trial steps runs at most k + 2 Jacobian passes (start, one per accepted step,
the closing pass) and k trial costs; the achieved figure takes every step as accepted, so it is an upper bound
on the useful work.

    python scripts/refine_points_timing.py [--reps 20] [--out profiles/refine_points_timing.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

FMA_SEEN, FMA_JAC, FMA_COST = 75, 80, 25
LOSSES = ("linear", "soft_l1", "huber", "cauchy", "arctan")


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


def copy_rate(torch, nbytes=2 << 30, reps=10):
    """Bytes moved per second (read + write) by a device-to-device copy larger than the L2."""
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 0.0
    for _ in range(reps):
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * nbytes / (e0.elapsed_time(e1) * 1e-3))
    del a, b
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--out", default="profiles/refine_points_timing.json")
    args = ap.parse_args()
    import multicam_calibration_b200 as mcc
    from multicam_calibration_b200 import _native
    from multicam_calibration_b200.synthetic import make_keypoints
    torch = _native.require_cuda()
    lib = _native.load()
    fma = ctypes.c_double()
    _native.check(lib.mcba_measure_fp64_peak(0, ctypes.byref(fma)))
    bw = copy_rate(torch)

    all_uvs, ext, intr, _ = make_keypoints(args.points, 6, sigma=0.3, p_missing=0.2, seed=0)
    uvs = np.stack(all_uvs)
    C, P, _ = uvs.shape
    Ks = np.ascontiguousarray(np.stack([K for K, _ in intr]))
    dists = np.zeros((C, 5))
    for c, (_, d) in enumerate(intr):
        dists[c, :len(d)] = np.asarray(d)[:5]
    ext = np.ascontiguousarray(ext)
    tri = mcc.triangulate(all_uvs, list(ext), intr)
    views = (~np.isnan(uvs).any(-1)).sum(0)
    d_uv = _native.to_device(uvs)
    d_init = _native.to_device(tri)
    f64 = dict(dtype=torch.float64, device="cuda")
    out = dict(points=torch.empty((P, 3), **f64), cost=torch.empty(P, **f64), rms=torch.empty(P, **f64),
               status=torch.empty(P, dtype=torch.int8, device="cuda"),
               iters=torch.empty(P, dtype=torch.int16, device="cuda"), cov=torch.empty((P, 6), **f64))
    ptr = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())  # noqa: E731
    h = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    stream = torch.cuda.current_stream()

    def call(loss, init):
        opt = _native.RefineOptions(loss=_native.REFINE_LOSSES[loss], f_scale=1.0, sigma=1.0, ftol=1e-12,
                                    xtol=1e-12, gtol=1e-10, max_iter=50, flags=0)
        _native.check(lib.mcba_refine_points(0, ctypes.c_void_p(stream.cuda_stream), ptr(d_uv), C, P, h(ext), h(Ks),
                                             h(dists), ptr(init), ctypes.byref(opt), ptr(out["points"]),
                                             ptr(out["cost"]), ptr(out["rms"]), ptr(out["status"]),
                                             ptr(out["iters"]), ptr(out["cov"]), None, None))

    def timed(fn, reps):
        fn()
        fn()
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms))

    rows = []
    for loss in LOSSES:
        ms = timed(lambda: call(loss, d_init), args.reps)
        ms_tri = timed(lambda: call(loss, None), args.reps)
        it = _native.to_host(out["iters"]).astype(np.int64)
        st = _native.to_host(out["status"])
        live = st >= 0
        nv = views[live]
        fmas = float((nv * (FMA_SEEN + FMA_JAC * (it[live] + 2) + FMA_COST * it[live])).sum())
        nbytes = P * C * 16 + P * (24 + 24 + 8 + 8 + 1 + 2 + 48)   # observations, start, outputs with covariance
        mcc.refine_points(all_uvs, ext, intr, loss=loss)
        api = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mcc.refine_points(all_uvs, ext, intr, loss=loss)
            api.append(1e3 * (time.perf_counter() - t0))
        rows.append(dict(loss=loss, kernel_ms_median=ms, with_triangulation_ms_median=ms_tri,
                         public_call_ms_median=float(np.median(api)),
                         iterations_mean=float(it[live].mean()), iterations_max=int(it.max()),
                         status_histogram={int(k): int(v) for k, v in zip(*np.unique(st, return_counts=True))},
                         fp64_fma_upper_bound=fmas, fp64_share_of_peak=fmas / (ms * 1e-3) / fma.value,
                         bytes=nbytes, bytes_share_of_copy_rate=nbytes / (ms * 1e-3) / bw))
        print(json.dumps(rows[-1]), flush=True)
    result = dict(gpu=gpu_identity(), points=P, cameras=C, fp64_fma_per_s_measured=fma.value,
                  d2d_copy_bytes_per_s_measured=bw, fma_per_view=dict(seen=FMA_SEEN, jacobian_pass=FMA_JAC,
                                                                      trial_cost=FMA_COST), losses=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
