"""Device time of ``point_covariance`` (``mcba_point_covariance``) at configs[4]: 1 M keypoints x 6 cameras,
sigma 0.3 px, 20 % missing views, points from ``refine_points`` (linear loss).  The median of 20 calls by CUDA
events around the C ABI call on device buffers, with and without the sensitivity output, and the time of the
public numpy call; FP64 FMAs counted from shapes against ``mcba_measure_fp64_peak``, measured in the same run, and
the card's name and power limit.

FMA count per point with |V| seen views (n = 12 |V| parameters): the product S cov S^T restricted to the seen
cameras, 3 n^2 + 6 n.  The kernel issues more: it runs the product over the columns of all cameras, in passes
of 96 columns, for the cameras seen by any of the four points of a batch; that figure is reported too.

    python scripts/point_covariance_timing.py [--reps 20] [--out profiles/point_covariance_timing.json]
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--out", default="profiles/point_covariance_timing.json")
    args = ap.parse_args()
    import multicam_calibration_b200 as mcc
    from multicam_calibration_b200 import _native
    from multicam_calibration_b200.synthetic import make_keypoints
    from refine_points_timing import gpu_identity
    torch = _native.require_cuda()
    lib = _native.load()
    fma = ctypes.c_double()
    _native.check(lib.mcba_measure_fp64_peak(0, ctypes.byref(fma)))

    all_uvs, ext, intr, _ = make_keypoints(args.points, 6, sigma=0.3, p_missing=0.2, seed=0)
    uvs = np.stack(all_uvs)
    C, P, _ = uvs.shape
    n = 12 * C
    Ks = np.ascontiguousarray(np.stack([K for K, _ in intr]))
    dists = np.zeros((C, 5))
    for c, (_, d) in enumerate(intr):
        dists[c, :len(d)] = np.asarray(d)[:5]
    ext = np.ascontiguousarray(ext)
    res = mcc.refine_points(uvs, ext, intr)
    rng = np.random.default_rng(1)
    A = rng.normal(size=(n, n + 8))
    cov = np.ascontiguousarray(A @ A.T * 1e-3)
    cov[6:12] = cov[:, 6:12] = 0.0          # camera 0's extrinsics: the gauge

    seen = ~np.isnan(uvs).any(-1)           # the "seen" rule on these finite pixels
    live = np.isfinite(res.covariance).all((1, 2))
    nv = 12 * seen.sum(0)[live].astype(np.float64)
    fmas = float((3 * nv * nv + 6 * nv).sum())
    batches = seen[:, :P - P % 4].reshape(C, -1, 4).any(-1).sum(0)   # cameras seen in each batch of four points
    issued = float((batches * 12 * (3 * 4) * (96 * -(-n // 96))).sum())

    d_uv = _native.to_device(uvs)
    d_pts = _native.to_device(res.points)
    f64 = dict(dtype=torch.float64, device="cuda")
    d_meas = torch.empty((P, 6), **f64)
    d_cal = torch.empty((P, 6), **f64)
    d_sens = torch.empty((P, 3, n), **f64)
    ptr = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())  # noqa: E731
    h = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    stream = torch.cuda.current_stream()

    def call(sens):
        _native.check(lib.mcba_point_covariance(0, ctypes.c_void_p(stream.cuda_stream), ptr(d_uv), C, P, h(ext),
                                                h(Ks), h(dists), ptr(d_pts), h(cov), 0, 1.0, 1.0, ptr(d_meas),
                                                ptr(d_cal), ptr(d_sens if sens else None)))

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
    for sens in (False, True):
        ms = timed(lambda: call(sens), args.reps)
        api = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mcc.point_covariance(uvs, ext, intr, res.points, cov, sensitivity=sens)
            api.append(1e3 * (time.perf_counter() - t0))
        rows.append(dict(sensitivity=sens, call_ms_median=ms, public_call_ms_median=float(np.median(api)),
                         fp64_fma_product=fmas, fp64_share_of_peak=fmas / (ms * 1e-3) / fma.value,
                         fp64_fma_issued=issued, issued_share_of_peak=issued / (ms * 1e-3) / fma.value,
                         output_bytes=P * 96 + (P * 3 * n * 8 if sens else 0)))
        print(json.dumps(rows[-1]), flush=True)
    result = dict(gpu=gpu_identity(), points=P, cameras=C, live_points=int(live.sum()),
                  fp64_fma_per_s_measured=fma.value, runs=rows,
                  note="call_ms: CUDA events around mcba_point_covariance on device buffers (camera and covariance "
                       "upload of 41 KB, one kernel, stream synchronisation)")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
