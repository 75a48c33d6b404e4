"""Reprojection-error quality control: drop-in for the numeric part of
``multicam_calibration.viz.plot_residuals`` (reference viz.py:70-210).

``reprojection_residuals`` is the numeric core (viz.py:155-177) on the GPU: projection of the board
corners without distortion, undistortion of the detections, one homography per (camera, frame) that
carries the projections into the board's own coordinates (``mcba_homography_transfer``) and the
per-camera median distance to the true corners (exact, by radix selection on the device).
``plot_residuals`` keeps the reference's signature and return values and draws the same figure when
matplotlib is installed.
"""
import ctypes

import numpy as np

from . import _native
from ._native import check


def _device_median(lib, dev, stream, d_vals):
    """np.nanmedian of a non-negative float64 device vector (NaN = skip), exact: radix selection
    over 256-bin histograms of the bit patterns (the selection loop of the frame-sharded front end)."""
    from .distributed import kth_smallest
    torch = _native.require_cuda()
    d_hist = torch.empty(256, dtype=torch.int64, device=d_vals.device)

    def histogram(prefix, prefix_bits):
        check(lib.mcba_key_histogram(dev, stream, ctypes.c_void_p(d_vals.data_ptr()), d_vals.numel(),
                                     ctypes.c_uint64(prefix), prefix_bits, ctypes.c_void_p(d_hist.data_ptr())))
        return d_hist.cpu().numpy()

    n = int(histogram(0, 0).sum())
    if n == 0:
        return float("nan")
    same = lambda a: np.asarray(a)
    if n & 1:
        return kth_smallest(histogram, [n // 2], reduce=same)[0]
    lo, hi = kth_smallest(histogram, [n // 2 - 1, n // 2], reduce=same)
    return 0.5 * (lo + hi)


def reprojection_residuals(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints, calib_poses):
    """Numeric core of ``plot_residuals`` (viz.py:155-177).

    Returns ``(median_error (C,), reprojections (C,F,N,2), transformed_reprojections (C,F,N,2))``:
    the median distance between the board corners and the reprojections carried into the board's
    plane (board units), the distortion-free projections of the corners, and those projections in
    board coordinates (NaN where a frame has a missing corner)."""
    torch = _native.require_cuda()
    lib = _native.load()
    dev = torch.cuda.current_device()
    uvs = np.ascontiguousarray(all_calib_uvs, dtype=np.float64)
    obj = np.ascontiguousarray(calib_objpoints, dtype=np.float64)
    poses = np.ascontiguousarray(calib_poses, dtype=np.float64).reshape(-1, 6)
    C, F, N, _ = uvs.shape
    if poses.shape[0] != F or obj.shape != (N, 3) or len(all_extrinsics) != C or len(all_intrinsics) != C:
        raise ValueError("reprojection_residuals: inconsistent shapes")
    if F == 0:   # no frame, no distance: empty outputs and NaN medians (empty tensors have no device pointer)
        return np.full(C, np.nan), np.zeros((C, 0, N, 2)), np.zeros((C, 0, N, 2))
    ext =np.ascontiguousarray(np.stack([np.asarray(e, dtype=np.float64) for e in all_extrinsics]))
    Ks = np.ascontiguousarray(np.stack([np.asarray(K, dtype=np.float64) for K, _ in all_intrinsics]))
    dist = np.zeros((C, 5))
    for c, (_, d) in enumerate(all_intrinsics):
        d = np.asarray(d, dtype=np.float64).ravel()[:5]
        dist[c, :d.size] = d
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    hp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    device = f"cuda:{dev}"
    d_uvs, d_obj, d_pose = _native.to_device(uvs, dev), _native.to_device(obj, dev), _native.to_device(poses, dev)
    d_world = torch.empty((F, N, 3), dtype=torch.float64, device=device)
    check(lib.mcba_embed_points(dev, stream, ptr(d_pose), F, ptr(d_obj), N, ptr(d_world)))
    d_rep = torch.empty((C, F, N, 2), dtype=torch.float64, device=device)
    check(lib.mcba_project_points_multi(dev, stream, ptr(d_world), F * N, C, hp(ext), hp(Ks), None, ptr(d_rep)))   # no distortion (viz.py:161-163)
    d_tr = torch.empty((C, F, N, 2), dtype=torch.float64, device=device)
    d_err = torch.empty((C, F, N), dtype=torch.float64, device=device)
    check(lib.mcba_homography_transfer(dev, stream, ptr(d_uvs), ptr(d_rep), ptr(d_obj), C, F, N, hp(Ks), hp(dist),
                                       ptr(d_tr), ptr(d_err)))
    median_error = np.array([_device_median(lib, dev, stream, d_err[c].reshape(-1)) for c in range(C)])
    return median_error, _native.to_host(d_rep), _native.to_host(d_tr)


def plot_residuals(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints, calib_poses, max_points=10000,
                   marker_size=1, target_size=250, n_cols=3, inches_per_axis=5, hide_axes=True):
    """Reference signature and return values (viz.py:70-210): ``(fig, median_error, reprojections,
    transformed_reprojections)``; the numbers come from :func:`reprojection_residuals`."""
    median_error, reprojections, transformed = reprojection_residuals(all_calib_uvs, all_extrinsics, all_intrinsics,
                                                                      calib_objpoints, calib_poses)
    try:
        import matplotlib.pyplot as plt
    except ImportError as e:
        raise ImportError("plot_residuals draws with matplotlib, which is not installed; "
                          "reprojection_residuals(...) returns the numbers without it") from e
    obj = np.asarray(calib_objpoints, dtype=float)
    n_cameras = len(median_error)
    n_rows = int(np.ceil(n_cameras / n_cols))
    fig, axes = plt.subplots(n_rows, n_cols)
    axes = np.atleast_1d(axes)
    for cam in range(n_cameras):
        pts = transformed[cam].reshape(-1, 2)
        keep = np.nonzero(~np.isnan(pts).any(-1))[0]
        if len(keep) > max_points:
            keep = np.random.choice(keep, max_points, replace=False)
        ax = axes.flat[cam]
        ax.scatter(*obj[:, :2].T, c="k", s=target_size, marker="+", linewidth=0.5)
        ax.scatter(*pts[keep].T, c="r", s=marker_size, linewidth=0)
        ax.set_title(f"camera {cam} (median error={median_error[cam]:.2f})", fontsize=10)
        ax.set_aspect("equal")
        if len(keep):
            lo, hi = np.percentile(pts[keep], 1, axis=0), np.percentile(pts[keep], 99, axis=0)
            pad = 0.1 * (hi - lo)
            ax.set_xlim(lo[0] - pad[0], hi[0] + pad[0])
            ax.set_ylim(lo[1] - pad[1], hi[1] + pad[1])
        if hide_axes:
            ax.axis("off")
    for i in range(n_cameras, n_rows * n_cols):
        axes.flat[i].axis("off")
    aspect = np.ptp(obj[:, 1]) / np.ptp(obj[:, 0])
    fig.set_size_inches((n_cols * inches_per_axis, n_rows * inches_per_axis * aspect))
    return fig, median_error, reprojections, transformed
