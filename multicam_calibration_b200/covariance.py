"""How well a calibration is determined: the covariance of the camera parameters and board poses.

``scipy.optimize.least_squares`` returns ``result.jac``, the robust-scaled Jacobian J~ whose J~^T J~ is the
Gauss-Newton matrix, and its users get standard errors from ``inv(J~^T J~) * 2 cost / (m - n)``.  The B200
engine never materialises J~ (16.8 M x 300 k at 6 cameras x 50,000 frames); :func:`calibration_covariance`
computes the same quantity from the reduced camera system and the per-frame factors of one device evaluation
(``mcba_covariance``).
"""
import ctypes
from dataclasses import dataclass
from typing import Optional

import numpy as np


@dataclass
class CalibrationCovariance:
    """``camera`` (12C, 12C) in the order of ``serialize_params`` (per camera fx fy cx cy k1 k2 rvec tvec);
    ``camera_std`` (C, 12); ``poses`` (F, 6, 6) ``[rvec | tvec]`` and ``pose_std`` (F, 6), or None;
    ``sigma2`` the residual variance used (px^2), ``dof`` = m - p, ``n_residuals`` = m, ``cost`` at the
    parameters."""
    camera: np.ndarray
    camera_std: np.ndarray
    poses: Optional[np.ndarray]
    pose_std: Optional[np.ndarray]
    sigma2: float
    dof: float
    n_residuals: int
    cost: float


def _std(diag):
    with np.errstate(invalid="ignore"):
        return np.sqrt(diag)


def calibration_covariance(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints, calib_poses,
                           reference_camera=0, loss="soft_l1", f_scale=1.0, sigma=None, poses=True, fixed=None):
    """Covariance of the calibration ``(all_extrinsics, all_intrinsics, calib_poses)``.

    The arguments are ordered like ``bundle_adjust``'s and take its outputs directly:
    ``calibration_covariance(uvs[:, use_frames], ext, intr, objpoints, poses)``.

    The Gauss-Newton matrix is J~^T J~ with J~ the residual Jacobian row-scaled exactly as
    ``least_squares(loss=loss, f_scale=f_scale)`` scales it (scipy's ``result.jac``).  The six extrinsic
    parameters of ``reference_camera`` are held fixed (the gauge): the result is the uncertainty of every
    other parameter in that camera's frame, and the reference camera's extrinsic rows and columns are 0.
    Cameras and frames without any finite observation are NaN.  The residual variance is ``sigma**2`` when
    ``sigma`` (px) is given, else ``2 cost / (m - p)``: m finite residual scalars, p = 12 observed cameras
    + 6 observed frames - 6 (with a mask: the free non-gauge parameters of the observed cameras + 6 observed frames).

    ``fixed`` (C, 12) bool, ``serialize_params`` order: parameters held fixed in the solve (``bundle_adjust``'s
    ``fixed``).  The result is conditional on them: their rows and columns are exactly 0, also for a camera
    without observations, and p counts the free parameters only.  A mask that holds all six extrinsics of some
    camera fixes the gauge itself: ``reference_camera`` must then be None or such a camera.  Otherwise the
    reference camera is the gauge, and the mask may hold no extrinsic entry.

    For ``loss='linear'`` this is the asymptotic covariance of the least-squares estimate.  For ``soft_l1``
    it is scipy's usual recipe applied to the robust-scaled Jacobian, not an M-estimator sandwich
    covariance.

    Raises ``ValueError`` for bad arguments or residuals that are not finite at the parameters, and
    ``numpy.linalg.LinAlgError`` when a frame's pose or the gauge-fixed camera system is singular (too few
    or collinear corners, a camera that sees too little).  Runs on the current CUDA device only, also when
    ``torch.distributed`` is initialised.
    """
    from .bundle_adjustment import _problem_for, serialize_params
    from .engine import check_fixed

    uvs = all_calib_uvs if hasattr(all_calib_uvs, "is_cuda") else np.asarray(all_calib_uvs, dtype=np.float64)
    if uvs.ndim != 4 or uvs.shape[-1] != 2:
        raise ValueError("all_calib_uvs must be (C, F, N, 2)")
    C, F = int(uvs.shape[0]), int(uvs.shape[1])
    if reference_camera is not None:
        if isinstance(reference_camera, (bool, np.bool_)) or not isinstance(reference_camera, (int, np.integer)):
            raise ValueError("reference_camera must be None or an integer camera index")
        if not 0 <= int(reference_camera) < C:
            raise ValueError(f"reference_camera {reference_camera} is not in [0, {C})")
        reference_camera = int(reference_camera)
    check_fixed(fixed, C)
    if loss not in ("linear", "soft_l1"):
        raise ValueError("loss must be 'linear' or 'soft_l1'")
    if not (np.isfinite(f_scale) and f_scale > 0):
        raise ValueError("f_scale must be finite and positive")
    if sigma is not None and not (np.isfinite(sigma) and sigma > 0):
        raise ValueError("sigma must be None or a finite positive noise level in pixels")
    if len(all_extrinsics) != C or len(all_intrinsics) != C:
        raise ValueError(f"all_extrinsics and all_intrinsics must have one entry per camera ({C})")
    calib_poses = np.asarray(calib_poses, dtype=np.float64)
    if calib_poses.shape != (F, 6):
        raise ValueError(f"calib_poses must be ({F}, 6)")
    x = serialize_params(all_extrinsics, all_intrinsics, calib_poses)
    if not np.isfinite(x).all():
        raise ValueError("Residuals are not finite at the given parameters (non-finite parameters).")

    prob = _problem_for(uvs, calib_objpoints)
    cam, pose, info = prob.covariance(x, reference_camera=reference_camera, loss=loss, f_scale=float(f_scale),
                                      sigma=sigma, poses=poses, fixed=fixed)
    return CalibrationCovariance(
        camera=cam, camera_std=_std(np.diag(cam)).reshape(C, 12),
        poses=pose, pose_std=None if pose is None else _std(np.einsum("fii->fi", pose)),
        sigma2=info["sigma2"], dof=info["dof"], n_residuals=info["n_residuals"], cost=info["cost"])


@dataclass
class PointCovariance:
    """``total = measurement + calibration`` (P, 3, 3) each: the uncertainty of refined points from the pixel
    noise of their own observations and from the calibration; ``sensitivity`` (P, 3, 12C) ``dX/dtheta`` in the
    order of ``serialize_params``, zero for unseen cameras, or None."""
    total: np.ndarray
    measurement: np.ndarray
    calibration: np.ndarray
    sensitivity: Optional[np.ndarray]


def _camera_covariance(cov, C):
    a = cov.camera if isinstance(cov, CalibrationCovariance) else cov
    a = np.asarray(a)
    if not (np.issubdtype(a.dtype, np.floating) or np.issubdtype(a.dtype, np.integer)):
        raise ValueError(f"point_covariance: cov must be a CalibrationCovariance or a real array, got dtype {a.dtype}")
    a = np.ascontiguousarray(a, dtype=np.float64)
    n = 12 * C
    if a.shape != (n, n):
        raise ValueError(f"point_covariance: the camera covariance must be ({n}, {n}) for {C} cameras, got {a.shape}")
    if np.isinf(a).any():
        raise ValueError("point_covariance: the camera covariance must hold finite numbers or NaN")
    nan = np.isnan(a)
    if not np.array_equal(nan, nan.T):
        raise ValueError("point_covariance: the camera covariance is not symmetric (NaN pattern)")
    d = np.diag(a)
    if (d < 0).any():
        raise ValueError("point_covariance: the camera covariance has a negative diagonal entry")
    with np.errstate(invalid="ignore"):
        scale = np.sqrt(np.outer(d, d))
        asym = np.abs(a - a.T) > 1e-9 * scale + 1e-300
    if asym.any():
        raise ValueError("point_covariance: the camera covariance is not symmetric")
    return a


def point_covariance(all_uvs, all_extrinsics, all_intrinsics, points, cov, loss="linear", f_scale=1.0, sigma=1.0,
                     sensitivity=False):
    """Covariance of refined points including the calibration's uncertainty (``mcba_point_covariance``).

    ``all_uvs``, ``all_extrinsics``, ``all_intrinsics``, ``loss``, ``f_scale`` and ``sigma`` are taken as
    ``refine_points`` takes them; ``points`` (P, 3) are the points to evaluate, normally ``refine_points(...).points``;
    ``cov`` is a :class:`CalibrationCovariance` or its (12C, 12C) ``camera`` array.  Per point X over its seen
    views, with J~ scaled as ``refine_points``' covariance scales it:

    * ``measurement = sigma^2 inv(J~_X^T J~_X)``, bit-identical to ``refine_points(...).covariance`` at X;
    * ``S_c = -inv(J~_X^T J~_X) J~_X^T J~_c`` (3 x 12), the Gauss-Newton sensitivity dX/dtheta_c of the minimiser
      to camera c's parameters;
    * ``calibration = sum_{c,d seen} S_c cov[c,d] S_d^T`` and ``total = measurement + calibration`` (the keypoint's
      pixel noise is independent of the calibration data).

    The calibration part is in the gauge of ``cov``: the reference camera's frame, or that of the camera pinned by
    ``fixed=``.  Held parameters have zero rows and contribute nothing; unseen cameras do not enter.  A point
    with fewer than two seen views, a non-finite X or a non-positive-definite J~_X^T J~_X is NaN in every output;
    where a seen pair of cameras has NaN in its block of ``cov`` (a camera without observations in the
    calibration), ``calibration`` and ``total`` are NaN.  For robust losses this is the Gauss-Newton recipe of
    ``refine_points``' covariance, not a sandwich estimator.

    ``sensitivity=True`` also returns S as (P, 3, 12C), zero for unseen cameras: ``S_i cov S_j^T`` is the
    cross-covariance of points i and j (e.g. for the uncertainty of a distance between two keypoints).  It is
    8 * 36 C bytes per point (1.7 GB at 1 M points and 6 cameras).
    """
    from . import _native
    from .geometry import _device_ctx, _h, _loss_args, _real_array, _rig_args, check
    who = "point_covariance"
    loss_code, f_scale, sigma = _loss_args(loss, f_scale, sigma, who)
    uv, ext, Ks, dists = _rig_args(all_uvs, all_extrinsics, all_intrinsics, who)
    C, P, _ = uv.shape
    X = _real_array("points", points, who)
    if X.shape != (P, 3):
        raise ValueError(f"{who}: points must be ({P}, 3), got {X.shape}")
    cam = _camera_covariance(cov, C)

    torch, lib, dev = _device_ctx()
    d_uv = _native.to_device(uv, dev)
    d_X = _native.to_device(X, dev)
    f64 = dict(dtype=torch.float64, device=d_uv.device)
    d_meas = torch.empty((P, 6), **f64)
    d_cal = torch.empty((P, 6), **f64)
    d_sens = torch.empty((P, 3, 12 * C), **f64) if sensitivity else None

    def ptr(t):
        return None if t is None or t.numel() == 0 else ctypes.c_void_p(t.data_ptr())
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.mcba_point_covariance(dev, stream, ptr(d_uv), C, P, _h(ext), _h(Ks), _h(dists), ptr(d_X), _h(cam),
                                    loss_code, f_scale, sigma, ptr(d_meas), ptr(d_cal), ptr(d_sens)))
    full = [0, 1, 2, 1, 3, 4, 2, 4, 5]
    meas = _native.to_host(d_meas)[:, full].reshape(P, 3, 3)
    cal = _native.to_host(d_cal)[:, full].reshape(P, 3, 3)
    return PointCovariance(total=meas + cal, measurement=meas, calibration=cal,
                           sensitivity=_native.to_host(d_sens) if sensitivity else None)
