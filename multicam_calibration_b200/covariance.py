"""How well a calibration is determined: the covariance of the camera parameters and board poses.

``scipy.optimize.least_squares`` returns ``result.jac``, the robust-scaled Jacobian J~ whose J~^T J~ is the
Gauss-Newton matrix, and its users get standard errors from ``inv(J~^T J~) * 2 cost / (m - n)``.  The B200
engine never materialises J~ (16.8 M x 300 k at 6 cameras x 50,000 frames); :func:`calibration_covariance`
computes the same quantity from the reduced camera system and the per-frame factors of one device evaluation
(``mcba_covariance``).
"""
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
