"""Drop-in for ``multicam_calibration.geometry`` (reference geometry.py:8-433).

Same names, argument order, broadcasting and NaN conventions.  The batched
functions of the hot path (``project_points``, ``undistort_points``,
``triangulate``) run on the GPU through ``libmcba``; the small algebraic
helpers (a handful of 3x3 / 4x4 operations the reference calls once per camera
or frame) are host numpy, as SURVEY.md section 2 scopes them.
"""
import ctypes
from typing import NamedTuple, Optional

import numpy as np

from . import _native
from ._native import check

na = np.newaxis


# ----------------------------------------------------------------------------
# small host helpers (API surface)
# ----------------------------------------------------------------------------
def rodrigues(r):
    """Rotation vector (...,3) -> matrix (...,3,3) (geometry.py:8-35)."""
    r = np.asarray(r, dtype=float)
    theta = np.sqrt((r * r).sum(-1))
    k = r / np.where(theta == 0, 1.0, theta)[..., na]
    kx, ky, kz = k[..., 0], k[..., 1], k[..., 2]
    zero = np.zeros_like(kx)
    Kmat = np.stack([np.stack([zero, -kz, ky], -1),
                     np.stack([kz, zero, -kx], -1),
                     np.stack([-ky, kx, zero], -1)], -2)
    s = np.sin(theta)[..., na, na]
    c = (1 - np.cos(theta))[..., na, na]
    return s * Kmat + c * (Kmat @ Kmat) + np.eye(3)


def rodrigues_inv(R):
    """Rotation matrix (...,3,3) -> vector (...,3) (geometry.py:38-65)."""
    R = np.asarray(R, dtype=float)
    axis = np.stack([R[..., 2, 1] - R[..., 1, 2],
                     R[..., 0, 2] - R[..., 2, 0],
                     R[..., 1, 0] - R[..., 0, 1]], axis=-1)
    angle = np.arccos((np.trace(R, axis1=-2, axis2=-1) - 1) / 2)[..., na]
    norm = np.linalg.norm(axis, axis=-1, keepdims=True)
    norm = norm + (norm == 0)
    return axis * angle / norm


def get_transformation_matrix(t):
    """(...,6) -> (...,4,4) (geometry.py:155-175)."""
    t = np.asarray(t, dtype=float)
    T = np.zeros((*t.shape[:-1], 4, 4))
    T[..., :3, :3] = rodrigues(t[..., :3])
    T[..., :3, 3] = t[..., 3:]
    T[..., 3, 3] = 1
    return T


def get_transformation_vector(T):
    """(...,4,4) -> (...,6) (geometry.py:178-197)."""
    T = np.asarray(T, dtype=float)
    return np.concatenate([rodrigues_inv(T[..., :3, :3]), T[..., :3, 3]], axis=-1)


def euclidean_to_homogenous(x_euclidean):
    """Append a one (geometry.py:232-252)."""
    x = np.asarray(x_euclidean)
    return np.concatenate((x, np.ones((*x.shape[:-1], 1))), axis=-1)


def homogeneous_to_euclidean(x_homogenous):
    """Divide by the last coordinate (geometry.py:255-274)."""
    x = np.asarray(x_homogenous)
    return x[..., :-1] / x[..., -1:]


def apply_rigid_transform(transform, points):
    """Transform (6,) or (...,4,4) applied to points (...,3) (geometry.py:128-152)."""
    transform = np.asarray(transform, dtype=float)
    if transform.shape == (6,):
        transform = get_transformation_matrix(transform)
    hom = euclidean_to_homogenous(points)
    return np.matmul(transform, hom[..., na])[..., :3, 0]


def get_projection_matrix(extrinsics, intrinsics):
    """``P = K [R | t]`` (geometry.py:200-229)."""
    camera_matrix, _ = intrinsics
    return np.matmul(camera_matrix, get_transformation_matrix(np.asarray(extrinsics, dtype=float))[:3])


def rigid_transform_from_correspondences(source_points, target_points):
    """Kabsch fit, returns (6-vector, rmsd) (geometry.py:68-125)."""
    src = np.asarray(source_points, dtype=float).reshape(-1, 3)
    dst = np.asarray(target_points, dtype=float).reshape(-1, 3)
    mu_s, mu_d = src.mean(0), dst.mean(0)
    U, _, Vt = np.linalg.svd((src - mu_s).T @ (dst - mu_d))
    R = Vt.T @ U.T
    if np.linalg.det(R) < 0:
        Vt[-1, :] *= -1
        R = Vt.T @ U.T
    t = np.concatenate((rodrigues_inv(R), mu_d - R @ mu_s))
    moved = apply_rigid_transform(t, src)
    rmsd = np.sqrt(np.mean(np.sum((moved - dst) ** 2, axis=1)))
    return t, rmsd


# ----------------------------------------------------------------------------
# GPU-backed batched functions
# ----------------------------------------------------------------------------
def _device_ctx():
    torch = _native.require_cuda()
    return torch, _native.load(), torch.cuda.current_device()


def _h(a):
    return np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(ctypes.c_void_p)


def project_points(points, extrinsics, camera_matrix, dist_coefs=None):
    """Project (...,3) world points to (...,2) pixels (geometry.py:277-325)."""
    torch, lib, dev = _device_ctx()
    pts = np.ascontiguousarray(points, dtype=np.float64)
    lead = pts.shape[:-1]
    d_pts = _native.to_device(pts.reshape(-1, 3), dev)
    d_uv = torch.empty((d_pts.shape[0], 2), dtype=torch.float64, device=d_pts.device)
    ext = np.ascontiguousarray(extrinsics, dtype=np.float64)
    K = np.ascontiguousarray(camera_matrix, dtype=np.float64)
    dist = None if dist_coefs is None else np.ascontiguousarray(np.asarray(dist_coefs, dtype=np.float64)[:2])
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.mcba_project_points(dev, stream, ctypes.c_void_p(d_pts.data_ptr()), d_pts.shape[0],
                                  _h(ext), _h(K), None if dist is None else _h(dist),
                                  ctypes.c_void_p(d_uv.data_ptr())))
    return _native.to_host(d_uv).reshape(*lead, 2)


def project_points_multi(points, all_extrinsics, all_intrinsics, _device_points=None):
    """``np.stack([project_points(points, ext, K, dist) for ...])`` in one pass over the points
    (``mcba_project_points_multi``): (...,3) -> (C,...,2).  ``all_intrinsics`` is the reference's
    list of ``(camera_matrix, dist_coefs)``; every camera must either have distortion or not."""
    torch, lib, dev = _device_ctx()
    if _device_points is None:
        pts = np.ascontiguousarray(points, dtype=np.float64)
        lead = pts.shape[:-1]
        d_pts = _native.to_device(pts.reshape(-1, 3), dev)
    else:
        d_pts, lead = _device_points
    C = len(all_extrinsics)
    ext = np.ascontiguousarray(np.stack([np.asarray(e, dtype=np.float64) for e in all_extrinsics]))
    Ks = np.ascontiguousarray(np.stack([np.asarray(K, dtype=np.float64) for K, _ in all_intrinsics]))
    has = [d is not None for _, d in all_intrinsics]
    if any(has) != all(has):
        raise ValueError("project_points_multi: dist_coefs must be given for every camera or for none")
    dist = None
    if all(has):
        dist = np.ascontiguousarray(np.stack([np.asarray(d, dtype=np.float64).ravel()[:2] for _, d in all_intrinsics]))
    d_uv = torch.empty((C, d_pts.shape[0], 2), dtype=torch.float64, device=d_pts.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.mcba_project_points_multi(dev, stream, ctypes.c_void_p(d_pts.data_ptr()), d_pts.shape[0], C,
                                        _h(ext), _h(Ks), None if dist is None else _h(dist),
                                        ctypes.c_void_p(d_uv.data_ptr())))
    return _native.to_host(d_uv).reshape(C, *lead, 2)


def undistort_points(uvs, camera_matrix, dist_coefs):
    """NaN-aware ``cv2.undistortPoints(uv, K, dist, None, K)`` (geometry.py:328-358)."""
    torch, lib, dev = _device_ctx()
    uv = np.ascontiguousarray(uvs, dtype=np.float64)
    shape = uv.shape
    d_in = _native.to_device(uv.reshape(-1, 2), dev)
    d_out = torch.empty_like(d_in)
    dist = np.zeros(5)
    dc = np.asarray(dist_coefs, dtype=np.float64).ravel()[:5]
    dist[:dc.size] = dc
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.mcba_undistort_points(dev, stream, ctypes.c_void_p(d_in.data_ptr()), d_in.shape[0],
                                    _h(camera_matrix), _h(dist), ctypes.c_void_p(d_out.data_ptr())))
    return _native.to_host(d_out).reshape(shape)


def triangulate(all_uvs, all_extrinsics, all_intrinsics):
    """Robust all-pairs triangulation (geometry.py:361-433): list of C arrays
    (P,2) with NaN = missing -> (P,3), NaN where fewer than two views."""
    torch, lib, dev = _device_ctx()
    uv = np.ascontiguousarray(np.stack([np.asarray(u, dtype=np.float64) for u in all_uvs]))
    C, P, _ = uv.shape
    ext = np.ascontiguousarray(np.stack([np.asarray(e, dtype=np.float64) for e in all_extrinsics]))
    Ks = np.ascontiguousarray(np.stack([np.asarray(K, dtype=np.float64) for K, _ in all_intrinsics]))
    dists = np.zeros((C, 5))
    for c, (_, dc) in enumerate(all_intrinsics):
        dc = np.asarray(dc, dtype=np.float64).ravel()[:5]
        dists[c, :dc.size] = dc
    d_uv = _native.to_device(uv, dev)
    d_out = torch.empty((P, 3), dtype=torch.float64, device=d_uv.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.mcba_triangulate(dev, stream, ctypes.c_void_p(d_uv.data_ptr()), C, P, _h(ext), _h(Ks),
                               _h(dists), ctypes.c_void_p(d_out.data_ptr())))
    return _native.to_host(d_out)


class RefinedPoints(NamedTuple):
    """Result of :func:`refine_points`; per-point arrays over the P points."""
    points: np.ndarray        # (P, 3) refined points
    cost: np.ndarray          # (P,) 0.5 sum rho at the result
    rms: np.ndarray           # (P,) reprojection RMS in px over the point's finite scalars
    n_views: np.ndarray       # (P,) int, seen views
    status: np.ndarray        # (P,) int8: 1 gtol, 2 ftol, 3 xtol, 4 ftol + xtol, 0 max_iter, -1, -2
    iterations: np.ndarray    # (P,) int16, trial steps
    covariance: Optional[np.ndarray]    # (P, 3, 3) or None
    view_errors: Optional[np.ndarray]   # (C, P) px, NaN where unseen, or None


def _real_array(name, a, who="refine_points"):
    a = np.asarray(a)
    if not (np.issubdtype(a.dtype, np.floating) or np.issubdtype(a.dtype, np.integer)):
        raise ValueError(f"{who}: {name} must be a real array, got dtype {a.dtype}")
    return np.ascontiguousarray(a, dtype=np.float64)


def _positive(name, v, who="refine_points"):
    if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)) \
            or not (0 < float(v) < np.inf):
        raise ValueError(f"{who}: {name} must be a finite number > 0, got {v!r}")
    return float(v)


def _loss_args(loss, f_scale, sigma, who="refine_points"):
    """Validated (loss code, f_scale, sigma) of refine_points and point_covariance."""
    if callable(loss) or not isinstance(loss, str) or loss not in _native.REFINE_LOSSES:
        raise ValueError(f"{who}: loss must be one of {sorted(_native.REFINE_LOSSES)}, got {loss!r}")
    return _native.REFINE_LOSSES[loss], _positive("f_scale", f_scale, who), _positive("sigma", sigma, who)


def _rig_args(all_uvs, all_extrinsics, all_intrinsics, who="refine_points"):
    """Validated (uv (C,P,2), ext (C,6), Ks (C,3,3), dists (C,5)) of refine_points and point_covariance."""
    if isinstance(all_uvs, np.ndarray):
        uv = _real_array("all_uvs", all_uvs, who)
    else:
        uv = np.stack([_real_array("all_uvs", u, who) for u in all_uvs]) if len(all_uvs) else np.zeros((0, 0, 2))
    if uv.ndim != 3 or uv.shape[2] != 2:
        raise ValueError(f"{who}: all_uvs must be C arrays (P, 2) or one (C, P, 2) array, got {uv.shape}")
    C, P, _ = uv.shape
    if not 1 <= C <= 32:
        raise ValueError(f"{who}: 1 <= n_cameras <= 32, got {C}")
    ext = _real_array("all_extrinsics", all_extrinsics, who)
    if ext.shape != (C, 6):
        raise ValueError(f"{who}: all_extrinsics must be ({C}, 6), got {ext.shape}")
    if len(all_intrinsics) != C:
        raise ValueError(f"{who}: all_intrinsics must have {C} entries, got {len(all_intrinsics)}")
    Ks = np.empty((C, 3, 3))
    dists = np.zeros((C, 5))
    for c, intr in enumerate(all_intrinsics):
        if len(intr) != 2:
            raise ValueError(f"{who}: all_intrinsics entries must be (camera_matrix, dist_coefs)")
        K = _real_array("camera_matrix", intr[0], who)
        dc = _real_array("dist_coefs", intr[1], who).ravel()
        if K.shape != (3, 3) or not 2 <= dc.size:
            raise ValueError(f"{who}: camera {c}: camera_matrix must be (3, 3) and dist_coefs hold at "
                             f"least k1, k2, got {K.shape} and {dc.size} coefficients")
        Ks[c] = K
        dists[c, :min(dc.size, 5)] = dc[:5]
    return uv, ext, Ks, dists


def refine_points(all_uvs, all_extrinsics, all_intrinsics, points=None, *, loss="linear", f_scale=1.0, sigma=1.0,
                  max_iter=50, ftol=1e-12, xtol=1e-12, gtol=1e-10, covariance=True, view_errors=False):
    """Least-squares refinement of triangulated points on the device (``mcba_refine_points``).

    Per point, Levenberg-Marquardt on ``0.5 sum_views sum_{u,v} f_scale^2 rho((r / f_scale)^2)`` with
    ``r = observed - project_points(X, ext_c, K_c, dist_c)``: the model of ``project_points`` and the bundle
    adjustment (full K with skew, k1 and k2 only).  ``loss`` is one of scipy's ``linear``, ``soft_l1``,
    ``huber``, ``cauchy``, ``arctan`` with scipy's formulas and ``f_scale``; the ftol / xtol / gtol tests are
    scipy's (``least_squares``), applied per point.

    Inputs are ``triangulate``'s: ``all_uvs`` a list of C ``(P, 2)`` arrays or a ``(C, P, 2)`` array, NaN
    marking a missing view; a view whose pixel does not undistort to a finite point (NaN, +-inf, an
    overflowing value) is unseen, as in ``triangulate``.  ``points=None`` starts from ``triangulate``'s
    result, computed in the same device call; a given ``(P, 3)`` start is used as is.  The start's
    triangulation undistorts with all five coefficients of ``dist`` while the objective uses k1, k2 only: with
    non-zero p1, p2 or k3 the two models disagree and the refined point minimises the two-coefficient one.

    A view behind a camera at the start still enters the objective as ``project_points`` evaluates it
    (through the camera centre).  Status per point: 1 gtol, 2 ftol, 3 xtol, 4 ftol and xtol, 0 ``max_iter``
    trial steps reached (the point is refined in all of these); -1 fewer than two seen views (NaN point, as
    ``triangulate`` gives); -2 a non-finite start or cost at the start (a view on a camera's Z = 0 plane), or
    damping beyond its bound: the start is returned unchanged.  ``covariance`` is
    ``sigma^2 inv(J~^T J~)`` at the result with ``J~`` scaled for the robust loss as scipy's ``result.jac``.
    """
    loss_code, f_scale, sigma = _loss_args(loss, f_scale, sigma)
    if isinstance(max_iter, (bool, np.bool_)) or not isinstance(max_iter, (int, np.integer)) \
            or not 1 <= max_iter <= 32767:
        raise ValueError(f"refine_points: max_iter must be an integer in [1, 32767], got {max_iter!r}")
    tols = {}
    for name, v in (("ftol", ftol), ("xtol", xtol), ("gtol", gtol)):
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)) \
                or not (0 <= float(v) < np.inf):
            raise ValueError(f"refine_points: {name} must be a finite number >= 0, got {v!r}")
        tols[name] = float(v)
    uv, ext, Ks, dists = _rig_args(all_uvs, all_extrinsics, all_intrinsics)
    C, P, _ = uv.shape
    init = None
    if points is not None:
        init = _real_array("points", points)
        if init.shape != (P, 3):
            raise ValueError(f"refine_points: points must be ({P}, 3), got {init.shape}")

    torch, lib, dev = _device_ctx()
    d_uv = _native.to_device(uv, dev)
    d_init = None if init is None else _native.to_device(init, dev)
    f64 = dict(dtype=torch.float64, device=d_uv.device)
    d_pts = torch.empty((P, 3), **f64)
    d_cost = torch.empty((P,), **f64)
    d_rms = torch.empty((P,), **f64)
    d_status = torch.empty((P,), dtype=torch.int8, device=d_uv.device)
    d_iters = torch.empty((P,), dtype=torch.int16, device=d_uv.device)
    d_nv = torch.empty((P,), dtype=torch.int8, device=d_uv.device)
    d_cov = torch.empty((P, 6), **f64) if covariance else None
    d_verr = torch.empty((C, P), **f64) if view_errors else None
    opt = _native.RefineOptions(loss=loss_code, f_scale=f_scale, sigma=sigma,
                                max_iter=int(max_iter), flags=0, **tols)

    def ptr(t):
        return None if t is None else ctypes.c_void_p(t.data_ptr())
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.mcba_refine_points(dev, stream, ptr(d_uv), C, P, _h(ext), _h(Ks), _h(dists), ptr(d_init),
                                 ctypes.byref(opt), ptr(d_pts), ptr(d_cost), ptr(d_rms), ptr(d_status),
                                 ptr(d_iters), ptr(d_cov), ptr(d_verr), ptr(d_nv)))
    cov = None
    if covariance:
        cov = _native.to_host(d_cov)[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(P, 3, 3)
    return RefinedPoints(_native.to_host(d_pts), _native.to_host(d_cost), _native.to_host(d_rms),
                         _native.to_host(d_nv).astype(np.int64), _native.to_host(d_status),
                         _native.to_host(d_iters), cov, _native.to_host(d_verr) if view_errors else None)
