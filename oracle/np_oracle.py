"""numpy restatement of the reference's bundle-adjustment hot path (CPU oracle).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  Every function cites
the reference lines (relative to ``/root/reference/multicam_calibration/``) or
the scipy 1.18.1 lines (relative to ``site-packages/scipy/``) it restates.
The restatement is validated against the unmodified reference in the build
container by ``tests/golden/make_golden.py`` and on every test run against the
committed fixtures it produced (``tests/test_oracle_golden.py``).

Parameter vector (``bundle_adjustment.py:128-157``): per camera
``[fx, fy, cx, cy, k1, k2, rx, ry, rz, tx, ty, tz]`` (12), then per frame
``[rho_x, rho_y, rho_z, tau_x, tau_y, tau_z]`` (6).
"""
import itertools

import numpy as np

EPS = np.finfo(float).eps
CAM_BLOCK = 12
POSE_BLOCK = 6


# --------------------------------------------------------------------------
# geometry (geometry.py)
# --------------------------------------------------------------------------
def skew(v):
    """[v]x for v of shape (..., 3)."""
    v = np.asarray(v, dtype=float)
    S = np.zeros(v.shape[:-1] + (3, 3))
    S[..., 0, 1], S[..., 0, 2] = -v[..., 2], v[..., 1]
    S[..., 1, 0], S[..., 1, 2] = v[..., 2], -v[..., 0]
    S[..., 2, 0], S[..., 2, 1] = -v[..., 1], v[..., 0]
    return S


def rodrigues(r):
    """Rotation vector -> matrix, geometry.py:8-35.

    ``R = I + sin(th) K + (1 - cos(th)) K^2`` with ``K = [r]x / th``; ``th == 0``
    divides by one instead (geometry.py:30), giving ``R = I``.
    """
    r = np.asarray(r, dtype=float)
    th = np.sqrt(np.sum(r * r, axis=-1))[..., None, None]
    K = skew(r) / np.where(th == 0, 1.0, th)
    R = np.sin(th) * K + (1.0 - np.cos(th)) * (K @ K)
    return R + np.eye(3)


def rodrigues_inv(R):
    """Rotation matrix -> vector, geometry.py:38-65."""
    R = np.asarray(R, dtype=float)
    w = np.stack([R[..., 2, 1] - R[..., 1, 2],
                  R[..., 0, 2] - R[..., 2, 0],
                  R[..., 1, 0] - R[..., 0, 1]], axis=-1)
    th = np.arccos((np.trace(R, axis1=-2, axis2=-1) - 1.0) / 2.0)[..., None]
    nw = np.linalg.norm(w, axis=-1, keepdims=True)
    nw = nw + (nw == 0)
    return w * th / nw


def transformation_matrix(t):
    """(...,6) -> (...,4,4) ``[R t; 0 1]``, geometry.py:155-175."""
    t = np.asarray(t, dtype=float)
    T = np.zeros(t.shape[:-1] + (4, 4))
    T[..., :3, :3] = rodrigues(t[..., :3])
    T[..., :3, 3] = t[..., 3:]
    T[..., 3, 3] = 1.0
    return T


def transformation_vector(T):
    """Inverse of :func:`transformation_matrix`, geometry.py:178-197."""
    return np.concatenate([rodrigues_inv(T[..., :3, :3]), T[..., :3, 3]], axis=-1)


def apply_rigid_transform(transform, points):
    """geometry.py:128-152 -- transform is (6,) or (...,4,4)."""
    transform = np.asarray(transform, dtype=float)
    if transform.shape == (6,):
        transform = transformation_matrix(transform)
    points = np.asarray(points, dtype=float)
    hom = np.concatenate([points, np.ones(points.shape[:-1] + (1,))], axis=-1)
    return np.matmul(transform, hom[..., None])[..., :3, 0]


def project_points(points, extrinsics, camera_matrix, dist_coefs=None):
    """Pinhole + (k1, k2) radial projection, geometry.py:277-325."""
    Xc = apply_rigid_transform(np.asarray(extrinsics, dtype=float), points)
    if dist_coefs is not None:
        k1, k2 = dist_coefs[0], dist_coefs[1]
        xy = Xc[..., :2] / Xc[..., 2:]
        r2 = np.sum(xy * xy, axis=-1)
        d = 1 + k1 * r2 + k2 * r2 ** 2
        Xc = Xc * np.stack([d, d, np.ones_like(d)], axis=-1)
    uvw = np.matmul(np.asarray(camera_matrix, dtype=float), Xc[..., None])[..., 0]
    return uvw[..., :2] / uvw[..., 2:]


def projection_matrix(extrinsics, intrinsics):
    """``P = K [R | t]``, geometry.py:200-229."""
    return np.asarray(intrinsics[0], dtype=float) @ transformation_matrix(extrinsics)[:3]


def undistort_points(uvs, camera_matrix, dist_coefs, n_iter=5):
    """geometry.py:328-358 + OpenCV ``undistortPoints(uv, K, dist5, None, K)``.

    OpenCV is an un-vendored binary dependency; its documented algorithm is a
    FIXED 5-iteration fixed-point inversion of the full (k1,k2,p1,p2,k3) model
    (SURVEY.md Appendix B; validated against cv2 4.13.0 by make_golden.py).
    Rows containing a NaN stay NaN (geometry.py:350-356).
    """
    uvs = np.asarray(uvs, dtype=float)
    K = np.asarray(camera_matrix, dtype=float)
    dc = np.zeros(5)
    dc[:len(dist_coefs)] = np.asarray(dist_coefs, dtype=float)[:5]
    k1, k2, p1, p2, k3 = dc
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    x0 = (uvs[..., 0] - cx) / fx
    y0 = (uvs[..., 1] - cy) / fy
    x, y = x0.copy(), y0.copy()
    with np.errstate(invalid="ignore"):
        for _ in range(n_iter):
            r2 = x * x + y * y
            icd = 1.0 / (1.0 + ((k3 * r2 + k2) * r2 + k1) * r2)
            dx = 2 * p1 * x * y + p2 * (r2 + 2 * x * x)
            dy = p1 * (r2 + 2 * y * y) + 2 * p2 * x * y
            x = (x0 - dx) * icd
            y = (y0 - dy) * icd
    # new camera matrix P = K applied in full (skew included); the input
    # normalisation above ignores skew, exactly as OpenCV does
    out = np.stack([x * fx + y * K[0, 1] + cx, y * fy + cy], axis=-1)
    out[np.isnan(uvs).any(-1)] = np.nan
    return out


def triangulate_pair(Pi, Pj, uvi, uvj):
    """Homogeneous DLT of ``cv2.triangulatePoints`` (geometry.py:416-422).

    Per point the 4x4 system ``[u P[2] - P[0]; v P[2] - P[1]]`` for both views;
    the solution is the right singular vector of the smallest singular value,
    de-homogenised (geometry.py:255-274).
    """
    A = np.stack([uvi[:, 0, None] * Pi[2] - Pi[0],
                  uvi[:, 1, None] * Pi[2] - Pi[1],
                  uvj[:, 0, None] * Pj[2] - Pj[0],
                  uvj[:, 1, None] * Pj[2] - Pj[1]], axis=1)
    X = np.linalg.svd(A)[2][:, -1, :]
    return X[:, :3] / X[:, 3:]


def triangulate(all_uvs, all_extrinsics, all_intrinsics):
    """All-pairs DLT + per-coordinate nanmedian, geometry.py:361-433."""
    C = len(all_extrinsics)
    P = all_uvs[0].shape[0]
    und = [undistort_points(uv, K, dc) for uv, (K, dc) in zip(all_uvs, all_intrinsics)]
    Ps = [projection_matrix(e, i) for e, i in zip(all_extrinsics, all_intrinsics)]
    pair_pts = []
    for i, j in itertools.combinations(range(C), 2):
        pts = np.full((P, 3), np.nan)
        ok = ~(np.isnan(und[i]).any(-1) | np.isnan(und[j]).any(-1))
        if ok.any():
            pts[ok] = triangulate_pair(Ps[i], Ps[j], und[i][ok], und[j][ok])
        pair_pts.append(pts)
    pair_pts = np.stack(pair_pts)                      # (pairs, P, 3)
    out = np.full((P, 3), np.nan)
    some = ~np.isnan(pair_pts).all(axis=(0, 2))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", category=RuntimeWarning)
        out[some] = np.nanmedian(pair_pts[:, some], axis=0)
    return out


# --------------------------------------------------------------------------
# bundle_adjustment.py
# --------------------------------------------------------------------------
def embed_calib_objpoints(calib_objpoints, calib_poses):
    """(N,3),(F,6) -> (F,N,3) world points, bundle_adjustment.py:10-30."""
    T = transformation_matrix(calib_poses)[:, None]
    obj = np.asarray(calib_objpoints, dtype=float)
    hom = np.concatenate([obj, np.ones((len(obj), 1))], axis=-1)[None, :, :, None]
    return (T @ hom)[..., :3, 0]


def predict_calib_uvs(all_extrinsics, all_intrinsics, calib_objpoints, calib_poses):
    """(C,F,N,2) predictions, bundle_adjustment.py:33-63."""
    world = embed_calib_objpoints(calib_objpoints, calib_poses)
    return np.stack([project_points(world, e, K, dc)
                     for e, (K, dc) in zip(all_extrinsics, all_intrinsics)])


def serialize_params(all_extrinsics, all_intrinsics, calib_poses):
    """bundle_adjustment.py:128-157."""
    rows = []
    for ext, (K, dc) in zip(all_extrinsics, all_intrinsics):
        rows.append(np.r_[K[0, 0], K[1, 1], K[0, 2], K[1, 2], dc[0], dc[1], ext])
    rows.append(np.asarray(calib_poses, dtype=float).ravel())
    return np.concatenate(rows)


def deserialize_params(x, n_cameras):
    """bundle_adjustment.py:160-192."""
    cam = np.asarray(x[:CAM_BLOCK * n_cameras]).reshape(n_cameras, CAM_BLOCK)
    intr = []
    for p in cam:
        K = np.eye(3)
        K[0, 0], K[1, 1], K[0, 2], K[1, 2] = p[:4]
        intr.append((K, np.r_[p[4:6], 0.0, 0.0, 0.0]))
    return cam[:, 6:].copy(), intr, np.asarray(x[CAM_BLOCK * n_cameras:]).reshape(-1, POSE_BLOCK)


def residuals(params, all_calib_uvs, calib_objpoints):
    """observed - predicted, NaN entries removed element-wise in C order,
    bundle_adjustment.py:66-98."""
    ext, intr, poses = deserialize_params(params, all_calib_uvs.shape[0])
    pred = predict_calib_uvs(ext, intr, calib_objpoints, poses)
    return (all_calib_uvs - pred)[~np.isnan(all_calib_uvs)]


def sparsity_pattern(all_calib_uvs):
    """Same pattern as bundle_adjustment.py:101-125 (18 ones per row), built as
    CSR instead of a Python-list lil_matrix."""
    from scipy.sparse import csr_matrix
    C, F, N, _ = all_calib_uvs.shape
    mask = ~np.isnan(all_calib_uvs)
    cam_ix = np.broadcast_to(np.arange(C)[:, None, None, None], mask.shape)[mask]
    frm_ix = np.broadcast_to(np.arange(F)[None, :, None, None], mask.shape)[mask]
    m = cam_ix.size
    cols = np.concatenate([cam_ix[:, None] * CAM_BLOCK + np.arange(CAM_BLOCK),
                           C * CAM_BLOCK + frm_ix[:, None] * POSE_BLOCK + np.arange(POSE_BLOCK)],
                          axis=1)
    indptr = np.arange(m + 1) * 18
    return csr_matrix((np.ones(m * 18, dtype=int), cols.ravel(), indptr),
                      shape=(m, C * CAM_BLOCK + F * POSE_BLOCK))


def select_frames(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints,
                  calib_poses, n_frames=10000, outlier_threshold=None, verbose=True):
    """Frame eligibility, outlier filter and sub-sampling,
    bundle_adjustment.py:265-296 (consumes the global numpy RNG like :296)."""
    import warnings
    use = np.nonzero((~np.isnan(all_calib_uvs).any((-1, -2))).sum(0) > 1)[0]
    pred = predict_calib_uvs(all_extrinsics, all_intrinsics, calib_objpoints, calib_poses[use])
    err = np.linalg.norm(all_calib_uvs[:, use] - pred, axis=-1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", category=RuntimeWarning)
        worst = np.nanmax(np.nanmean(err, axis=-1), axis=0)
    if outlier_threshold is None:
        outlier_threshold = 5 * np.nanmedian(err)
    exclude = np.nan_to_num(worst) > outlier_threshold
    use = use[~exclude]
    if verbose:
        print(f"Excluding {int(exclude.sum())} out of {len(use)} frames "
              f"based on an outlier threshold of {outlier_threshold}")
    if not (n_frames is None or n_frames > len(use)):
        use = np.random.choice(use, n_frames, replace=False)
    return use, outlier_threshold


def bundle_adjust(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints,
                  calib_poses, n_frames=10000, outlier_threshold=None, **opt_kwargs):
    """The reference CPU path end to end, bundle_adjustment.py:195-327:
    scipy ``least_squares`` (trf, soft_l1, x_scale='jac', ftol=1e-4) on
    :func:`residuals` with the finite-difference sparsity pattern."""
    from scipy.optimize import least_squares
    C = all_calib_uvs.shape[0]
    kw = dict(verbose=2, x_scale="jac", ftol=1e-4, method="trf", loss="soft_l1")
    kw.update(opt_kwargs)
    use, _ = select_frames(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints,
                           calib_poses, n_frames, outlier_threshold)
    uv = all_calib_uvs[:, use]
    if "jac" not in kw or kw["jac"] in ("2-point", "3-point"):
        kw["jac_sparsity"] = sparsity_pattern(uv)
    x0 = serialize_params(all_extrinsics, all_intrinsics, calib_poses[use])
    result = least_squares(residuals, x0, args=(uv, calib_objpoints), **kw)
    ext, intr, poses = deserialize_params(result.x, C)
    return ext, intr, poses, use, result


# --------------------------------------------------------------------------
# analytic Jacobian (SURVEY.md Appendix A; the formulae the CUDA path must match)
# --------------------------------------------------------------------------
def so3_right_jacobian(r):
    """``J_r(r) = I - (1-cos th)/th^2 [r]x + (th - sin th)/th^3 [r]x^2``."""
    r = np.asarray(r, dtype=float)
    th2 = np.sum(r * r, axis=-1)[..., None, None]
    th = np.sqrt(th2)
    small = th < 1e-4
    ths = np.where(small, 1.0, th)
    a = np.where(small, 0.5 - th2 / 24.0, (1 - np.cos(ths)) / ths ** 2)
    b = np.where(small, 1.0 / 6.0 - th2 / 120.0, (ths - np.sin(ths)) / ths ** 3)
    S = skew(r)
    return np.eye(3) - a * S + b * (S @ S)


def rotated_point_jacobian(r, p):
    """``d(R(r) p)/dr = -R(r) [p]x J_r(r)`` for r (...,3), p (...,3)."""
    return -rodrigues(r) @ skew(p) @ so3_right_jacobian(r)


def jacobian_blocks(params, n_cameras, calib_objpoints):
    """Per-(c,f,n) Jacobian of the PREDICTION (residual Jacobian is its negative).

    Returns ``Jc (C,F,N,2,12)`` w.r.t. camera c's 12 parameters and
    ``Jp (C,F,N,2,6)`` w.r.t. frame f's pose, plus predictions ``(C,F,N,2)``.
    """
    C = n_cameras
    cam = np.asarray(params[:CAM_BLOCK * C]).reshape(C, CAM_BLOCK)
    poses = np.asarray(params[CAM_BLOCK * C:]).reshape(-1, POSE_BLOCK)
    F = len(poses)
    obj = np.asarray(calib_objpoints, dtype=float)
    N = len(obj)
    Rp = rodrigues(poses[:, :3])                                   # (F,3,3)
    Xw = np.einsum("fij,nj->fni", Rp, obj) + poses[:, None, 3:]    # (F,N,3)
    dXw_drho = rotated_point_jacobian(poses[:, None, :3], obj[None])   # (F,N,3,3)
    Jc = np.zeros((C, F, N, 2, CAM_BLOCK))
    Jp = np.zeros((C, F, N, 2, POSE_BLOCK))
    pred = np.zeros((C, F, N, 2))
    for c in range(C):
        fx, fy, cx, cy, k1, k2 = cam[c, :6]
        rc, tc = cam[c, 6:9], cam[c, 9:12]
        Rc = rodrigues(rc)
        Xc = Xw @ Rc.T + tc
        Z = Xc[..., 2]
        x, y = Xc[..., 0] / Z, Xc[..., 1] / Z
        r2 = x * x + y * y
        d = 1 + k1 * r2 + k2 * r2 * r2
        dp = k1 + 2 * k2 * r2
        pred[c, ..., 0] = fx * x * d + cx
        pred[c, ..., 1] = fy * y * d + cy
        Jc[c, ..., 0, 0] = x * d
        Jc[c, ..., 1, 1] = y * d
        Jc[c, ..., 0, 2] = 1
        Jc[c, ..., 1, 3] = 1
        Jc[c, ..., 0, 4] = fx * x * r2
        Jc[c, ..., 1, 4] = fy * y * r2
        Jc[c, ..., 0, 5] = fx * x * r2 * r2
        Jc[c, ..., 1, 5] = fy * y * r2 * r2
        A = np.zeros((F, N, 2, 2))
        A[..., 0, 0] = fx * (d + 2 * x * x * dp)
        A[..., 0, 1] = fx * 2 * x * y * dp
        A[..., 1, 0] = fy * 2 * x * y * dp
        A[..., 1, 1] = fy * (d + 2 * y * y * dp)
        B = np.zeros((F, N, 2, 3))
        B[..., 0, 0] = 1 / Z
        B[..., 1, 1] = 1 / Z
        B[..., 0, 2] = -x / Z
        B[..., 1, 2] = -y / Z
        G = A @ B                                                  # (F,N,2,3)
        Jc[c, ..., 6:9] = G @ rotated_point_jacobian(rc, Xw)
        Jc[c, ..., 9:12] = G
        GR = G @ Rc
        Jp[c, ..., 0:3] = GR @ dXw_drho
        Jp[c, ..., 3:6] = GR
    return Jc, Jp, pred


def dense_residual_jacobian(params, all_calib_uvs, calib_objpoints):
    """Residual Jacobian (m, 12C+6F) in the reference row order (C order over
    (c,f,n,uv), NaN scalars dropped) -- small problems only."""
    C, F, N, _ = all_calib_uvs.shape
    Jc, Jp, _ = jacobian_blocks(params, C, calib_objpoints)
    mask = ~np.isnan(all_calib_uvs)
    ci, fi, ni, ui = np.nonzero(mask)
    J = np.zeros((ci.size, CAM_BLOCK * C + POSE_BLOCK * F))
    rows = np.arange(ci.size)
    for s in range(CAM_BLOCK):
        J[rows, ci * CAM_BLOCK + s] = -Jc[ci, fi, ni, ui, s]
    for s in range(POSE_BLOCK):
        J[rows, CAM_BLOCK * C + fi * POSE_BLOCK + s] = -Jp[ci, fi, ni, ui, s]
    return J


# --------------------------------------------------------------------------
# robust loss and the normal equations scipy's fixed point is defined by
# --------------------------------------------------------------------------
def loss_rho(f, loss="soft_l1", f_scale=1.0):
    """``rho, rho', rho''`` of ``z = (f/f_scale)^2`` (scipy
    optimize/_lsq/least_squares.py:195-201, 226-252); rho is scaled by
    f_scale^2, rho'' divided by it, as scipy's ``loss_function`` does."""
    z = (np.asarray(f) / f_scale) ** 2
    if loss == "linear":
        return z * f_scale ** 2, np.ones_like(z), np.zeros_like(z)
    if loss != "soft_l1":
        raise ValueError(loss)
    t = 1 + z
    return (2 * (t ** 0.5 - 1)) * f_scale ** 2, t ** -0.5, (-0.5 * t ** -1.5) / f_scale ** 2


def robust_scale(J, f, loss="soft_l1", f_scale=1.0, hessian="triggs"):
    """scipy optimize/_lsq/common.py:720-731: row-scale J and f so that
    ``J~^T J~`` is the Triggs-corrected Gauss-Newton matrix and ``J~^T f~`` the
    gradient of ``0.5 sum rho``.  ``hessian='irls'`` uses the majorising weight
    ``rho'`` instead (same gradient and cost; the engine's far-from-minimum mode)."""
    rho, r1, r2 = loss_rho(f, loss, f_scale)
    w = r1 if hessian == "irls" else np.maximum(r1 + 2 * r2 * f ** 2, EPS)
    s = np.sqrt(w)
    return J * s[:, None], f * r1 / s, 0.5 * rho.sum()


def normal_equations(params, all_calib_uvs, calib_objpoints, loss="soft_l1", f_scale=1.0,
                     hessian="triggs"):
    """Dense ``H = J~^T J~`` (n,n), ``g = J~^T f~`` (n,), cost -- small problems."""
    f = residuals(params, all_calib_uvs, calib_objpoints)
    J = dense_residual_jacobian(params, all_calib_uvs, calib_objpoints)
    Js, fs, cost = robust_scale(J, f, loss, f_scale, hessian)
    return Js.T @ Js, Js.T @ fs, cost


def reduced_camera_system(H, g, n_cameras, lam=0.0, D2=None):
    """Schur complement of the (damped) pose blocks (SURVEY.md Appendix A).

    ``S = U - W V^-1 W^T``, ``b = g_c - W V^-1 g_p`` with
    ``U = H_cc + lam D2_c``, ``V = blkdiag_f(H_ff + lam D2_f)``.
    """
    nc = CAM_BLOCK * n_cameras
    Hd = H.copy()
    if lam:
        D2 = np.diag(H).copy() if D2 is None else D2
        Hd[np.diag_indices_from(Hd)] += lam * D2
    U, W, V = Hd[:nc, :nc], Hd[:nc, nc:], Hd[nc:, nc:]
    F = (H.shape[0] - nc) // POSE_BLOCK
    S, b = U.copy(), g[:nc].copy()
    for f in range(F):
        sl = slice(f * POSE_BLOCK, (f + 1) * POSE_BLOCK)
        Vi = np.linalg.inv(V[sl, sl])
        S -= W[:, sl] @ Vi @ W[:, sl].T
        b -= W[:, sl] @ Vi @ g[nc:][sl]
    return S, b


def lm_step(H, g, n_cameras, lam, D2):
    """Full damped step ``-(H + lam diag(D2))^-1 g`` through the Schur route."""
    nc = CAM_BLOCK * n_cameras
    S, b = reduced_camera_system(H, g, n_cameras, lam, D2)
    dc = -np.linalg.solve(S, b)
    Hd = H + lam * np.diag(D2)
    dp = np.zeros(H.shape[0] - nc)
    for f in range(dp.size // POSE_BLOCK):
        sl = slice(f * POSE_BLOCK, (f + 1) * POSE_BLOCK)
        slg = slice(nc + f * POSE_BLOCK, nc + (f + 1) * POSE_BLOCK)
        dp[sl] = -np.linalg.solve(Hd[slg, slg], g[slg] + Hd[:nc, slg].T @ dc)
    return np.concatenate([dc, dp])


def robust_cost(params, all_calib_uvs, calib_objpoints, loss="soft_l1", f_scale=1.0):
    f = residuals(params, all_calib_uvs, calib_objpoints)
    return 0.5 * loss_rho(f, loss, f_scale)[0].sum()


def reprojection_rms(params, all_calib_uvs, calib_objpoints):
    """sqrt(mean f^2) over finite scalar residuals (px)."""
    f = residuals(params, all_calib_uvs, calib_objpoints)
    return float(np.sqrt(np.mean(f * f)))


def analytic_jac_for_scipy(params, all_calib_uvs, calib_objpoints):
    """CSR residual Jacobian usable as ``least_squares(jac=...)`` so that the
    convergence oracle's stationarity is not finite-difference limited
    (SURVEY.md H2)."""
    from scipy.sparse import csr_matrix
    C, F, N, _ = all_calib_uvs.shape
    Jc, Jp, _ = jacobian_blocks(params, C, calib_objpoints)
    mask = ~np.isnan(all_calib_uvs)
    ci, fi, ni, ui = np.nonzero(mask)
    m = ci.size
    vals = np.concatenate([-Jc[ci, fi, ni, ui], -Jp[ci, fi, ni, ui]], axis=1)
    cols = np.concatenate([ci[:, None] * CAM_BLOCK + np.arange(CAM_BLOCK),
                           C * CAM_BLOCK + fi[:, None] * POSE_BLOCK + np.arange(POSE_BLOCK)], axis=1)
    return csr_matrix((vals.ravel(), cols.ravel(), np.arange(m + 1) * 18),
                      shape=(m, C * CAM_BLOCK + F * POSE_BLOCK))


def sparse_gauss_newton_polish(x, all_calib_uvs, calib_objpoints, fun=None, n_iter=40, lam=1e-8,
                               gtol=1e-9, trace=None):
    """Tight minimiser of ``0.5 sum soft_l1(f^2)`` at sizes where a dense Jacobian does not fit
    (BASELINE configs[0]: 210 000 x 3 072): Gauss-Newton on scipy's Triggs-scaled normal equations
    (optimize/_lsq/common.py:720-731) assembled sparse from the analytic Jacobian and factored with
    SuperLU (``scipy.sparse.linalg.splu``); ``lam * diag`` keeps the 6-D rigid gauge (SURVEY.md H1)
    non-singular, a step is kept only if it does not raise the cost.  ``fun`` is the residual
    function (default: the oracle's; the fixture generator passes the reference's).  Returns
    ``(x, cost, ||g||_inf)`` with ``g = J^T (rho' f)`` the gradient at the returned point."""
    from scipy.sparse import diags
    from scipy.sparse.linalg import splu
    fun = residuals if fun is None else fun
    x = np.asarray(x, dtype=float).copy()
    cost_of = lambda p: 0.5 * loss_rho(fun(p, all_calib_uvs, calib_objpoints))[0].sum()
    cost, stalled = cost_of(x), 0
    for it in range(n_iter):
        f = fun(x, all_calib_uvs, calib_objpoints)
        J = analytic_jac_for_scipy(x, all_calib_uvs, calib_objpoints)
        _, r1, r2 = loss_rho(f)
        g = J.T @ (r1 * f)
        gnorm = float(np.abs(g).max())
        if trace is not None:
            trace.append((it, cost, gnorm))
        if gnorm < gtol or stalled >= 3:
            break
        Js = diags(np.sqrt(np.maximum(r1 + 2 * r2 * f ** 2, EPS))) @ J
        H = (Js.T @ Js).tocsc()
        step = -splu((H + diags(lam * H.diagonal())).tocsc()).solve(g)
        cost_new = cost_of(x + step)
        if cost_new <= cost:
            x, cost, stalled = x + step, cost_new, (stalled + 1 if cost_new == cost else 0)
        else:
            lam *= 10.0
            stalled += 1
    return x, cost, gnorm


# --------------------------------------------------------------------------
# initialisation algebra (calibration.py; SURVEY.md 8(f) row N2)
# --------------------------------------------------------------------------
def estimate_pairwise_camera_transform(camera1_poses, camera2_poses):
    """calibration.py:116-143 -- median over the frames both cameras detected of
    ``vec(T2 inv(T1))`` (4x4 matrices, LAPACK inverse, like the reference)."""
    p1, p2 = np.asarray(camera1_poses, dtype=float), np.asarray(camera2_poses, dtype=float)
    both = ~(np.isnan(p1).any(1) | np.isnan(p2).any(1))
    rel = transformation_matrix(p2[both]) @ np.linalg.inv(transformation_matrix(p1[both]))
    return np.median(transformation_vector(rel), axis=0)


def camera_spanning_tree(all_calib_poses, root=0):
    """calibration.py:146-197 -- networkx maximum spanning tree over the co-detection counts
    (networkx is the reference's own, unpinned, dependency for this step), edges oriented away
    from the root and ordered by hop distance."""
    import networkx as nx
    poses = np.asarray(all_calib_poses, dtype=float)
    seen = ~np.isnan(poses).any(2)
    n = len(poses)
    graph = nx.Graph()
    graph.add_nodes_from(range(n))
    graph.add_weighted_edges_from((i, j, (seen[i] & seen[j]).sum()) for i in range(n) for j in range(i + 1, n))
    tree = nx.maximum_spanning_tree(graph)
    hops = nx.shortest_path_length(tree, source=root)
    oriented = [tuple(sorted(e, key=hops.get)) for e in tree.edges]
    return sorted(oriented, key=lambda e: hops[e[0]])


def estimate_all_extrinsics(all_calib_poses, root=0):
    """calibration.py:200-242 -- chain the pairwise transforms along the spanning tree."""
    poses = np.asarray(all_calib_poses, dtype=float)
    T = [None] * len(poses)
    T[root] = np.eye(4)
    tree = camera_spanning_tree(poses, root=root)
    for c1, c2 in tree:
        T[c2] = transformation_matrix(estimate_pairwise_camera_transform(poses[c1], poses[c2])) @ T[c1]
    return np.array([transformation_vector(t) for t in T]), tree


def consensus_calib_poses(all_calib_poses, all_extrinsics):
    """calibration.py:245-277 -- board poses of every detecting camera mapped to world
    coordinates (``inv(T_world->cam) T_board->cam``), nanmedian over cameras."""
    import warnings
    poses = np.asarray(all_calib_poses, dtype=float)
    world = np.full_like(poses, np.nan)
    for c, (p, ext) in enumerate(zip(poses, np.asarray(all_extrinsics, dtype=float))):
        ok = ~np.isnan(p).any(-1)
        world[c, ok] = transformation_vector(np.linalg.inv(transformation_matrix(ext)) @ transformation_matrix(p[ok]))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", category=RuntimeWarning)
        return np.nanmedian(world, axis=0)


# --------------------------------------------------------------------------
# gauge-invariant comparison helpers (SURVEY.md H1)
# --------------------------------------------------------------------------
def relative_camera_transforms(all_extrinsics):
    """``T_c T_0^-1`` (C,4,4): invariant to the global rigid gauge."""
    T = transformation_matrix(np.asarray(all_extrinsics, dtype=float))
    return T @ np.linalg.inv(T[0])


# --------------------------------------------------------------------------
# dense restatement of the device Levenberg-Marquardt loop (small problems)
# --------------------------------------------------------------------------
def lm_solve(x0, all_calib_uvs, calib_objpoints, ftol=1e-4, xtol=1e-8, gtol=1e-8, max_nfev=None,
             loss="soft_l1", f_scale=1.0, lambda0=1e-3, lambda_min=1e-12, lambda_max=1e12, trace=None,
             hessian="auto"):
    """Mirror of ``mcba_lm_run`` (csrc/mcba_api.cu) with dense numpy algebra:
    Gauss-Newton weights IRLS -> Triggs once a step changes the cost by < 1 %
    (``hessian='auto'``), Marquardt scaling D^2 = running max of diag(J~^T J~), Nielsen damping update,
    gain ratio from ``pred = -0.5 g.d + 0.5 lam d^T D^2 d`` and scipy's termination
    tests (optimize/_lsq/common.py:705-717).  Returns (x, info dict)."""
    C = all_calib_uvs.shape[0]
    x = np.asarray(x0, dtype=float).copy()
    max_nfev = 100 * x.size if max_nfev is None else max_nfev
    irls = hessian != "triggs" and loss != "linear"
    mode = lambda: "irls" if irls else "triggs"
    H, g, cost = normal_equations(x, all_calib_uvs, calib_objpoints, loss, f_scale, mode())
    D2 = np.diag(H).copy()
    lam, nu, nfev, njev, it, status = lambda0, 2.0, 1, 1, 0, None
    if np.abs(g).max() < gtol:
        status = 1
    while status is None:
        if nfev >= max_nfev:
            status = 0
            break
        D2e = np.where(D2 == 0, 1.0, D2)
        try:
            step = lm_step(H, g, C, lam, D2e)
            ok = np.isfinite(step).all()
        except np.linalg.LinAlgError:
            ok = False
        nfev += 1
        if ok:
            cost_new = robust_cost(x + step, all_calib_uvs, calib_objpoints, loss, f_scale)
            pred = -0.5 * g @ step + 0.5 * lam * step @ (D2e * step)
            actual = cost - cost_new
            ratio = actual / pred if pred > 0 else -1.0
            sn, xn = np.linalg.norm(step), np.linalg.norm(x)
            f_ok = actual < ftol * cost and ratio > 0.25
            x_ok = sn < xtol * (xtol + xn)
            term = 4 if (f_ok and x_ok) else 2 if f_ok else 3 if x_ok else None
        else:
            actual, ratio, term, sn = -1.0, -1.0, None, np.nan
        if ok and actual > 0:
            x = x + step
            lam = max(lambda_min, lam * max(0.1, 1.0 - (2.0 * ratio - 1.0) ** 3))
            nu = 2.0
            it += 1
            if irls and hessian == "auto" and actual < 1e-2 * cost:
                irls = False
            H, g, cost = normal_equations(x, all_calib_uvs, calib_objpoints, loss, f_scale, mode())
            D2 = np.maximum(D2, np.diag(H))
            njev += 1
            if trace is not None:
                trace.append((it, nfev, cost, actual, sn, np.abs(g).max(), lam, ratio))
            if term is not None:
                status = term
            elif np.abs(g).max() < gtol:
                status = 1
        else:
            if term in (3, 4):
                status = 3
                break
            lam *= nu
            nu *= 2.0
            if lam > lambda_max:
                status = -1
            else:   # the pose damping is part of the factorisation: rebuild at the same point
                H, g, cost = normal_equations(x, all_calib_uvs, calib_objpoints, loss, f_scale, mode())
                D2 = np.maximum(D2, np.diag(H))
    return x, dict(cost=cost, nfev=nfev, njev=njev, iterations=it, status=status,
                   optimality=float(np.abs(g).max()), grad=g, lam=lam)


# --------------------------------------------------------------------------
# reprojection-error QC: numeric core of viz.plot_residuals (viz.py:155-177)
# --------------------------------------------------------------------------
FLT_EPS = float(np.finfo(np.float32).eps)


def homography_dlt(src, dst, round32=True):
    """First half of ``cv2.findHomography(src, dst)`` with ``method=0`` (viz.py:166).

    OpenCV is an un-vendored binary dependency (4.13.0 in the build container); this restates the
    documented algorithm of calib3d's ``HomographyEstimatorCallback::runKernel``: both point sets are
    converted to float32, centred and scaled by the mean absolute deviation per axis, the 9x9
    normal matrix of the DLT rows ``[X Y 1 0 0 0 -xX -xY -x]`` / ``[0 0 0 X Y 1 -yX -yY -y]`` is
    accumulated and its eigenvector of the smallest eigenvalue, de-normalised and divided by
    ``H[2,2]``, is the estimate.  Returns ``(H0, src32, dst32)`` (the rounded points as float64).
    Pinned numerically against cv2 through ``tests/golden/qc.npz``.  ``round32=False`` skips the
    float32 conversion (not what OpenCV does; the tests use it as a wrong kernel).
    """
    t = np.float32 if round32 else np.float64
    M = np.asarray(src, dtype=t).astype(np.float64)
    m = np.asarray(dst, dtype=t).astype(np.float64)
    n = len(M)
    cM, cm = M.sum(0) / n, m.sum(0) / n
    sM, sm = n / np.abs(M - cM).sum(0), n / np.abs(m - cm).sum(0)
    X, x = (M - cM) * sM, (m - cm) * sm
    L = np.zeros((2 * n, 9))
    L[0::2, 0], L[0::2, 1], L[0::2, 2] = X[:, 0], X[:, 1], 1.0
    L[0::2, 6], L[0::2, 7], L[0::2, 8] = -x[:, 0] * X[:, 0], -x[:, 0] * X[:, 1], -x[:, 0]
    L[1::2, 3], L[1::2, 4], L[1::2, 5] = X[:, 0], X[:, 1], 1.0
    L[1::2, 6], L[1::2, 7], L[1::2, 8] = -x[:, 1] * X[:, 0], -x[:, 1] * X[:, 1], -x[:, 1]
    H0 = np.linalg.eigh(L.T @ L)[1][:, 0].reshape(3, 3)
    inv_norm = np.array([[1 / sm[0], 0, cm[0]], [0, 1 / sm[1], cm[1]], [0, 0, 1.0]])
    norm2 = np.array([[sM[0], 0, -cM[0] * sM[0]], [0, sM[1], -cM[1] * sM[1]], [0, 0, 1.0]])
    H = inv_norm @ H0 @ norm2
    return H / H[2, 2], M, m


def homography_residuals(h, M, m, want_jac=True):
    """Reprojection residuals and Jacobian of the 8 free entries of H (``H[2,2] = 1``): OpenCV's
    ``HomographyRefineCallback::compute``."""
    ww = h[6] * M[:, 0] + h[7] * M[:, 1] + 1.0
    ww = np.where(np.abs(ww) > EPS, 1.0 / np.where(ww == 0, 1.0, ww), 0.0)
    xi = (h[0] * M[:, 0] + h[1] * M[:, 1] + h[2]) * ww
    yi = (h[3] * M[:, 0] + h[4] * M[:, 1] + h[5]) * ww
    r = np.empty(2 * len(M))
    r[0::2], r[1::2] = xi - m[:, 0], yi - m[:, 1]
    if not want_jac:
        return r, None
    J = np.zeros((2 * len(M), 8))
    J[0::2, 0], J[0::2, 1], J[0::2, 2] = M[:, 0] * ww, M[:, 1] * ww, ww
    J[0::2, 6], J[0::2, 7] = -M[:, 0] * ww * xi, -M[:, 1] * ww * xi
    J[1::2, 3], J[1::2, 4], J[1::2, 5] = M[:, 0] * ww, M[:, 1] * ww, ww
    J[1::2, 6], J[1::2, 7] = -M[:, 0] * ww * yi, -M[:, 1] * ww * yi
    return r, J


def homography_refine(H, M, m, max_iters=10, eps=FLT_EPS):
    """Second half of ``cv2.findHomography`` for more than four points: OpenCV's ``LMSolver`` (calib3d
    levmarq.cpp, Nash's Marquardt variant) on the reprojection error, at most 10 iterations, step and
    residual tolerance FLT_EPSILON; damping ``lambda * diag(J^T J at the start)``, ``lambda`` starts
    at 1, halves (to 0 below 0.75) after a good step and is rebuilt from ``1 / max diag(A^-1)`` after a
    bad one."""
    x = H.ravel()[:8].copy()
    r, J = homography_residuals(x, M, m)
    S = float(r @ r)
    A, v = J.T @ J, J.T @ r
    D = np.diag(A).copy()
    lam, lc, it = 1.0, 0.75, 0
    while True:
        try:
            d = np.linalg.solve(A + np.diag(lam * D), v)
        except np.linalg.LinAlgError:
            break
        xd = x - d
        rd, _ = homography_residuals(xd, M, m, want_jac=False)
        Sd = float(rd @ rd)
        dS = float(d @ (2.0 * v - A @ d))
        R = (S - Sd) / (dS if abs(dS) > EPS else 1.0)
        if R > 0.75:
            lam *= 0.5
            if lam < lc:
                lam = 0.0
        elif R < 0.25:
            t = float(d @ v)
            nu = min(max((Sd - S) / (t if abs(t) > EPS else 1.0) + 2.0, 2.0), 10.0)
            if lam == 0.0:
                try:
                    lam = lc = 1.0 / max(EPS, float(np.abs(np.diag(np.linalg.inv(A))).max()))
                except np.linalg.LinAlgError:
                    break
                nu *= 0.5
            lam *= nu
        if Sd < S:
            S, x = Sd, xd
            r, J = homography_residuals(x, M, m)
            A, v = J.T @ J, J.T @ r
        it += 1
        if not (it < max_iters and np.abs(d).max() >= eps and np.abs(r).max() >= eps):
            break
    return np.append(x, 1.0).reshape(3, 3)


def find_homography(src, dst):
    """``cv2.findHomography(src, dst)[0]`` for N > 4 points, default method (viz.py:166)."""
    H0, M, m = homography_dlt(src, dst)
    return homography_refine(H0, M, m)


def perspective_transform(points, H):
    """``cv2.perspectiveTransform`` of (N,2) float64 points (viz.py:167-169): ``w = 1 / (H[2] . [x y 1])``
    when ``|.| > eps``, else 0."""
    p = np.asarray(points, dtype=float)
    w = p @ H[2, :2] + H[2, 2]
    w = np.where(np.abs(w) > EPS, 1.0 / np.where(w == 0, 1.0, w), 0.0)
    return np.stack([(p @ H[0, :2] + H[0, 2]) * w, (p @ H[1, :2] + H[1, 2]) * w], axis=-1)


def reprojection_transfer(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints, calib_poses):
    """Numeric core of ``viz.plot_residuals`` (viz.py:155-177): per camera the distortion-free
    projection of the board corners, the undistorted detections, and for every frame whose corners
    were all detected the homography detections -> board plane, through which the projections are
    carried into the board's own coordinates; the median distance to the true corners per camera.
    Returns ``(median_error (C,), reprojections (C,F,N,2), transformed_reprojections (C,F,N,2))``."""
    uvs = np.asarray(all_calib_uvs, dtype=float)
    obj = np.asarray(calib_objpoints, dtype=float)
    C, F, N, _ = uvs.shape
    median_error = np.zeros(C)
    reprojections = np.zeros((C, F, N, 2))
    transformed = np.full((C, F, N, 2), np.nan)
    pts = embed_calib_objpoints(obj, calib_poses)
    for cam in range(C):
        reprojections[cam] = project_points(pts, all_extrinsics[cam], all_intrinsics[cam][0])
        und = undistort_points(uvs[cam], *all_intrinsics[cam])
        valid = np.nonzero(~np.isnan(und).any((-1, -2)))[0]
        for t in valid:
            transformed[cam, t] = perspective_transform(reprojections[cam, t], find_homography(und[t], obj[:, :2]))
        errors = np.linalg.norm(transformed[cam, valid] - obj[:, :2], axis=-1)
        median_error[cam] = np.median(errors)
    return median_error, reprojections, transformed
