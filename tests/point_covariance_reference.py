"""Numpy restatement of ``point_covariance``: the calibration's uncertainty carried into refined points.

Built on ``refine_reference`` (residual, Jacobian in X, scipy's robust weights, the "seen" rule) and on the
oracle's camera Jacobian ``orc.jacobian_blocks``, evaluated with one identity board pose whose object points are
the world points.  ``jacobian_blocks`` has no skew; :func:`camera_jacobian` adds the skew terms of K, which the
projection of ``refine_points`` carries as a constant.
"""
import numpy as np

from oracle import np_oracle as orc
import refine_reference as rr


def camera_params(ext, K, dist):
    """serialize_params' 12 camera parameters: fx fy cx cy k1 k2 rvec tvec."""
    return np.r_[K[0, 0], K[1, 1], K[0, 2], K[1, 2], dist[0], dist[1], ext]


def camera_jacobian(X, ext, Ks, dists):
    """(C, P, 2, 12) Jacobian of the predicted pixel w.r.t. each camera's parameters at world points X (P, 3)."""
    C, P = len(ext), len(X)
    J = np.zeros((C, P, 2, 12))
    with np.errstate(all="ignore"):
        for c in range(C):
            params = np.r_[camera_params(ext[c], Ks[c], dists[c]), np.zeros(6)]
            J[c] = orc.jacobian_blocks(params, 1, X)[0][0, 0]
            s = Ks[c, 0, 1]
            if s == 0.0:
                continue
            # u gains s y d: d/d(k1, k2) s y (r^2, r^4); d/dXc s [dxy, dyy] B, B = d(x, y)/dXc
            R = orc.rodrigues(ext[c, :3])
            Xc = X @ R.T + ext[c, 3:]
            iz = 1 / Xc[:, 2]
            x, y = Xc[:, 0] * iz, Xc[:, 1] * iz
            k1, k2 = dists[c, :2]
            r2 = x * x + y * y
            d = 1 + r2 * (k1 + k2 * r2)
            dd = 2 * (k1 + 2 * k2 * r2)
            dxy, dyy = dd * x * y, d + dd * y * y
            J[c, :, 0, 4] += s * y * r2
            J[c, :, 0, 5] += s * y * r2 * r2
            g = s * np.stack([dxy * iz, dyy * iz, -(dxy * x + dyy * y) * iz], -1)        # (P, 3)
            J[c, :, 0, 6:9] += np.einsum("pi,pij->pj", g, orc.rotated_point_jacobian(ext[c, :3], X))
            J[c, :, 0, 9:12] += g
    return J


def sensitivity(X, uvs, ext, intr, loss="linear", f_scale=1.0):
    """(S (P, 3, 12C), H = J~_X^T J~_X (P, 3, 3), seen (C, P), valid (P,)): S = -H^-1 J~_X^T J~_c per seen camera,
    zero for unseen cameras, NaN where the point is not valid (fewer than two seen views, non-finite X, H not
    positive definite)."""
    ext, Ks, dists = rr.rig(ext, intr)
    uvs = np.asarray(uvs, dtype=float)
    X = np.asarray(X, dtype=float)
    C, P = uvs.shape[:2]
    seen = rr.seen_views(uvs, Ks, dists)
    valid = (seen.sum(0) >= 2) & np.isfinite(X).all(1)
    Xs = np.where(valid[:, None], X, 0.0)
    f, JX = rr.residuals(Xs, uvs, ext, Ks, dists)
    Jc = camera_jacobian(Xs, ext, Ks, dists)
    m = np.broadcast_to(seen[..., None], f.shape)
    f = np.where(m, f, 0.0)
    JX = np.where(m[..., None], JX, 0.0)
    Jc = np.where(m[..., None], Jc, 0.0)
    _, r1, r2 = rr.loss_rho(f, loss, f_scale)
    w = np.where(m, np.maximum(r1 + 2 * r2 * f ** 2, rr.EPS), 0.0)
    H = np.einsum("cpk,cpki,cpkj->pij", w, JX, JX)
    valid &= rr._chol_ok(H)
    B = np.einsum("cpk,cpki,cpkj->pcij", w, JX, Jc)                    # (P, C, 3, 12)
    S = np.full((P, 3, C, 12), np.nan)
    if valid.any():
        S[valid] = -np.einsum("pij,pcjk->pick", np.linalg.inv(H[valid]), B[valid])
    return S.reshape(P, 3, 12 * C), H, seen, valid


def point_covariance(uvs, ext, intr, X, cam_cov, loss="linear", f_scale=1.0, sigma=1.0, sens=None):
    """(measurement, calibration, S), (P, 3, 3), (P, 3, 3), (P, 3, 12C): sigma^2 H^-1 and
    sum_{c,d seen} S_c cov[c,d] S_d^T, the latter NaN where a seen-seen block of cam_cov holds NaN."""
    S, H, seen, valid = sensitivity(X, uvs, ext, intr, loss, f_scale) if sens is None else sens
    C, P = seen.shape
    cam_cov = np.asarray(cam_cov, dtype=float)
    meas = np.full((P, 3, 3), np.nan)
    cal = np.full((P, 3, 3), np.nan)
    if valid.any():
        meas[valid] = sigma ** 2 * np.linalg.inv(H[valid])
    masks, inverse = np.unique(seen.T, axis=0, return_inverse=True)
    for k, mask in enumerate(masks):
        pts = np.flatnonzero((inverse.ravel() == k) & valid)
        if pts.size == 0:
            continue
        cols = np.flatnonzero(np.repeat(mask, 12))
        Sv = S[pts][:, :, cols]
        cal[pts] = np.einsum("pik,kl,pjl->pij", Sv, cam_cov[np.ix_(cols, cols)], Sv)
    return meas, cal, S


def random_camera_covariance(C, seed=0, held=None, nan_cameras=()):
    """A (12C, 12C) covariance with calibration-like scales and correlations; ``held`` (C, 12) bool rows and
    columns are 0 (camera 0's extrinsics when None), ``nan_cameras`` rows and columns NaN."""
    rng = np.random.default_rng(seed)
    std = np.tile([2.0, 2.0, 1.0, 1.0, 2e-3, 1e-3, 1e-3, 1e-3, 1e-3, 0.5, 0.5, 0.5], C)
    A = rng.normal(size=(12 * C, 12 * C + 8))
    corr = A @ A.T
    d = np.sqrt(np.diag(corr))
    cov = corr / np.outer(d, d) * np.outer(std, std)
    if held is None:
        held = np.zeros((C, 12), dtype=bool)
        held[0, 6:] = True
    h = np.asarray(held).ravel()
    cov[h] = 0.0
    cov[:, h] = 0.0
    for c in nan_cameras:
        cov[12 * c:12 * c + 12] = np.nan
        cov[:, 12 * c:12 * c + 12] = np.nan
    return cov
