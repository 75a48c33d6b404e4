"""Numpy restatement of ``refine_points``: the per-point least-squares problem, vectorised over points.

Built on the oracle's projection (``orc.project_points``) and robust loss (``orc.loss_rho``, extended here
with scipy's ``huber``, ``cauchy`` and ``arctan``).  Provides the residual, the analytic 2 x 3 Jacobian of
every view, the robust cost, gradient and Triggs-scaled normal matrix (scipy's ``result.jac``), the
covariance, and the damped Gauss-Newton iteration the kernel runs, decision for decision, with scipy's
ftol / xtol / gtol tests per point.
"""
import numpy as np

from oracle import np_oracle as orc

EPS = np.finfo(float).eps
LOSSES = ("linear", "soft_l1", "huber", "cauchy", "arctan")
LAMBDA0, LAMBDA_MIN, LAMBDA_MAX = 1e-4, 1e-12, 1e16


def loss_rho(f, loss, f_scale=1.0):
    """``rho * f_scale^2, rho', rho'' / f_scale^2`` of ``z = (f / f_scale)^2``, as scipy's loss_function."""
    if loss in ("linear", "soft_l1"):
        return orc.loss_rho(f, loss, f_scale)
    z = (np.asarray(f, dtype=float) / f_scale) ** 2
    if loss == "huber":
        small = z <= 1
        with np.errstate(divide="ignore"):
            s = np.sqrt(z)
            r0 = np.where(small, z, 2 * s - 1)
            r1 = np.where(small, 1.0, 1 / np.where(small, 1.0, s))
            r2 = np.where(small, 0.0, -0.5 * np.where(small, 1.0, z) ** -1.5)
    elif loss == "cauchy":
        t = 1 + z
        r0, r1, r2 = np.log1p(z), 1 / t, -1 / t ** 2
    elif loss == "arctan":
        t = 1 + z ** 2
        r0, r1, r2 = np.arctan(z), 1 / t, -2 * z / t ** 2
    else:
        raise ValueError(loss)
    return r0 * f_scale ** 2, r1, r2 / f_scale ** 2


def rig(ext, intr):
    """(C,6), reference intrinsics list -> Ks (C,3,3), dists (C,5)."""
    Ks = np.stack([np.asarray(K, dtype=float) for K, _ in intr])
    dists = np.zeros((len(intr), 5))
    for c, (_, d) in enumerate(intr):
        d = np.asarray(d, dtype=float).ravel()[:5]
        dists[c, :d.size] = d
    return np.asarray(ext, dtype=float), Ks, dists


def seen_views(uvs, Ks, dists):
    """(C,P) bool: the pixel undistorts to a finite point (triangulate's rule)."""
    with np.errstate(all="ignore"):
        und = np.stack([orc.undistort_points(u, K, d) for u, K, d in zip(uvs, Ks, dists)])
    return np.isfinite(und).all(-1)


def residuals(X, uvs, ext, Ks, dists):
    """f = observed - project_points (C,P,2) and the Jacobian of the projection d(u,v)/dX (C,P,2,3)."""
    C = len(ext)
    f = np.empty(uvs.shape)
    J = np.empty(uvs.shape + (3,))
    with np.errstate(all="ignore"):
        for c in range(C):
            f[c] = uvs[c] - orc.project_points(X, ext[c], Ks[c], dists[c, :2])
            R = orc.rodrigues(ext[c, :3])
            Xc = X @ R.T + ext[c, 3:]
            iz = 1 / Xc[:, 2]
            xn, yn = Xc[:, 0] * iz, Xc[:, 1] * iz
            k1, k2 = dists[c, :2]
            r2 = xn * xn + yn * yn
            d = 1 + r2 * (k1 + k2 * r2)
            dd = 2 * (k1 + 2 * k2 * r2)
            dxx, dxy, dyy = d + dd * xn * xn, dd * xn * yn, d + dd * yn * yn
            fx, s, fy = Ks[c, 0, 0], Ks[c, 0, 1], Ks[c, 1, 1]
            A = np.stack([np.stack([fx * dxx + s * dxy, fx * dxy + s * dyy], -1),
                          np.stack([fy * dxy, fy * dyy], -1)], -2) * iz[:, None, None]   # (P,2,2)
            G = np.concatenate([A, -(A[..., 0] * xn[:, None] + A[..., 1] * yn[:, None])[..., None]], -1)
            J[c] = G @ R
    return f, J


def normal_equations(X, uvs, seen, ext, Ks, dists, loss, f_scale, weights="triggs"):
    """cost (P,), gradient (P,3), J~^T J~ (P,3,3) over the seen views: with scipy's robust scaling
    (``weights="triggs"``, scipy's ``result.jac``), or the IRLS majoriser rho' the iteration uses."""
    f, J = residuals(X, uvs, ext, Ks, dists)
    m = np.broadcast_to(seen[..., None], f.shape)
    f = np.where(m, f, 0.0)
    J = np.where(m[..., None], J, 0.0)
    rho, r1, r2 = loss_rho(f, loss, f_scale)
    w = np.where(m, r1 if weights == "irls" else np.maximum(r1 + 2 * r2 * f ** 2, EPS), 0.0)
    cost = 0.5 * np.where(m, rho, 0.0).sum((0, 2))
    g = -np.einsum("cpk,cpki->pi", r1 * f, J)
    H = np.einsum("cpk,cpki,cpkj->pij", w, J, J)
    return cost, g, H


def cost_only(X, uvs, seen, ext, Ks, dists, loss, f_scale):
    f, _ = residuals(X, uvs, ext, Ks, dists)
    rho = loss_rho(np.where(seen[..., None], f, 0.0), loss, f_scale)[0]
    return 0.5 * np.where(seen[..., None], rho, 0.0).sum((0, 2))


def covariance(X, uvs, seen, ext, Ks, dists, loss, f_scale, sigma=1.0):
    return sigma ** 2 * np.linalg.inv(normal_equations(X, uvs, seen, ext, Ks, dists, loss, f_scale)[2])


def refine(uvs, ext, intr, X0, loss="linear", f_scale=1.0, max_iter=50, ftol=1e-12, xtol=1e-12, gtol=1e-10):
    """The kernel's iteration for every point at once: returns (points, status, iterations, cost)."""
    ext, Ks, dists = rig(ext, intr)
    uvs = np.asarray(uvs, dtype=float)
    P = uvs.shape[1]
    seen = seen_views(uvs, Ks, dists)
    n_views = seen.sum(0)
    X0 = np.asarray(X0, dtype=float)
    X = X0.copy()
    status = np.zeros(P, dtype=np.int64)
    iters = np.zeros(P, dtype=np.int64)
    lam = np.full(P, LAMBDA0)
    live = n_views >= 2
    status[~live] = -1
    X[~live] = np.nan
    cost = np.full(P, np.nan)
    g = np.zeros((P, 3))
    H = np.zeros((P, 3, 3))
    fin = live & np.isfinite(X0).all(1)
    if fin.any():
        cost[fin], g[fin], H[fin] = normal_equations(X[fin], uvs[:, fin], seen[:, fin], ext, Ks, dists, loss, f_scale,
                                                     "irls")
    bad = live & ~np.isfinite(cost)
    status[bad] = -2
    act = live & ~bad
    while act.any():
        i = np.flatnonzero(act)
        gt = np.abs(g[i]).max(1) < gtol
        status[i[gt]] = 1
        act[i[gt]] = False
        mx = ~gt & (iters[i] >= max_iter)
        status[i[mx]] = 0
        act[i[mx]] = False
        i = np.flatnonzero(act)
        if i.size == 0:
            break
        iters[i] += 1
        A = H[i] + lam[i, None, None] * np.eye(3) * np.diagonal(H[i], axis1=1, axis2=2)[:, None, :]
        ok = _chol_ok(A)
        dx = np.zeros((i.size, 3))
        if ok.any():
            dx[ok] = np.linalg.solve(A[ok], -g[i[ok]][..., None])[..., 0]
        Xn = X[i] + dx
        cn = np.full(i.size, np.nan)
        if ok.any():
            cn[ok] = cost_only(Xn[ok], uvs[:, i[ok]], seen[:, i[ok]], ext, Ks, dists, loss, f_scale)
        tried = ok & np.isfinite(cn)
        pred = -(g[i] * dx).sum(1) - 0.5 * np.einsum("pi,pij,pj->p", dx, H[i], dx)
        dF = cost[i] - cn
        with np.errstate(all="ignore"):
            ratio = np.where(pred > 0, dF / np.where(pred > 0, pred, 1), np.where((pred == 0) & (dF == 0), 1.0, 0.0))
        ftol_ok = tried & (dF < ftol * cost[i]) & (ratio > 0.25)
        xtol_ok = tried & (np.linalg.norm(dx, axis=1) < xtol * (xtol + np.linalg.norm(X[i], axis=1)))
        term = np.where(ftol_ok & xtol_ok, 4, np.where(ftol_ok, 2, np.where(xtol_ok, 3, 0)))
        acc = tried & (dF > 0)
        X[i[acc]] = Xn[acc]
        cost[i[acc]] = cn[acc]
        status[i[term > 0]] = term[term > 0]
        act[i[term > 0]] = False
        go = term == 0
        up = i[go & acc]
        lam[up] = np.maximum(lam[up] * 0.1, LAMBDA_MIN)
        if up.size:
            cost[up], g[up], H[up] = normal_equations(X[up], uvs[:, up], seen[:, up], ext, Ks, dists, loss, f_scale,
                                                       "irls")
        down = i[go & ~acc]
        lam[down] *= 10
        blown = down[lam[down] > LAMBDA_MAX]
        status[blown] = -2
        act[blown] = False
    X[status == -2] = X0[status == -2]
    out_cost = np.full(P, np.nan)
    have = (status != -1) & np.isfinite(X).all(1)
    if have.any():
        out_cost[have] = cost_only(X[have], uvs[:, have], seen[:, have], ext, Ks, dists, loss, f_scale)
    return X, status, iters, out_cost


def _chol_ok(A):
    """(P,3,3) -> (P,) bool: the three Cholesky pivots are positive and finite (the kernel's chol3)."""
    with np.errstate(all="ignore"):
        d0 = A[:, 0, 0]
        l10, l20 = A[:, 0, 1] / np.sqrt(d0), A[:, 0, 2] / np.sqrt(d0)
        d1 = A[:, 1, 1] - l10 * l10
        l21 = (A[:, 1, 2] - l20 * l10) / np.sqrt(d1)
        d2 = A[:, 2, 2] - l20 * l20 - l21 * l21
        piv = np.stack([d0, d1, d2], 1)
    return ((piv > 0) & (piv < np.inf)).all(1)


def view_errors(X, uvs, seen, ext, Ks, dists):
    f, _ = residuals(X, uvs, ext, Ks, dists)
    return np.where(seen, np.linalg.norm(f, axis=-1), np.nan)
