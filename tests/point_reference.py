"""Reference helpers for ``tests/test_point_kernels.py``: error bounds of the pairwise DLT solve and
a few deliberately wrong triangulations that the bounds must reject.

For one camera pair the device solves ``A X = 0`` for the 4x4 DLT matrix ``A`` (k5_points.cu:310-321)
and de-homogenises ``X``.  With the singular values ``s1 >= s2 >= s3 >= s4`` of ``A`` and
``x = (p, 1) / |(p, 1)|`` for a returned point ``p``, a backward-stable solve satisfies

* residual:      ``|A x| <= s4 + c eps s1``               (whatever the gap ``s3 - s4``);
* forward error: ``angle(x, v4) <= c eps s1 / (s3 - s4)``  (``v4`` the exact smallest right vector).

Moving ``x`` by an angle ``t`` moves ``p = x[:3] / x[3]`` by at most ``t s (1 + |p|)``, ``s = |(p, 1)|``,
and a per-coordinate median is 1-Lipschitz, so the all-pairs triangulation of a point is within the
largest such bound among its pairs.  ``c`` is a fixed multiple of the unit roundoff, not a per-test
constant; the tests print the largest measured/bound ratio.
"""
import itertools

import numpy as np

from oracle import np_oracle as orc

EPS = np.finfo(float).eps
C_BOUND = 64.0


def projection_matrices(extrinsics, intrinsics):
    return np.stack([orc.projection_matrix(e, i) for e, i in zip(extrinsics, intrinsics)])


def dlt(und_i, und_j, Pi, Pj):
    """(n,2), (n,2) undistorted pixels of two cameras -> (n,4,4) DLT matrices, row order of the kernel."""
    return np.stack([und_i[:, 0, None] * Pi[2] - Pi[0], und_i[:, 1, None] * Pi[2] - Pi[1],
                     und_j[:, 0, None] * Pj[2] - Pj[0], und_j[:, 1, None] * Pj[2] - Pj[1]], axis=1)


def svd_bound(A, c=C_BOUND):
    """Singular values (n,4), smallest right singular vectors (n,4) and the angle bound (n,)."""
    _, sig, vt = np.linalg.svd(A)
    with np.errstate(divide="ignore"):
        theta = c * EPS * sig[:, 0] / (sig[:, 2] - sig[:, 3])
    return sig, vt[:, -1, :], theta


def unit_homogeneous(p):
    """``(p, 1) / |(p, 1)|`` for finite points, computed without overflow."""
    x = np.concatenate([p, np.ones((len(p), 1))], axis=1)
    m = np.abs(x).max(1, keepdims=True)
    x = x / m
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def angle(x, v):
    """Angle between the lines spanned by unit vectors x and v (accurate near 0)."""
    d = np.minimum(np.linalg.norm(x - v, axis=1), np.linalg.norm(x + v, axis=1))
    return 2.0 * np.arcsin(np.minimum(d / 2.0, 1.0))


def pair_ratios(A, p, c=C_BOUND):
    """Measured/bound ratios of one pair's solution ``p`` (n,3), NaN where ``p`` is not finite: the
    residual's excess over s4, ``(|A x| - s4) / (c eps s1)``, and the forward error
    ``angle(x, v4) / theta``.  Both must be <= 1."""
    sig, v, theta = svd_bound(A, c)
    fin = np.isfinite(p).all(1)
    res = np.full(len(p), np.nan)
    fwd = np.full(len(p), np.nan)
    x = unit_homogeneous(p[fin])
    res[fin] = (np.linalg.norm(np.einsum("nij,nj->ni", A[fin], x), axis=1) - sig[fin, 3]) / (c * EPS * sig[fin, 0])
    fwd[fin] = angle(x, v[fin]) / theta[fin]
    return res, fwd


def point_tolerance(und, Ps, c=C_BOUND):
    """Per-point tolerance of an all-pairs triangulation against another fp64 one, and the number
    of pairs of every point.  ``und`` (C,P,2) undistorted pixels, NaN where a view is not seen;
    ``Ps`` (C,3,4).  Each side is within the largest pair bound ``theta s (1 + |p|)`` of the exact
    median, so two of them are within twice that."""
    C, P, _ = und.shape
    seen = ~np.isnan(und).any(-1)
    tol = np.zeros(P)
    npairs = np.zeros(P, dtype=np.int64)
    for i, j in itertools.combinations(range(C), 2):
        idx = np.nonzero(seen[i] & seen[j])[0]
        if idx.size == 0:
            continue
        _, v, theta = svd_bound(dlt(und[i, idx], und[j, idx], Ps[i], Ps[j]), c)
        with np.errstate(divide="ignore", invalid="ignore"):
            p = v[:, :3] / v[:, 3:]
        s = np.sqrt(1.0 + (p * p).sum(1))
        b = 2.0 * theta * s * (1.0 + np.linalg.norm(p, axis=1))
        tol[idx] = np.fmax(tol[idx], np.where(np.isfinite(b), b, np.inf))
        npairs[idx] += 1
    return tol, npairs


def qr_settles(A):
    """numpy restatement of ``null_vector_qr``'s exit test (k5_points.cu:193-274): True where the
    Householder QR + inverse iteration settles, False where the kernel falls back to the Jacobi SVD."""
    R = np.array(A, dtype=float)
    n = len(R)
    with np.errstate(all="ignore"):
        for k in range(3):
            col = R[:, k:, k].copy()
            alpha = -np.copysign(np.sqrt((col * col).sum(1)), R[:, k, k])
            v = col
            v[:, 0] -= alpha
            vv = (v * v).sum(1)
            beta = np.where(vv > 0, 2.0 / np.where(vv > 0, vv, 1.0), 0.0)
            for j in range(k + 1, 4):
                d = beta * (v * R[:, k:, j]).sum(1)
                R[:, k:, j] -= d[:, None] * v
            R[:, k, k] = alpha
        scale = np.abs(R[:, 0, 0]) + np.abs(R[:, 1, 1]) + np.abs(R[:, 2, 2])
        alive = (scale > 0) & (scale < np.inf)
        for k in range(3):
            alive &= ~(np.abs(R[:, k, k]) < 1e-12 * scale)
        r33 = np.where(np.abs(R[:, 3, 3]) < 1e-300, 1e-300, R[:, 3, 3])
        i0, i1, i2, i3 = 1 / R[:, 0, 0], 1 / R[:, 1, 1], 1 / R[:, 2, 2], 1 / r33
        y = np.empty((n, 4))
        y[:, 3] = 1.0
        y[:, 2] = -R[:, 2, 3] * i2
        y[:, 1] = -(R[:, 1, 2] * y[:, 2] + R[:, 1, 3]) * i1
        y[:, 0] = -(R[:, 0, 1] * y[:, 1] + R[:, 0, 2] * y[:, 2] + R[:, 0, 3]) * i0
        y /= np.sqrt((y * y).sum(1, keepdims=True))
        ok = np.zeros(n, dtype=bool)
        for it in range(8):
            z0 = y[:, 0] * i0
            z1 = (y[:, 1] - R[:, 0, 1] * z0) * i1
            z2 = (y[:, 2] - R[:, 0, 2] * z0 - R[:, 1, 2] * z1) * i2
            z3 = (y[:, 3] - R[:, 0, 3] * z0 - R[:, 1, 3] * z1 - R[:, 2, 3] * z2) * i3
            w = np.empty((n, 4))
            w[:, 3] = z3 * i3
            w[:, 2] = (z2 - R[:, 2, 3] * w[:, 3]) * i2
            w[:, 1] = (z1 - R[:, 1, 2] * w[:, 2] - R[:, 1, 3] * w[:, 3]) * i1
            w[:, 0] = (z0 - R[:, 0, 1] * w[:, 1] - R[:, 0, 2] * w[:, 2] - R[:, 0, 3] * w[:, 3]) * i0
            m = np.abs(w).max(1)
            alive &= (m > 0) & (m < np.inf)
            w /= np.where(alive, m, 1.0)[:, None]
            nrm = 1.0 / np.sqrt((w * w).sum(1))
            nrm = np.where((w * y).sum(1) < 0, -nrm, nrm)
            w *= nrm[:, None]
            diff = np.abs(w - y).max(1)
            step = alive & ~ok
            y[step] = w[step]
            ok |= step & (it >= 1) & (diff < 1e-13)
    return ok


# ---------------------------------------------------------------- two-camera rigs
def pair_rig(kind, n=2000, seed=0):
    """Two cameras and their pixels ``(all_uvs, ext (2,6), intr)``; one pair, so a triangulation is
    that pair's solution with no median.

    * ``ring``:     cameras 0 and 1 of the 6-camera ring of ``make_keypoints``, sigma 0.3 px;
    * ``baseline``: ring camera 0 and a copy moved 0.5 mm along its x axis, sigma 0.3 px (nearly
      parallel rays: about half the pairs take the Jacobi fallback);
    * ``parallel``: one orientation, one distortion-free camera matrix, a pure translation and
      identical pixels in both views, so the rays are parallel and the point is at infinity;
    * ``exact``:    the ``ring`` rig with sigma 0.
    """
    from multicam_calibration_b200.synthetic import make_keypoints
    sigma = 0.0 if kind == "exact" else 0.3
    all_uvs, ext, intr, pts = make_keypoints(n, 6, sigma=sigma, p_missing=0.0, seed=seed)
    if kind in ("ring", "exact"):
        return all_uvs[:2], ext[:2].copy(), intr[:2]
    rng = np.random.default_rng([seed, 11])
    e1 = ext[0].copy()
    if kind == "baseline":
        e1[3] -= 0.5                                    # camera centre moved 0.5 mm along its own x axis
        K, dc = intr[0]
        uv1 = orc.project_points(pts, e1, K, dc) + rng.normal(0, 0.3, (n, 2))
        return [all_uvs[0], uv1], np.stack([ext[0], e1]), [intr[0], intr[0]]
    assert kind == "parallel"
    e1[3:] += np.array([40.0, -25.0, 10.0])
    K = intr[0][0]
    nodist = (K, np.zeros(5))
    uv = np.stack([rng.uniform(0, 1280, n), rng.uniform(0, 1024, n)], axis=1)
    return [uv, uv.copy()], np.stack([ext[0], e1]), [nodist, nodist]


def ray_directions(uv, ext, K):
    """World directions of the viewing rays of undistorted pixels (n,2) of one camera."""
    R = orc.rodrigues(ext[:3])
    d = np.linalg.solve(K, np.concatenate([uv, np.ones((len(uv), 1))], axis=1).T).T @ R
    return d / np.linalg.norm(d, axis=1, keepdims=True)


# ---------------------------------------------------------------- wrong triangulations (sharpness)
def triangulate_variant(all_uvs, extrinsics, intrinsics, n_iter=5, median="mean", vector=-1):
    """``orc.triangulate`` with one thing changed: ``n_iter`` undistortion iterations, ``median='lower'``
    (lower middle value instead of the mean of the two middle ones) or ``vector=-2`` (the
    second-smallest right singular vector)."""
    C = len(extrinsics)
    P = all_uvs[0].shape[0]
    und = [orc.undistort_points(uv, K, dc, n_iter=n_iter) for uv, (K, dc) in zip(all_uvs, intrinsics)]
    Ps = projection_matrices(extrinsics, intrinsics)
    pair_pts = []
    for i, j in itertools.combinations(range(C), 2):
        pts = np.full((P, 3), np.nan)
        ok = ~(np.isnan(und[i]).any(-1) | np.isnan(und[j]).any(-1))
        if ok.any():
            X = np.linalg.svd(dlt(und[i][ok], und[j][ok], Ps[i], Ps[j]))[2][:, vector, :]
            pts[ok] = X[:, :3] / X[:, 3:]
        pair_pts.append(pts)
    pair_pts = np.stack(pair_pts)
    out = np.full((P, 3), np.nan)
    some = ~np.isnan(pair_pts).all(axis=(0, 2))
    vals = pair_pts[:, some]
    if median == "mean":
        with np.errstate(all="ignore"), np.testing.suppress_warnings() as sup:
            sup.filter(RuntimeWarning)
            out[some] = np.nanmedian(vals, axis=0)
    else:
        srt = np.sort(vals, axis=0)                       # NaNs last
        cnt = (~np.isnan(vals)).sum(0)
        k = np.maximum((cnt - 1) // 2, 0)
        out[some] = np.take_along_axis(srt, k[None], axis=0)[0]
        out[some] = np.where(cnt > 0, out[some], np.nan)
    return out
