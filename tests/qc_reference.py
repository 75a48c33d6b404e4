"""CPU references for the reprojection-error QC (viz.reprojection_residuals, k7_qc.cu) on a chosen set
of (camera, frame) pairs.

* :func:`transfer` runs the oracle's restatement of cv2's undistortPoints + findHomography +
  perspectiveTransform (``orc.reprojection_transfer``) per pair.  Keyword arguments switch on one
  plausible mistake at a time (no float32 rounding, no LM refinement, fewer undistortion iterations,
  skew in the normalisation), so the tests can show that their checks reject such a kernel.
* :func:`converged_minimiser` and :func:`sum_squares` are the path-independent reference: the
  float64 minimiser ``H*`` of findHomography's objective on the float32-rounded points, and the
  objective ``S(H)`` of any H.  :func:`recover_homography` reads the H a kernel used back from its
  transferred corners, so ``S`` can be evaluated for a kernel that only returns points.
* :func:`cv2_transfer` restates viz.plot_residuals:155-177 with the real OpenCV calls.
"""
import numpy as np

from oracle import np_oracle as orc

EPS = float(np.finfo(np.float64).eps)


class Scene:
    """Arguments of ``reprojection_residuals`` in the reference's types."""

    def __init__(self, uvs, ext, intr, obj, poses):
        self.uvs = np.asarray(uvs, dtype=np.float64)
        self.ext = np.asarray(ext, dtype=np.float64)
        self.intr = [(np.asarray(K, dtype=np.float64), np.asarray(d, dtype=np.float64)) for K, d in intr]
        self.obj = np.asarray(obj, dtype=np.float64)
        self.poses = np.asarray(poses, dtype=np.float64)

    def args(self):
        return self.uvs, list(self.ext), self.intr, self.obj, self.poses

    def complete(self):
        """(C, F): the frames whose corners were all detected."""
        return ~np.isnan(self.uvs).any((-1, -2))


def reprojections(scene, pairs):
    """(P, N, 2) distortion-free projections of the board corners for the (camera, frame) ``pairs``."""
    out = np.empty((len(pairs), len(scene.obj), 2))
    for c in np.unique(pairs[:, 0]):
        sel = np.nonzero(pairs[:, 0] == c)[0]
        pts = orc.embed_calib_objpoints(scene.obj, scene.poses[pairs[sel, 1]])
        out[sel] = orc.project_points(pts, scene.ext[c], scene.intr[c][0], None)
    return out


def undistort(uv, K, dist, n_iter=5, skew_in_norm=False):
    """``orc.undistort_points``; ``skew_in_norm`` also removes the skew from the input normalisation
    (OpenCV does not: it uses the skew only in the output camera matrix)."""
    if not skew_in_norm:
        return orc.undistort_points(uv, K, dist, n_iter=n_iter)
    y = (uv[..., 1] - K[1, 2]) / K[1, 1]
    shifted = uv.copy()
    shifted[..., 0] = uv[..., 0] - K[0, 1] * y
    return orc.undistort_points(shifted, K, dist, n_iter=n_iter)


def degenerate(src, dst):
    """findHomography's DLT rejects a point set with zero mean absolute deviation along an axis (a
    board seen edge-on, or a board of one row): cv2 returns None, the kernel NaN rows."""
    M = np.asarray(src, dtype=np.float32).astype(np.float64)
    m = np.asarray(dst, dtype=np.float32).astype(np.float64)
    dev = lambda a: np.abs(a - a.sum(0) / len(a)).sum(0)
    return bool((dev(M) < EPS).any() or (dev(m) < EPS).any())


def homography(src, dst, round32=True, refine=True):
    """``orc.find_homography`` split into its halves.  Returns ``(H, H_dlt, M, m)`` with ``M``, ``m``
    the float32-rounded points both are fitted to (also when ``round32`` is off, so a variant is
    scored on the points the kernel sees)."""
    H0, M, m = orc.homography_dlt(src, dst)
    if not round32:
        H0, Mf, mf = orc.homography_dlt(src, dst, round32=False)
    H = orc.homography_refine(H0, *((M, m) if round32 else (Mf, mf))) if refine else H0
    return H, H0, M, m


def transfer(scene, pairs, n_iter=5, skew_in_norm=False, round32=True, refine=True):
    """Oracle transfer of the projections into the board plane for ``pairs`` ((P, 2) camera, frame).

    Returns a dict: ``tr`` (P, N, 2) (NaN rows where a corner is missing or the board is
    degenerate), ``rep`` (P, N, 2), ``H`` / ``H_dlt`` (P, 3, 3), ``M`` / ``m`` (P, N, 2) the rounded
    points of each fit."""
    pairs = np.asarray(pairs)
    P, N = len(pairs), len(scene.obj)
    rep = reprojections(scene, pairs)
    dst = scene.obj[:, :2]
    out = dict(tr=np.full((P, N, 2), np.nan), rep=rep, H=np.full((P, 3, 3), np.nan),
               H_dlt=np.full((P, 3, 3), np.nan), M=np.full((P, N, 2), np.nan), m=np.full((P, N, 2), np.nan))
    for i, (c, f) in enumerate(pairs):
        uv = scene.uvs[c, f]
        if np.isnan(uv).any():
            continue
        und = undistort(uv, *scene.intr[c], n_iter=n_iter, skew_in_norm=skew_in_norm)
        if degenerate(und, dst):
            continue
        H, H0, M, m = homography(und, dst, round32=round32, refine=refine)
        out["tr"][i] = orc.perspective_transform(rep[i], H)
        out["H"][i], out["H_dlt"][i], out["M"][i], out["m"][i] = H, H0, M, m
    return out


def camera_medians(tr, obj, how="mid"):
    """Per camera ``np.nanmedian`` of the distances of ``tr`` (C, F, N, 2) to the board corners;
    ``how="lower"`` takes the lower middle value of an even count instead (a plausible mistake)."""
    err = np.linalg.norm(tr - obj[:, :2], axis=-1).reshape(len(tr), -1)
    out = np.full(len(tr), np.nan)
    for c, e in enumerate(err):
        e = np.sort(e[~np.isnan(e)])
        if len(e):
            out[c] = e[(len(e) - 1) // 2] if how == "lower" else np.median(e)
    return out


# ------------------------------------------------------------------ the path-independent reference
def sum_squares(H, M, m):
    """S(H): findHomography's objective (squared reprojection error of M -> m) of ``H / H[2, 2]``."""
    h = (np.asarray(H, dtype=np.float64) / H[2, 2]).ravel()[:8]
    r, _ = orc.homography_residuals(h, M, m, want_jac=False)
    return float(r @ r)


def converged_minimiser(H, M, m, max_iter=50):
    """The float64 minimiser H* of S on the rounded points: MINPACK's Levenberg-Marquardt from ``H``
    (ten LM iterations leave a board seen at a grazing angle far from it, where undamped Gauss-Newton
    would not descend), then Gauss-Newton (least squares on J, not the normal equations) until the
    relative step is below 1e-14 or S stops decreasing."""
    from scipy.optimize import least_squares
    h = (np.asarray(H, dtype=np.float64) / H[2, 2]).ravel()[:8].copy()
    h = least_squares(lambda p: orc.homography_residuals(p, M, m, want_jac=False)[0], h,
                      jac=lambda p: orc.homography_residuals(p, M, m)[1], method="lm",
                      xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=2000).x
    r, J = orc.homography_residuals(h, M, m)
    S = float(r @ r)
    for _ in range(max_iter):
        d = np.linalg.lstsq(J, r, rcond=None)[0]
        hn = h - d
        rn, Jn = orc.homography_residuals(hn, M, m)
        Sn = float(rn @ rn)
        if Sn > S:
            break
        h, r, J, S = hn, rn, Jn, Sn
        if np.abs(d).max() <= 1e-14 * np.abs(h).max():
            break
    return np.append(h, 1.0).reshape(3, 3)


def recover_homography(rep, tr):
    """The homography that carried the points ``rep`` (N, 2) to ``tr`` (N, 2), read back by a
    Hartley-normalised float64 DLT (the data are exact up to rounding, so this is H to ~1e-15)."""
    def norm(p):
        c = p.mean(0)
        s = np.sqrt(2.0) / np.sqrt(((p - c) ** 2).sum(1)).mean()
        return np.array([[s, 0, -s * c[0]], [0, s, -s * c[1]], [0, 0, 1.0]])
    T1, T2 = norm(rep), norm(tr)
    a = rep @ T1[:2, :2].T + T1[:2, 2]
    b = tr @ T2[:2, :2].T + T2[:2, 2]
    n = len(a)
    L = np.zeros((2 * n, 9))
    L[0::2, 0:2], L[0::2, 2] = a, 1.0
    L[0::2, 6:8], L[0::2, 8] = -b[:, :1] * a, -b[:, 0]
    L[1::2, 3:5], L[1::2, 5] = a, 1.0
    L[1::2, 6:8], L[1::2, 8] = -b[:, 1:] * a, -b[:, 1]
    Hn = np.linalg.svd(L)[2][-1].reshape(3, 3)
    H = np.linalg.inv(T2) @ Hn @ T1
    return H / H[2, 2]


# ------------------------------------------------------------------ OpenCV
def cv2_transfer(scene, pairs):
    """viz.plot_residuals:155-177 with the real OpenCV calls, per (camera, frame) pair:
    ``undistortPoints(uv, K, dist, P=K)``, ``findHomography(und, obj[:, :2])`` and
    ``perspectiveTransform`` of the distortion-free projections.  (P, N, 2), NaN rows where a
    corner is missing."""
    import cv2
    pairs = np.asarray(pairs)
    rep = reprojections(scene, pairs)
    dst = scene.obj[:, :2]
    out = np.full(rep.shape, np.nan)
    for i, (c, f) in enumerate(pairs):
        uv = scene.uvs[c, f]
        if np.isnan(uv).any():
            continue
        K, dist = scene.intr[c]
        und = cv2.undistortPoints(uv[:, None], K, dist[:5], P=K)[:, 0]
        H = cv2.findHomography(und, dst)[0]
        out[i] = cv2.perspectiveTransform(rep[i][None], H)[0]
    return out
