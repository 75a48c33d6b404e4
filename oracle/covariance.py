"""Covariance of the calibration (``mcba_covariance``, ``calibration_covariance``) in plain numpy.

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  Definition: ``s^2 inv(H)`` with
``H = J~^T J~``, J~ the residual Jacobian row-scaled by scipy's robust-loss weights
(``np_oracle.robust_scale(..., hessian="triggs")``), after removing the rows and columns of the reference
camera's 6 extrinsics (the gauge), of cameras without a finite observation (NaN) and of frames without one
(NaN).  ``s^2 = sigma^2`` or ``2 cost / (m - p)`` with m finite residual scalars and p the parameters left.

* :func:`dense_covariance` inverts the dense matrix (small problems);
* :func:`blockwise_covariance` uses the block inverse from ``blockwise.BlockwiseEvaluation(lam=0)``:
  ``Sigma_cam = S^-1`` and ``Sigma_f = V_f^-1 + V_f^-1 W_f^T Sigma_cam W_f V_f^-1``, with the engine's
  singularity rule: a relative Cholesky pivot ``s_j / A_jj <= 1e-12`` of an observed frame's pose block or
  of the Jacobi-scaled gauge-fixed camera system raises ``numpy.linalg.LinAlgError``.
"""
import numpy as np

from . import blockwise
from . import np_oracle as orc

PIVOT_TOL = 1e-12


def _observed(uvs):
    fin = ~np.isnan(uvs)
    return fin.any(axis=(1, 2, 3)), fin.any(axis=(0, 2, 3)), int(fin.sum())


def _cam_keep(C, observed, ref):
    """pos per camera row: -2 unobserved camera, -1 gauge, else kept."""
    pos = np.zeros(12 * C, dtype=int)
    for r in range(12 * C):
        c = r // 12
        pos[r] = -2 if not observed[c] else (-1 if (c == ref and r % 12 >= 6) else 0)
    return pos


def _pad_camera(inv_kept, pos):
    nc = pos.size
    keep = pos >= 0
    out = np.zeros((nc, nc))
    out[np.ix_(keep, keep)] = inv_kept
    bad = pos == -2
    out[bad, :] = np.nan
    out[:, bad] = np.nan
    return out


def _s2(sigma, cost, m, p):
    if sigma is not None:
        return float(sigma) ** 2, m - p
    if m <= p:
        raise ValueError(f"{m} residuals do not exceed the {p} free parameters")
    return 2.0 * cost / (m - p), m - p


def relative_pivots(A):
    """Relative pivots ``s_j / A_jj`` of the unpivoted Cholesky factorisation of each matrix of ``A (..., n, n)``
    (0 where a pivot is not positive, as the engine's factor stores it)."""
    A = np.array(A, dtype=float)
    n = A.shape[-1]
    diag = np.einsum("...ii->...i", A).copy()
    L = np.zeros_like(A)
    rel = np.empty(A.shape[:-1])
    for j in range(n):
        s = A[..., j, j] - np.einsum("...k,...k->...", L[..., j, :j], L[..., j, :j])
        with np.errstate(divide="ignore", invalid="ignore"):
            rel[..., j] = np.where(diag[..., j] > 0, s / diag[..., j], 0.0)
        ljj = np.sqrt(np.maximum(s, 0.0))
        inv = np.where(s > 0, 1.0 / np.where(s > 0, ljj, 1.0), 0.0)
        L[..., j, j] = ljj
        L[..., j + 1:, j] = (A[..., j + 1:, j] - np.einsum("...ik,...k->...i", L[..., j + 1:, :j], L[..., j, :j])) * inv[..., None]
    return np.where(rel > 0, rel, 0.0)


def _scaled_inverse(A):
    """inv(A) through the Jacobi-scaled Cholesky; LinAlgError for a relative pivot <= PIVOT_TOL."""
    d = np.sqrt(np.diag(A))
    if not (d > 0).all():
        raise np.linalg.LinAlgError("camera system: zero diagonal entry")
    As = A / d[:, None] / d[None, :]
    if relative_pivots(As).min() <= PIVOT_TOL:
        raise np.linalg.LinAlgError("the gauge-fixed camera system is not positive definite after Jacobi scaling")
    L = np.linalg.cholesky(As)
    Li = np.linalg.inv(L)
    return (Li.T @ Li) / d[:, None] / d[None, :]


def dense_covariance(x, uvs, obj, reference_camera=0, loss="soft_l1", f_scale=1.0, sigma=None):
    """``dict(camera (12C,12C), poses (F,6,6), sigma2, dof, m, cost)`` from the dense Jacobian."""
    uvs = np.asarray(uvs, dtype=float)
    C, F = uvs.shape[:2]
    nc = 12 * C
    f = orc.residuals(x, uvs, obj)
    J = orc.dense_residual_jacobian(x, uvs, obj)
    Js, _, cost = orc.robust_scale(J, f, loss, f_scale, "triggs")
    H = Js.T @ Js
    cam_obs, frame_obs, m = _observed(uvs)
    pos = _cam_keep(C, cam_obs, reference_camera)
    free = np.concatenate([pos >= 0, np.repeat(frame_obs, 6)])
    p = int(free.sum())
    s2, dof = _s2(sigma, cost, m, p)
    inv = np.zeros((H.shape[0], H.shape[0]))
    inv[np.ix_(free, free)] = _scaled_inverse(H[np.ix_(free, free)])
    camera = _pad_camera(inv[np.ix_(pos >= 0, pos >= 0)], pos) * s2
    poses = np.stack([inv[nc + 6 * i:nc + 6 * i + 6, nc + 6 * i:nc + 6 * i + 6] for i in range(F)]) * s2
    poses[~frame_obs] = np.nan
    return dict(camera=camera, poses=poses, sigma2=s2, dof=dof, m=m, cost=cost)


def blockwise_covariance(x, uvs, obj, reference_camera=0, loss="soft_l1", f_scale=1.0, sigma=None, poses=True,
                         chunk=2048):
    """The same from ``BlockwiseEvaluation(lam=0)`` (any number of frames); also ``min_pose_pivot`` and
    ``empty_frames``."""
    uvs = np.asarray(uvs, dtype=float)
    C, F = uvs.shape[:2]
    ev = blockwise.BlockwiseEvaluation(x, uvs, obj, lam=0.0, loss=loss, f_scale=f_scale, hessian="triggs", chunk=chunk)
    cam_obs, frame_obs, m = _observed(uvs)
    if not cam_obs[reference_camera]:
        raise ValueError(f"reference camera {reference_camera} has no observations")
    live = ~ev.empty
    rel = relative_pivots(ev.Vd[live]).min(axis=1) if live.any() else np.array([np.inf])
    n_sing = int((rel <= PIVOT_TOL).sum())
    if n_sing:
        raise np.linalg.LinAlgError(f"{n_sing} frame(s) have a singular pose block")
    pos = _cam_keep(C, cam_obs, reference_camera)
    keep = pos >= 0
    p = int(keep.sum()) + 6 * int(live.sum())
    s2, dof = _s2(sigma, ev.cost, m, p)
    sig = np.zeros((12 * C, 12 * C))
    sig[np.ix_(keep, keep)] = _scaled_inverse(ev.S[np.ix_(keep, keep)])
    out = dict(camera=_pad_camera(sig[np.ix_(keep, keep)], pos) * s2, sigma2=s2, dof=dof, m=m, cost=ev.cost,
               min_pose_pivot=float(rel.min()), empty_frames=int(ev.empty.sum()), poses=None)
    if poses:
        P = np.full((F, 6, 6), np.nan)
        for s in range(0, F, chunk):
            e = min(F, s + chunk)
            Vi = np.linalg.inv(ev.Vd[s:e])
            A = np.matmul(ev.W[s:e], Vi)                                   # (f, 12C, 6)
            blk = Vi + np.matmul(A.transpose(0, 2, 1), np.matmul(sig, A))
            blk = 0.5 * (blk + blk.transpose(0, 2, 1))
            P[s:e] = blk * s2
        P[ev.empty] = np.nan
        out["poses"] = P
    return out
