"""Reference for camera parameters held fixed (``fixed=``), built on the unmodified oracle: the masked damped step
from ``blockwise.BlockwiseEvaluation`` and the masked covariance in its dense and blockwise forms.

A held parameter is one more column removed from the least-squares problem.  The Schur complement of the
restricted problem is the sub-matrix of S, so the masked step solves the free rows of the damped reduced system and
back-substitutes the poses with the held entries of delta_cam at 0.  The covariance removes the held rows and
columns as well (exactly 0, which wins over the NaN of an unobserved camera).  Gauge rule: a mask that holds all six
extrinsics of some camera replaces the gauge (``reference_camera`` None or such a camera); otherwise the reference
camera is the gauge and the mask may hold no extrinsic entry (``ValueError``)."""
import numpy as np

from oracle import blockwise
from oracle import covariance as ocov
from oracle import np_oracle as orc


def masked_step(ev, fixed, lam=None, D2cam=None):
    """``BlockwiseEvaluation.step`` on the free sub-system: ``[delta_cam (12C) | delta_pose (6F)]``, held entries of
    delta_cam exactly 0."""
    lam = ev.lam if lam is None else float(lam)
    d2 = ev.diag_U.copy()
    if D2cam is not None:
        d2 = np.maximum(d2, D2cam)
    d2[d2 == 0.0] = 1.0
    free = ~np.asarray(fixed, dtype=bool).ravel()
    dcam = np.zeros(ev.b.size)
    A = ev.S + lam * np.diag(d2)
    if free.any():
        dcam[free] = -np.linalg.solve(A[np.ix_(free, free)], ev.b[free])
    rhs = ev.g_pose + np.einsum("fai,a->fi", ev.W, dcam)
    dpose = -np.linalg.solve(ev.Vd, rhs[:, :, None])[:, :, 0]
    dpose[ev.empty] = 0.0
    return np.concatenate([dcam, dpose.ravel()])


def gauge(C, reference_camera, fixed):
    """The camera whose extrinsics are the gauge, or None when the mask pins one itself; ValueError for the
    combinations the engine rejects."""
    held = np.zeros((C, 12), dtype=bool) if fixed is None else np.asarray(fixed, dtype=bool)
    pinned = held[:, 6:].all(axis=1)
    if pinned.any():
        if reference_camera is not None and not pinned[reference_camera]:
            raise ValueError("reference_camera is not a camera whose six extrinsics are held")
        return None
    if reference_camera is None:
        raise ValueError("reference_camera None needs a camera whose six extrinsics are held")
    if held[:, 6:].any():
        raise ValueError("a partial extrinsic mask with a reference camera over-constrains the gauge")
    return reference_camera


def _cam_pos(C, observed, ref, fixed):
    """pos per camera row: -3 held by the mask, -2 unobserved camera, -1 gauge, else kept."""
    held = np.zeros(12 * C, dtype=bool) if fixed is None else np.asarray(fixed, dtype=bool).ravel()
    pos = np.zeros(12 * C, dtype=int)
    for r in range(12 * C):
        c = r // 12
        pos[r] = -3 if held[r] else -2 if not observed[c] else (-1 if (c == ref and r % 12 >= 6) else 0)
    return pos


def _pad_camera(inv_kept, pos):
    nc = pos.size
    keep = pos >= 0
    out = np.zeros((nc, nc))
    out[np.ix_(keep, keep)] = inv_kept
    bad = pos == -2
    out[bad, :] = np.nan
    out[:, bad] = np.nan
    out[pos == -3, :] = 0.0
    out[:, pos == -3] = 0.0
    return out


def _scaled_inverse(A):
    return A.copy() if A.size == 0 else ocov._scaled_inverse(A)


def dense_covariance(x, uvs, obj, reference_camera=0, loss="soft_l1", f_scale=1.0, sigma=None, fixed=None):
    """``ocov.dense_covariance`` with the mask: ``dict(camera, poses, sigma2, dof, m, cost)``."""
    uvs = np.asarray(uvs, dtype=float)
    C, F = uvs.shape[:2]
    nc = 12 * C
    f = orc.residuals(x, uvs, obj)
    J = orc.dense_residual_jacobian(x, uvs, obj)
    Js, _, cost = orc.robust_scale(J, f, loss, f_scale, "triggs")
    H = Js.T @ Js
    cam_obs, frame_obs, m = ocov._observed(uvs)
    pos = _cam_pos(C, cam_obs, gauge(C, reference_camera, fixed), fixed)
    free = np.concatenate([pos >= 0, np.repeat(frame_obs, 6)])
    s2, dof = ocov._s2(sigma, cost, m, int(free.sum()))
    inv = np.zeros((H.shape[0], H.shape[0]))
    inv[np.ix_(free, free)] = _scaled_inverse(H[np.ix_(free, free)])
    camera = _pad_camera(inv[np.ix_(pos >= 0, pos >= 0)], pos) * s2
    poses = np.stack([inv[nc + 6 * i:nc + 6 * i + 6, nc + 6 * i:nc + 6 * i + 6] for i in range(F)]) * s2
    poses[~frame_obs] = np.nan
    return dict(camera=camera, poses=poses, sigma2=s2, dof=dof, m=m, cost=cost)


def blockwise_covariance(x, uvs, obj, reference_camera=0, loss="soft_l1", f_scale=1.0, sigma=None, fixed=None,
                         chunk=2048):
    """``ocov.blockwise_covariance`` with the mask (any number of frames)."""
    uvs = np.asarray(uvs, dtype=float)
    C, F = uvs.shape[:2]
    ev = blockwise.BlockwiseEvaluation(x, uvs, obj, lam=0.0, loss=loss, f_scale=f_scale, hessian="triggs", chunk=chunk)
    cam_obs, frame_obs, m = ocov._observed(uvs)
    ref = gauge(C, reference_camera, fixed)
    if ref is not None and not cam_obs[ref]:
        raise ValueError(f"reference camera {ref} has no observations")
    live = ~ev.empty
    rel = ocov.relative_pivots(ev.Vd[live]).min(axis=1) if live.any() else np.array([np.inf])
    if (rel <= ocov.PIVOT_TOL).any():
        raise np.linalg.LinAlgError(f"{int((rel <= ocov.PIVOT_TOL).sum())} frame(s) have a singular pose block")
    pos = _cam_pos(C, cam_obs, ref, fixed)
    keep = pos >= 0
    s2, dof = ocov._s2(sigma, ev.cost, m, int(keep.sum()) + 6 * int(live.sum()))
    sig = np.zeros((12 * C, 12 * C))
    sig[np.ix_(keep, keep)] = _scaled_inverse(ev.S[np.ix_(keep, keep)])
    P = np.full((F, 6, 6), np.nan)
    for s in range(0, F, chunk):
        e = min(F, s + chunk)
        Vi = np.linalg.inv(ev.Vd[s:e])
        A = np.matmul(ev.W[s:e], Vi)                                   # (f, 12C, 6)
        blk = Vi + np.matmul(A.transpose(0, 2, 1), np.matmul(sig, A))
        P[s:e] = 0.5 * (blk + blk.transpose(0, 2, 1)) * s2
    P[ev.empty] = np.nan
    return dict(camera=_pad_camera(sig[np.ix_(keep, keep)], pos) * s2, poses=P, sigma2=s2, dof=dof, m=m, cost=ev.cost,
                empty_frames=int(ev.empty.sum()))
