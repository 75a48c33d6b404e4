"""Blockwise fp64 restatement of one evaluation of the reduced camera system, for any number of frames.

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  :func:`np_oracle.normal_equations` builds the
dense ``(12C + 6F)^2`` matrix and so stops at a few hundred frames.  This module computes the same
quantities (``np_oracle.robust_scale`` weights, ``np_oracle.reduced_camera_system`` elimination) frame
chunk by frame chunk from ``np_oracle.jacobian_blocks``, keeping only per-frame blocks:

* ``U_c = sum J_c^T w J_c`` (camera blocks), ``W_f = [sum J_c^T w J_f]_c`` (12C x 6 coupling of frame f),
  ``V_f = sum_c J_f^T w J_f`` (pose blocks), the gradient ``J^T (rho' f)`` and the cost;
* the Schur complement of the damped pose blocks, ``S = U - sum_f W_f V~_f^-1 W_f^T`` and
  ``b = g_cam - sum_f W_f V~_f^-1 g_f`` with ``V~_f = V_f + lam D_f^2``;
* the damped Levenberg-Marquardt step with the engine's documented damping rules (``mcba.h``,
  ``k2_common.cuh``, ``k3_solve.cu``): pose ``D_f^2 = max(D2pose, diag V_f)`` and camera
  ``D^2 = max(D2cam, diag U)`` (running maxima over the points of a solve, none by default), each entry that
  is 0 replaced by 1; at ``lam = 0`` a frame without observations contributes nothing.

It is pinned to the dense oracle by ``tests/test_host_cpu.py``.
"""
import numpy as np

from . import np_oracle as orc

EPS = np.finfo(float).eps


def _chunk_frames(C, N, chunk):
    """Frames per chunk: ``chunk``, or fewer so that one chunk's Jacobian blocks stay near 100 MB."""
    return max(1, min(chunk, (1 << 19) // max(1, C * N)))


def frame_blocks(x, uvs, obj, s, e, loss="soft_l1", f_scale=1.0, hessian="triggs"):
    """Blocks of frames ``s:e``: ``U (C,12,12)``, ``W (f,12C,6)``, ``V (f,6,6)``, ``g_cam (C,12)``,
    ``g_pose (f,6)``, cost, the number of finite scalars per frame ``(f,)``, the predictions ``(C,f,N,2)`` and the
    rounding scale of the gradient ``|J|^T (|rho'| (|uv| + |pred|))`` as ``(C,12)`` and ``(f,6)``: ``f = uv - pred``
    cancels, so each residual carries an error of order eps (|uv| + |pred|), far above that of the sums."""
    C, F, N, _ = uvs.shape
    nc = 12 * C
    sub = np.concatenate([x[:nc], x[nc + 6 * s:nc + 6 * e]])
    Jc, Jp, pred = orc.jacobian_blocks(sub, C, obj)            # prediction Jacobian; the residual's is -J
    f = uvs[:, s:e] - pred
    m = ~np.isnan(f)
    f0 = np.where(m, f, 0.0)
    rho, r1, r2 = orc.loss_rho(f0, loss, f_scale)
    w = r1 if hessian == "irls" else np.maximum(r1 + 2 * r2 * f0 ** 2, EPS)
    w = np.where(m, w, 0.0)
    wg = np.where(m, r1 * f0, 0.0)
    ws = np.where(m, np.abs(r1) * (np.abs(np.where(m, uvs[:, s:e], 0.0)) + np.abs(pred)), 0.0)
    n = e - s
    Jc = Jc.reshape(C, n, 2 * N, 12)
    Jp = Jp.reshape(C, n, 2 * N, 6)
    w = w.reshape(C, n, 2 * N, 1)
    wg = wg.reshape(C, n, 2 * N)
    ws = ws.reshape(C, n, 2 * N)
    Jcw = Jc * w
    U = np.matmul(Jcw.reshape(C, -1, 12).transpose(0, 2, 1), Jc.reshape(C, -1, 12))
    W = np.matmul(Jcw.transpose(0, 1, 3, 2), Jp)                # (C,f,12,6)
    V = np.matmul((Jp * w).transpose(0, 1, 3, 2), Jp).sum(0)    # (f,6,6)
    g_cam = -np.einsum("cmi,cm->ci", Jc.reshape(C, -1, 12), wg.reshape(C, -1))
    g_pose = -np.einsum("cfmi,cfm->fi", Jp, wg)
    cost = 0.5 * rho[m].sum()
    count = m.reshape(C, n, -1).sum((0, 2))
    r_cam = np.einsum("cmi,cm->ci", np.abs(Jc).reshape(C, -1, 12), ws.reshape(C, -1))
    r_pose = np.einsum("cfmi,cfm->fi", np.abs(Jp), ws)
    return U, W.transpose(1, 0, 2, 3).reshape(n, nc, 6), V, g_cam, g_pose, cost, count, pred, r_cam, r_pose


class BlockwiseEvaluation:
    """One evaluation at ``x``: ``S, b, g_cam, g_pose (F,6), cost, diag_U``, the predictions ``pred (C,F,N,2)``,
    the damped pose blocks and couplings (for :meth:`step`), ``empty`` (frames without a finite scalar) and
    ``g_round`` (12C + 6F), the rounding scale of the gradient (:func:`frame_blocks`).

    ``D2pose`` (F,6): a running Marquardt scaling of the poses carried over from earlier points; the pose damping
    is ``lam * max(D2pose, diag V_f)`` (an entry 0 -> 1), and ``self.D2pose`` holds that maximum afterwards.
    ``U``, ``W`` and the undamped ``V`` are kept, so :meth:`redamp` eliminates again for another ``lam``
    without walking the Jacobian again."""

    def __init__(self, x, uvs, obj, lam=0.0, loss="soft_l1", f_scale=1.0, hessian="triggs", chunk=2048,
                 D2pose=None):
        x = np.asarray(x, dtype=float)
        uvs = np.asarray(uvs, dtype=float)
        C, F, N, _ = uvs.shape
        nc = 12 * C
        self.C, self.F, self.chunk = C, F, chunk
        self.U = np.zeros((C, 12, 12))
        self.diag_U = np.zeros(nc)
        self.g_cam = np.zeros(nc)
        self.g_pose = np.zeros((F, 6))
        self.V = np.zeros((F, 6, 6))
        self.W = np.zeros((F, nc, 6))
        self.empty = np.zeros(F, dtype=bool)
        self.pred = np.empty((C, F, N, 2))
        self.g_round = np.zeros(nc + 6 * F)
        self.cost = 0.0
        step = _chunk_frames(C, N, chunk)
        for s in range(0, F, step):
            e = min(F, s + step)
            U, W, V, gc, gp, cost, count, self.pred[:, s:e], rc, rp = frame_blocks(x, uvs, obj, s, e, loss, f_scale,
                                                                                    hessian)
            self.g_round[:nc] += rc.ravel()
            self.g_round[nc + 6 * s:nc + 6 * e] = rp.ravel()
            self.U += U
            self.g_cam += gc.ravel()
            self.g_pose[s:e] = gp
            self.cost += cost
            self.V[s:e], self.W[s:e], self.empty[s:e] = V, W, count == 0
        for k in range(C):
            self.diag_U[12 * k:12 * k + 12] = np.diag(self.U[k])
        self.diag_V = np.einsum("fii->fi", self.V).copy()
        self.D2pose = self.diag_V.copy() if D2pose is None else np.maximum(D2pose, self.diag_V)
        self.redamp(lam)

    def redamp(self, lam):
        """Eliminate the poses again with pose damping ``lam``: sets ``lam, Vd, S, b``."""
        C, F, nc = self.C, self.F, 12 * self.C
        self.lam = float(lam)
        d2 = self.D2pose.copy()
        d2[d2 == 0.0] = 1.0
        self.Vd = self.V + self.lam * d2[:, :, None] * np.eye(6)
        if self.lam == 0.0:
            self.Vd[self.empty] = np.eye(6)                        # W_f = 0, g_f = 0: contributes nothing
        self.S = np.zeros((nc, nc))
        for k in range(C):
            self.S[12 * k:12 * k + 12, 12 * k:12 * k + 12] = self.U[k]
        zb = np.zeros(nc)
        step = max(1, min(self.chunk, F))
        for s in range(0, F, step):
            e = min(F, s + step)
            W, gp = self.W[s:e], self.g_pose[s:e]
            X = np.linalg.solve(self.Vd[s:e], np.concatenate([W.transpose(0, 2, 1), gp[:, :, None]], axis=2))
            self.S -= W.transpose(1, 0, 2).reshape(nc, -1) @ X[:, :, :nc].reshape(-1, nc)
            zb -= W.transpose(1, 0, 2).reshape(nc, -1) @ X[:, :, nc].reshape(-1)
        self.b = self.g_cam + zb
        return self

    def step(self, lam=None, D2cam=None):
        """Damped step ``[delta_cam (12C) | delta_pose (6F)]`` from this evaluation's system: camera damping
        ``lam * max(D2cam, diag U)`` (an entry 0 -> 1), pose damping as built."""
        lam = self.lam if lam is None else float(lam)
        d2 = self.diag_U.copy()
        if D2cam is not None:
            d2 = np.maximum(d2, D2cam)
        d2[d2 == 0.0] = 1.0
        dcam = -np.linalg.solve(self.S + lam * np.diag(d2), self.b)
        rhs = self.g_pose + np.einsum("fai,a->fi", self.W, dcam)
        dpose = -np.linalg.solve(self.Vd, rhs[:, :, None])[:, :, 0]
        dpose[self.empty] = 0.0
        return np.concatenate([dcam, dpose.ravel()])


def reduced_camera_system_blockwise(x, uvs, obj, lam=0.0, loss="soft_l1", f_scale=1.0, hessian="triggs", chunk=2048):
    """``S, b, g_cam, g_pose (F,6), cost`` of one evaluation (pose damping ``lam``, no camera damping)."""
    ev = BlockwiseEvaluation(x, uvs, obj, lam, loss, f_scale, hessian, chunk)
    return ev.S, ev.b, ev.g_cam, ev.g_pose, ev.cost


def damped_step_blockwise(x, uvs, obj, lam, loss="soft_l1", f_scale=1.0, hessian="triggs", D2cam=None, chunk=2048):
    """Damped step ``[delta_cam | delta_pose]`` at ``x`` with damping ``lam`` on cameras and poses."""
    return BlockwiseEvaluation(x, uvs, obj, lam, loss, f_scale, hessian, chunk).step(D2cam=D2cam)
