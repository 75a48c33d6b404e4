"""Covariance of the calibration (``calibration_covariance``, ``BAProblem.covariance``, ``mcba_covariance``).

CPU: the blockwise reference (oracle/covariance.py) against the dense one, the dense one against scipy's own
``result.jac`` recipe, and argument validation.  GPU: the engine against the blockwise reference at production
sizes and for every kernel variant, a statistical check that the predicted covariance matches the scatter of
solutions under known noise, the handle's state after a call, the error paths and the public call end to end."""
import ctypes

import numpy as np
import pytest

import multicam_calibration_b200 as mcc
from multicam_calibration_b200.synthetic import make_scene
from oracle import covariance as ocov
from oracle import np_oracle as orc


def _normalised_diff(A, B):
    """max |A - B| / sqrt(B_ii B_jj) over the finite entries of B (NaN / zero patterns must match)."""
    assert np.array_equal(np.isnan(A), np.isnan(B))
    d = np.sqrt(np.abs(np.einsum("...ii->...i", np.nan_to_num(B))))
    scale = d[..., :, None] * d[..., None, :]
    fin = ~np.isnan(B) & (scale > 0)
    assert (A[~np.isnan(B) & (scale == 0)] == 0).all()
    return float((np.abs(A - B)[fin] / scale[fin]).max()) if fin.any() else 0.0


def _small_scene(C=4, F=40, seed=0, empty_frame=None, no_camera=None):
    sc = make_scene(C, F, sigma=0.4, p_missing_view=0.2, p_missing_corner=0.05, seed=seed)
    uvs = sc.uvs.copy()
    if empty_frame is not None:
        uvs[:, empty_frame] = np.nan
    if no_camera is not None:
        uvs[no_camera] = np.nan
    return uvs, sc.objpoints, sc.x0()


def _cond_scaled(camera):
    keep = np.isfinite(np.diag(camera)) & (np.diag(camera) > 0)
    A = camera[np.ix_(keep, keep)]
    d = np.sqrt(np.diag(A))
    return float(np.linalg.cond(A / d[:, None] / d[None, :]))


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("loss,f_scale,ref,variant", [
    ("linear", 1.0, 0, None), ("soft_l1", 1.0, 0, None), ("soft_l1", 0.25, 0, None),
    ("soft_l1", 1.0, 2, None), ("linear", 1.0, 2, None), ("soft_l1", 0.25, 2, "holes")])
def test_blockwise_matches_dense(loss, f_scale, ref, variant):
    kw = dict(empty_frame=7, no_camera=1) if variant == "holes" else {}
    uvs, obj, x = _small_scene(seed=3, **kw)
    d = ocov.dense_covariance(x, uvs, obj, ref, loss, f_scale)
    b = ocov.blockwise_covariance(x, uvs, obj, ref, loss, f_scale)
    assert abs(b["sigma2"] - d["sigma2"]) <= 1e-12 * d["sigma2"]
    assert b["dof"] == d["dof"] and b["m"] == d["m"]
    # the two references sum in different orders: agreement is bounded by rounding of S (1e-16 - 1e-15 relative,
    # more where the soft_l1 weights span many decades at f_scale 0.25) times the condition number
    tol = max(1e-10, 1e-13 * _cond_scaled(d["camera"]))
    assert _normalised_diff(b["camera"], d["camera"]) <= tol
    assert _normalised_diff(b["poses"], d["poses"]) <= tol
    g = slice(12 * ref + 6, 12 * ref + 12)
    for c in (d["camera"][g], b["camera"][g], b["camera"][:, g]):
        assert (c[~np.isnan(c)] == 0).all()
    if variant == "holes":
        assert np.isnan(d["camera"][12:24]).all() and np.isnan(d["poses"][7]).all()
        assert b["empty_frames"] == 1


@pytest.mark.parametrize("loss", ["linear", "soft_l1"])
def test_dense_matches_scipy_result_jac(loss):
    """The definition is scipy's: ``inv(J^T J) 2 cost / (m - p)`` from ``least_squares``' ``res.jac``."""
    from scipy.optimize import least_squares
    sc = make_scene(3, 25, sigma=0.5, p_missing_view=0.1, seed=5)
    uvs, obj = sc.uvs, sc.objpoints
    f_scale = 0.5 if loss == "soft_l1" else 1.0
    res = least_squares(orc.residuals, sc.x0(), jac=orc.analytic_jac_for_scipy, args=(uvs, obj), loss=loss,
                        f_scale=f_scale, method="trf", ftol=1e-15, xtol=1e-15, gtol=1e-15, max_nfev=200)
    J = res.jac.toarray() if hasattr(res.jac, "toarray") else np.asarray(res.jac)
    keep = np.ones(J.shape[1], dtype=bool)
    keep[6:12] = False
    Jk = J[:, keep]
    m, p = J.shape[0], int(keep.sum())
    cov = np.linalg.inv(Jk.T @ Jk) * 2 * res.cost / (m - p)
    d = ocov.dense_covariance(res.x, uvs, obj, 0, loss, f_scale)
    full = np.zeros((J.shape[1], J.shape[1]))
    full[np.ix_(keep, keep)] = cov
    assert abs(d["sigma2"] - 2 * res.cost / (m - p)) <= 1e-10 * d["sigma2"]
    assert _normalised_diff(d["camera"], full[:36, :36]) <= 1e-8
    poses = np.stack([full[36 + 6 * i:42 + 6 * i, 36 + 6 * i:42 + 6 * i] for i in range(25)])
    assert _normalised_diff(d["poses"], poses) <= 1e-8


def test_argument_validation_without_cuda():
    sc = make_scene(3, 10, seed=1)
    ext, intr, poses = orc.deserialize_params(sc.x0(), 3)
    args = (sc.uvs, ext, intr, sc.objpoints, poses)
    for kw in (dict(reference_camera=3), dict(reference_camera=-1), dict(reference_camera=1.0),
               dict(sigma=0.0), dict(sigma=-1.0), dict(sigma=np.nan), dict(sigma=np.inf),
               dict(loss="huber"), dict(loss="soft_l1_irls"), dict(f_scale=0.0)):
        with pytest.raises(ValueError):
            mcc.calibration_covariance(*args, **kw)
    bad = poses.copy()
    bad[2, 4] = np.nan
    with pytest.raises(ValueError, match="not finite"):
        mcc.calibration_covariance(sc.uvs, ext, intr, sc.objpoints, bad)
    with pytest.raises(ValueError):
        mcc.calibration_covariance(sc.uvs, ext, intr, sc.objpoints, poses[:5])


# ------------------------------------------------------------------ GPU
def _scene(C, F, p=0.2, seed=0, corners=0.0, sigma=0.5):
    sc = make_scene(C, F, sigma=sigma, p_missing_view=p, p_missing_corner=corners, seed=seed)
    return sc.uvs, sc.objpoints, sc.x0()


def _outliers():
    sc = make_scene(6, 3000, sigma=0.4, p_missing_view=0.2, seed=32)
    uvs = sc.uvs.copy()
    rng = np.random.default_rng(32)
    bad = rng.choice(3000, 60, replace=False)
    uvs[:, bad] += (10.0 ** rng.uniform(3, 5, 60))[None, :, None, None] * rng.choice([-1.0, 1.0], (1, 60, 1, 2))
    return uvs, sc.objpoints, sc.x0()


def _no_cam2():
    uvs, obj, x = _scene(6, 50000)
    uvs[2] = np.nan
    return uvs, obj, x


# name -> (builder, loss, f_scale, reference camera)
PARITY = {
    "bench_6x50000": (lambda: _scene(6, 50000), "soft_l1", 1.0, 0),
    "6x50000_no_cam2": (_no_cam2, "soft_l1", 1.0, 0),
    "1x40000": (lambda: _scene(1, 40000, p=0.0, seed=8), "soft_l1", 1.0, 0),
    "16x8000": (lambda: _scene(16, 8000, seed=16), "soft_l1", 1.0, 0),
    "32x2000": (lambda: _scene(32, 2000, seed=19), "soft_l1", 1.0, 5),
    "6x3000_outliers_linear": (_outliers, "linear", 1.0, 0),
    "6x3000_outliers_fs0.25": (_outliers, "soft_l1", 0.25, 0),
    "6x8000_corners30": (lambda: _scene(6, 8000, seed=1, corners=0.3), "soft_l1", 1.0, 0),
    "6x8000_ref3": (lambda: _scene(6, 8000, seed=4), "soft_l1", 1.0, 3),
}


# The reference forms scipy's Gauss-Newton weight as rho' + 2 rho'' z = (1+z)^-1/2 - z (1+z)^-3/2, which loses
# log10(z) digits; the engine evaluates (1+z)^-3/2 directly (mcba_math.cuh).  At f_scale 0.25 the outlier corners
# reach z ~ 1e11, and the pose blocks of the frames they dominate differ by 6e-7 between the two -- the same amount
# by which the reference itself moves when only its weight is evaluated as (1+z)^-3/2.
POSE_TOL = {"6x3000_outliers_fs0.25": 1e-6}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PARITY))
def test_covariance_matches_blockwise_reference(name):
    fn, loss, f_scale, ref = PARITY[name]
    uvs, obj, x = fn()
    uvs = np.ascontiguousarray(uvs)
    prob = mcc.BAProblem(uvs, obj)
    cam, poses, info = prob.covariance(x, reference_camera=ref, loss=loss, f_scale=f_scale)
    want = ocov.blockwise_covariance(x, uvs, obj, ref, loss, f_scale)
    e_cam = _normalised_diff(cam, want["camera"])
    e_pose = _normalised_diff(poses, want["poses"])
    print(f"\n{name}: camera {e_cam:.2e}  poses {e_pose:.2e}  s2 {info['sigma2']:.6g}  cond(scaled camera system) "
          f"{_cond_scaled(want['camera']):.3e}  device ms eval {info['eval_ms']:.3f} camera {info['camera_ms']:.3f} "
          f"poses {info['pose_ms']:.3f}")
    tol = max(1e-7, 1e-13 * _cond_scaled(want["camera"]))   # rounding of S times the conditioning
    assert e_cam <= tol and e_pose <= POSE_TOL.get(name, tol)
    assert abs(info["sigma2"] - want["sigma2"]) <= 1e-12 * want["sigma2"]
    assert info["n_residuals"] == want["m"] and info["dof"] == want["dof"]
    assert info["empty_frames"] == want["empty_frames"]
    g = slice(12 * ref + 6, 12 * ref + 12)
    assert (cam[g][~np.isnan(cam[g])] == 0).all() and (cam[:, g][~np.isnan(cam[:, g])] == 0).all()
    unobs = np.isnan(uvs).all(axis=(1, 2, 3))
    assert np.isnan(cam[np.repeat(unobs, 12)]).all()
    assert np.isnan(np.diag(cam)).sum() == 12 * unobs.sum()
    empty = np.isnan(uvs).all(axis=(0, 2, 3))
    assert np.isnan(poses[empty]).all() and not np.isnan(poses[~empty]).any()
    prob.close()


def _align_to_reference(x, x_true, C, ref=0):
    """Rigid change of world frame that puts camera ``ref`` at its true extrinsics."""
    cams = x[:12 * C].reshape(C, 12).copy()
    poses = x[12 * C:].reshape(-1, 6).copy()
    tc = x_true[:12 * C].reshape(C, 12)[ref]
    R0, R0t = orc.rodrigues(cams[ref, 6:9]), orc.rodrigues(tc[6:9])
    A = R0t.T @ R0
    a = R0t.T @ (cams[ref, 9:12] - tc[9:12])
    for c in range(C):
        Rc = orc.rodrigues(cams[c, 6:9]) @ A.T
        cams[c, 9:12] = cams[c, 9:12] - Rc @ a
        cams[c, 6:9] = orc.rodrigues_inv(Rc)
    Rf = np.einsum("ij,fjk->fik", A, orc.rodrigues(poses[:, :3]))
    poses[:, 3:] = poses[:, 3:] @ A.T + a
    poses[:, :3] = orc.rodrigues_inv(Rf)
    return np.concatenate([cams.ravel(), poses.ravel()])


@pytest.mark.gpu
def test_covariance_predicts_the_scatter_of_solutions():
    """Linear loss, 6 cameras x 300 frames, sigma = 0.5 px, 64 seeded noise draws solved from the truth."""
    C, F, sigma = 6, 300, 0.5
    sc = make_scene(C, F, sigma=sigma, p_missing_view=0.2, seed=11)
    from multicam_calibration_b200.synthetic import forward_model
    x_true = np.concatenate([sc.true_cams.ravel(), sc.true_poses.ravel()])
    clean = forward_model(sc.true_cams, sc.true_poses, sc.objpoints)
    miss = np.isnan(sc.uvs)
    prob = mcc.BAProblem(np.where(miss, np.nan, clean), sc.objpoints)
    cam, poses, _ = prob.covariance(x_true, loss="linear", sigma=sigma)
    free = ~np.isclose(np.diag(cam), 0.0) & np.isfinite(np.diag(cam))
    cam_inv = np.linalg.inv(cam[np.ix_(free, free)])
    pose_inv = np.linalg.inv(poses)
    d_cam, d_pose, s2 = [], [], []
    rng = np.random.default_rng(12)
    for _ in range(64):
        uvs = np.where(miss, np.nan, clean + rng.normal(0, sigma, clean.shape))
        prob.set_observations(uvs)
        x, res = prob.solve(x_true, loss="linear", ftol=1e-14, xtol=1e-14, gtol=1e-12, max_nfev=100, verbose=0)
        xa = _align_to_reference(x, x_true, C)
        e = (xa - x_true)[:12 * C][free]
        d_cam.append(e @ cam_inv @ e / free.sum())
        ep = (xa - x_true)[12 * C:].reshape(F, 6)
        d_pose.append(np.einsum("fi,fij,fj->", ep, pose_inv, ep) / (6 * F))
        s2.append(2 * res.cost / (res.n_residuals - (12 * C + 6 * F - 6)))
    print(f"\nMahalanobis^2 per dimension: cameras {np.mean(d_cam):.4f} ({free.sum()} parameters), poses "
          f"{np.mean(d_pose):.4f}; mean s2 {np.mean(s2):.5f}")
    assert free.sum() == 66
    assert 0.85 <= np.mean(d_cam) <= 1.15
    assert 0.9 <= np.mean(d_pose) <= 1.1
    assert abs(np.mean(s2) - sigma ** 2) <= 0.03 * sigma ** 2


@pytest.mark.gpu
def test_handle_state_after_covariance():
    uvs, obj, x0 = _scene(6, 2000, seed=2)
    a, b = mcc.BAProblem(uvs, obj), mcc.BAProblem(uvs, obj)
    a.build_reduced(x0, lam=1e-3)
    b.build_reduced(x0, lam=1e-3)
    a.covariance(x0)
    Sa = a.build_reduced(x0, lam=1e-3)
    Sb = b.build_reduced(x0, lam=1e-3)
    for u, v in zip(Sa, Sb):
        assert np.array_equal(u, v)
    a.covariance(x0, loss="linear")
    xa, ra = a.solve(x0, verbose=0)
    xb, rb = mcc.BAProblem(uvs, obj).solve(x0, verbose=0)
    assert np.array_equal(xa, xb) and ra.nfev == rb.nfev


@pytest.mark.gpu
def test_covariance_after_pipelined_host_call():
    import torch
    from multicam_calibration_b200 import _native
    uvs, obj, x0 = _scene(6, 20000, seed=3)
    prob = mcc.BAProblem(uvs, obj)
    h_uvs = torch.from_numpy(np.ascontiguousarray(uvs)).pin_memory()
    h_x = torch.from_numpy(np.ascontiguousarray(x0)).pin_memory()
    h_obj = np.ascontiguousarray(obj)
    nc = 72
    S, bb, cost = np.empty((nc, nc)), np.empty(nc), ctypes.c_double()
    _native.check(prob.lib.mcba_build_reduced_host(
        prob._h, ctypes.c_void_p(h_uvs.data_ptr()), h_obj.ctypes.data_as(ctypes.c_void_p),
        ctypes.c_void_p(h_x.data_ptr()), 1e-3, 1, 1.0, S.ctypes.data_as(ctypes.c_void_p),
        bb.ctypes.data_as(ctypes.c_void_p), ctypes.cast(ctypes.byref(cost), ctypes.c_void_p)))
    cam, poses, info = prob.covariance(x0)
    cam2, poses2, info2 = mcc.BAProblem(uvs, obj).covariance(x0)
    assert _normalised_diff(cam, cam2) <= 1e-12 and _normalised_diff(poses, poses2) <= 1e-12
    assert info["sigma2"] == pytest.approx(info2["sigma2"], rel=1e-13)


@pytest.mark.gpu
def test_covariance_errors():
    uvs, obj, x = _scene(6, 200, seed=4, p=0.0)
    two = uvs.copy()
    two[:, 17] = np.nan
    two[0, 17, :2] = uvs[0, 17, :2]
    with pytest.raises(np.linalg.LinAlgError, match="1 frame"):
        mcc.BAProblem(two, obj).covariance(x)
    one = uvs.copy()
    one[2] = np.nan
    one[2, 5, 0] = uvs[2, 5, 0]
    with pytest.raises(np.linalg.LinAlgError, match="camera system"):
        mcc.BAProblem(one, obj).covariance(x)
    none = uvs.copy()
    none[0] = np.nan
    with pytest.raises(ValueError, match="no observations"):
        mcc.BAProblem(none, obj).covariance(x, reference_camera=0)
    bad = x.copy()
    bad[-1] = np.nan
    with pytest.raises(ValueError, match="not finite"):
        mcc.BAProblem(uvs, obj).covariance(bad)


@pytest.mark.gpu
def test_calibration_covariance_end_to_end():
    sc = make_scene(6, 500, sigma=0.3, p_missing_view=0.2, seed=7)
    ext, intr, poses = orc.deserialize_params(sc.x0(), 6)
    np.random.seed(0)
    e, i, p, use, res = mcc.bundle_adjust(sc.uvs, ext, intr, sc.objpoints, poses, n_frames=None, verbose=0)
    cov = mcc.calibration_covariance(sc.uvs[:, use], e, i, sc.objpoints, p)
    std = cov.camera_std
    assert std.shape == (6, 12) and cov.poses.shape == (len(use), 6, 6) and cov.pose_std.shape == (len(use), 6)
    assert (std[0, 6:] == 0).all()
    mask = np.ones_like(std, dtype=bool)
    mask[0, 6:] = False
    assert np.isfinite(std).all() and (std[mask] > 0).all()
    assert np.isfinite(cov.pose_std).all() and (cov.pose_std > 0).all()
    assert cov.dof > 0 and 0.05 < cov.sigma2 < 0.2
