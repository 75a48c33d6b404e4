"""point_covariance: the calibration's uncertainty carried into refined 3D points (k9_refine.cu).

CPU: the numpy reference (``tests/point_covariance_reference.py``) against its definition -- its sensitivity
dX/dtheta against central differences of per-point scipy re-solves with one camera parameter perturbed, its
camera Jacobian (with skew) against finite differences of the projection -- and the argument validation.
GPU: the engine against the reference element-wise for every loss, both kernel instantiations and missing views;
its sensitivity against central differences of device re-solves; the predicted covariance against the scatter
of points refined through 256 noisy calibrations; edge cases; configs[4] in full.
"""
import numpy as np
import pytest
from scipy.optimize import least_squares

from oracle import np_oracle as orc
import point_covariance_reference as pcr
import refine_reference as rr
import multicam_calibration_b200 as mcc
from multicam_calibration_b200.synthetic import forward_model, make_keypoints, make_scene

gpu = pytest.mark.gpu
F_SCALES = (0.5, 1.0, 3.0)
TIGHT = dict(ftol=1e-15, xtol=1e-15, gtol=1e-12, max_iter=1000)
# calibration-like standard deviations of fx fy cx cy k1 k2 rvec tvec (px, px, px, px, 1, 1, rad, mm): the scale of
# each parameter in a rig's covariance.  Finite-difference steps and sensitivity errors are measured in these units,
# so a parameter whose column of S is nearly zero for some point (k2 near the image centre) is judged by what it
# contributes to S cov S^T, not by its own size.
STD = np.array([2.0, 2.0, 1.0, 1.0, 2e-3, 1e-3, 1e-3, 1e-3, 1e-3, 0.5, 0.5, 0.5])


def scene(n, C=6, sigma=0.3, p_missing=0.2, seed=0):
    all_uvs, ext, intr, truth = make_keypoints(n, C, sigma=sigma, p_missing=p_missing, seed=seed)
    return np.stack(all_uvs), np.asarray(ext), intr, truth


def perturbed(ext, intr, c, k, eps):
    """The rig with parameter k (serialize_params order) of camera c moved by eps; K's skew kept."""
    ext = np.array(ext, dtype=float)
    intr = [(np.array(K, dtype=float), np.array(d, dtype=float)) for K, d in intr]
    K, d = intr[c]
    if k < 4:
        K[[0, 1, 0, 1][k], [0, 1, 2, 2][k]] += eps
    elif k < 6:
        d[k - 4] += eps
    else:
        ext[c, k - 6] += eps
    return ext, intr


def step(ext, intr, c, k):
    """1 / 100 of the parameter's scale: about 0.01 px on the image for every parameter."""
    return 1e-2 * STD[k]


def scipy_point(uvs, ext, intr, p, x0, loss, f_scale):
    """Per-point trf solve of point p over its seen views, at tight tolerances, then three IRLS Gauss-Newton steps
    (trf stops where a step no longer lowers the cost by ftol relative; these take X to the minimum's last bits)."""
    E, Ks, D = rr.rig(ext, intr)
    s = rr.seen_views(uvs, Ks, D)[:, p]
    u = uvs[s][:, p:p + 1]

    def fun(x):
        return rr.residuals(x[None], u, E[s], Ks[s], D[s])[0][:, 0].ravel()

    def jac(x):
        return -rr.residuals(x[None], u, E[s], Ks[s], D[s])[1][:, 0].reshape(-1, 3)
    x = least_squares(fun, x0, jac=jac, method="trf", loss=loss, f_scale=f_scale, ftol=1e-15, xtol=1e-15,
                      gtol=1e-15, max_nfev=2000).x
    for _ in range(3):
        _, g, H = rr.normal_equations(x[None], u, np.ones(u.shape[:2], dtype=bool), E[s], Ks[s], D[s], loss, f_scale,
                                      "irls")
        x = x - np.linalg.solve(H[0], g[0])
    return x


def weighted_error(S, S_ref):
    """Per point and coordinate: the largest difference of S diag(STD) relative to the largest entry of
    S_ref diag(STD), over all parameters given ((P, 3, 12 n) or (P, 3, n, 12)); (P, 3)."""
    P = len(S_ref)
    A = S.reshape(P, 3, -1, 12) * STD
    B = S_ref.reshape(P, 3, -1, 12) * STD
    d = np.abs(A - B).max((2, 3))
    scale = np.abs(B).max((2, 3))
    return np.where(scale > 0, d / np.where(scale > 0, scale, 1.0), np.where(d > 0, np.inf, 0.0))


def fd_sensitivity(solve, ext, intr, cams, P):
    """Central differences of X(theta) for every parameter of the given cameras, (P, 3, len(cams), 12): the
    five-point stencil at h = STD / 100, whose O(h^4) truncation stays below the re-solves' own scatter."""
    out = np.empty((P, 3, len(cams), 12))
    for i, c in enumerate(cams):
        for k in range(12):
            h = step(ext, intr, c, k)
            X = {j: solve(*perturbed(ext, intr, c, k, j * h)) for j in (-2, -1, 1, 2)}
            out[:, :, i, k] = (X[-2] - 8 * X[-1] + 8 * X[1] - X[2]) / (12 * h)
    return out


# ------------------------------------------------------------------ CPU: the reference against its definition
def test_reference_camera_jacobian_with_skew_matches_finite_differences():
    uvs, ext, intr, X = scene(50, C=3, sigma=0.0, p_missing=0.0, seed=4)
    intr = [(K.copy(), d) for K, d in intr]
    intr[1][0][0, 1] = 3.5                       # skew on camera 1
    E, Ks, D = rr.rig(ext, intr)
    J = pcr.camera_jacobian(X, E, Ks, D)
    for c in range(3):
        for k in range(12):
            h = step(E, intr, c, k)
            ep, ip = perturbed(E, intr, c, k, h)
            em, im = perturbed(E, intr, c, k, -h)
            up = orc.project_points(X, ep[c], ip[c][0], ip[c][1][:2])
            um = orc.project_points(X, em[c], im[c][0], im[c][1][:2])
            fd = (up - um) / (2 * h)
            scale = np.abs(J[c, :, :, k]).max()
            assert np.abs(fd - J[c, :, :, k]).max() <= 1e-6 * scale, (c, k)


@pytest.mark.parametrize("loss", rr.LOSSES)
def test_reference_sensitivity_is_the_derivative_of_the_minimiser(loss):
    """Noise-free keypoints at a scipy minimiser: S equals central differences of scipy re-solves for all 12
    parameters of two cameras, to 1e-6 of the largest entry of S diag(STD) per point and coordinate.

    With sigma = 0.3 px the residuals are not zero and the Gauss-Newton S drops the f * d2f term.  Measured on this
    scene: 1.3e-3 to 1.4e-3 of S diag(STD) for every loss; the gap is bounded by 3e-3."""
    cams = (1, 3)
    for sigma in (0.0, 0.3):
        uvs, ext, intr, truth = scene(40, C=4, sigma=sigma, p_missing=0.0, seed=21)
        pts = np.arange(6)
        for f_scale in (1.0,) if sigma else F_SCALES:
            X = np.stack([scipy_point(uvs, ext, intr, p, truth[p], loss, f_scale) for p in pts])

            def solve(e, i):
                return np.stack([scipy_point(uvs, e, i, p, X[j], loss, f_scale) for j, p in enumerate(pts)])
            fd = fd_sensitivity(solve, ext, intr, cams, pts.size)
            S = pcr.sensitivity(X, uvs[:, pts], ext, intr, loss, f_scale)[0].reshape(pts.size, 3, 4, 12)
            err = weighted_error(S[:, :, list(cams)], fd).max()
            print(f"{loss} f_scale {f_scale} sigma {sigma}: largest gap of S to re-solves {err:.2g} of S diag(STD)")
            assert err <= (1e-6 if sigma == 0.0 else 3e-3)


def _args(C=3, P=5):
    uvs, ext, intr, X = scene(P, C=C, seed=1)
    return uvs, ext, intr, X, pcr.random_camera_covariance(C)


def test_argument_validation_without_cuda():
    uvs, ext, intr, X, cov = _args()
    call = mcc.point_covariance
    with pytest.raises(ValueError, match="all_uvs"):
        call(uvs[..., :1], ext, intr, X, cov)
    with pytest.raises(ValueError, match="all_extrinsics"):
        call(uvs, ext[:2], intr, X, cov)
    with pytest.raises(ValueError, match="all_intrinsics"):
        call(uvs, ext, intr[:2], X, cov)
    with pytest.raises(ValueError, match="points must be"):
        call(uvs, ext, intr, X[:3], cov)
    with pytest.raises(ValueError, match=r"\(36, 36\)"):
        call(uvs, ext, intr, X, cov[:24, :24])
    bad = cov.copy()
    bad[0, 5] += 0.1
    with pytest.raises(ValueError, match="not symmetric"):
        call(uvs, ext, intr, X, bad)
    bad = cov.copy()
    bad[3, 3] = -1.0
    with pytest.raises(ValueError, match="negative diagonal"):
        call(uvs, ext, intr, X, bad)
    bad = cov.copy()
    bad[2, 7] = bad[7, 2] = np.inf
    with pytest.raises(ValueError, match="finite numbers or NaN"):
        call(uvs, ext, intr, X, bad)
    with pytest.raises(ValueError, match="n_cameras"):
        u33, e33, i33, X33 = scene(4, C=33)
        call(u33, e33, i33, X33, np.zeros((396, 396)))
    for kw, msg in ((dict(loss="l2"), "loss must be one of"), (dict(loss=None), "loss must be one of"),
                    (dict(f_scale=0.0), "f_scale must be a finite number > 0"),
                    (dict(f_scale=np.inf), "f_scale must be a finite number > 0"),
                    (dict(sigma=-1.0), "sigma must be a finite number > 0"),
                    (dict(sigma=True), "sigma must be a finite number > 0")):
        with pytest.raises(ValueError, match=msg):
            call(uvs, ext, intr, X, cov, **kw)
        with pytest.raises(ValueError, match=msg):
            mcc.refine_points(uvs, ext, intr, **kw)


def test_point_covariance_without_cuda_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    uvs, ext, intr, X, cov = _args()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mcc.point_covariance(uvs, ext, intr, X, cov)


# ------------------------------------------------------------------ GPU
def check_against_reference(pc, uvs, ext, intr, X, cov, loss="linear", f_scale=1.0, sigma=1.0, tol=1e-10):
    """The same NaN pattern, total = measurement + calibration, and per point: calibration element-wise normalised
    by sqrt(C_ii C_jj), sensitivity by :func:`weighted_error`, measurement relative to its largest entry, each to
    ``tol``.  Two fp64 evaluations of H^-1 in a different order differ by up to cond(H) eps relative, so a point
    whose J~^T J~ is ill-conditioned is held to max(tol, 100 eps cond(H)) instead: robust losses weight a residual
    beyond f_scale down to scipy's floor eps, and a point left with one or two full-weight scalars has
    cond(H) ~ 1e16 and a covariance that fp64 does not determine.  Returns the largest normalised differences of
    calibration and sensitivity and the number of points held to the relaxed bound."""
    meas, cal, S = pcr.point_covariance(uvs, ext, intr, X, cov, loss, f_scale, sigma)
    assert np.array_equal(np.isnan(pc.calibration), np.isnan(cal))
    assert np.array_equal(np.isnan(pc.measurement), np.isnan(meas))
    assert np.array_equal(pc.total, pc.measurement + pc.calibration, equal_nan=True)
    live = np.isfinite(meas).all((1, 2))
    kappa = np.ones(len(meas))
    kappa[live] = np.linalg.cond(meas[live])
    bound = np.maximum(tol, 100 * rr.EPS * kappa)
    ok = np.isfinite(cal).all((1, 2))
    d = np.sqrt(np.einsum("pii->pi", cal[ok]))
    scale = d[:, :, None] * d[:, None, :]
    e_cal = (np.abs(pc.calibration[ok] - cal[ok]) / np.where(scale > 0, scale, 1.0)).max((1, 2))
    assert (e_cal <= bound[ok]).all(), np.flatnonzero(ok)[e_cal > bound[ok]]
    e_meas = np.abs(pc.measurement[live] - meas[live]).max((1, 2)) / np.abs(meas[live]).max((1, 2))
    assert (e_meas <= bound[live]).all(), np.flatnonzero(live)[e_meas > bound[live]]
    e_sens = np.zeros(0)
    if pc.sensitivity is not None:
        assert np.array_equal(np.isnan(pc.sensitivity), np.isnan(S))
        e_sens = weighted_error(pc.sensitivity[live], S[live]).max(1)
        assert (e_sens <= bound[live]).all(), np.flatnonzero(live)[e_sens > bound[live]]
    tight = bound == tol
    return (float(e_cal[tight[ok]].max(initial=0.0)), float(e_sens[tight[live]].max(initial=0.0)) if e_sens.size
            else 0.0, int((~tight & live).sum()))


@gpu
@pytest.mark.parametrize("loss", rr.LOSSES)
@pytest.mark.parametrize("f_scale", F_SCALES)
def test_matches_reference_for_every_loss(loss, f_scale):
    """6 cameras, 3,000 points, sigma 0.3 px, 20 % missing views, 10 % of the points with a 30 px outlier."""
    uvs, ext, intr, truth = scene(3000, seed=5)
    rng = np.random.default_rng(6)
    seen = ~np.isnan(uvs).any(-1)
    for p in np.flatnonzero((rng.random(uvs.shape[1]) < 0.1) & (seen.sum(0) >= 3)):
        uvs[rng.choice(np.flatnonzero(seen[:, p])), p] += 30.0
    res = mcc.refine_points(uvs, ext, intr, loss=loss, f_scale=f_scale, sigma=0.3)
    cov = pcr.random_camera_covariance(6, seed=7)
    pc = mcc.point_covariance(uvs, ext, intr, res.points, cov, loss=loss, f_scale=f_scale, sigma=0.3,
                              sensitivity=True)
    assert np.array_equal(pc.measurement, res.covariance, equal_nan=True)   # bit-identical
    e = check_against_reference(pc, uvs, ext, intr, res.points, cov, loss, f_scale, 0.3)
    print(f"{loss} f_scale {f_scale}: calibration {e[0]:.2g}, sensitivity {e[1]:.2g} (well-conditioned points); "
          f"{e[2]} points held to 100 eps cond(H)")


@gpu
@pytest.mark.parametrize("C", (2, 3, 8, 9, 16, 17, 32))
def test_matches_reference_at_every_camera_count(C):
    """Both kernel instantiations (<= 8 cameras with the covariance in shared memory, <= 32 through L2),
    20 % missing views, skew on one camera, a cauchy loss."""
    uvs, ext, intr, _ = scene(1500, C=C, seed=C)
    intr = [(K.copy(), d) for K, d in intr]
    intr[C - 1][0][0, 1] = 2.0
    res = mcc.refine_points(uvs, ext, intr, loss="cauchy", f_scale=2.0)
    cov = pcr.random_camera_covariance(C, seed=C)
    pc = mcc.point_covariance(uvs, ext, intr, res.points, cov, loss="cauchy", f_scale=2.0, sensitivity=True)
    assert np.array_equal(pc.measurement, res.covariance, equal_nan=True)
    assert pc.sensitivity.shape == (1500, 3, 12 * C)
    e = check_against_reference(pc, uvs, ext, intr, res.points, cov, "cauchy", 2.0)
    print(f"C = {C}: {np.isfinite(pc.calibration).all((1, 2)).sum()} finite points, calibration {e[0]:.2g}, "
          f"sensitivity {e[1]:.2g}; {e[2]} points held to 100 eps cond(H)")


@gpu
@pytest.mark.parametrize("loss", rr.LOSSES)
def test_sensitivity_is_the_derivative_of_device_resolves(loss):
    """Noise-free keypoints: the device S against central differences of refine_points re-run with one
    parameter of camera 0 or 2 perturbed (ftol = xtol = 1e-15, gtol = 0), to 1e-6 of S diag(STD).

    soft_l1 is held to 1e-5: its re-solves stop where their steps fall below xtol, up to 1e-8 mm short of the
    minimum (two starts 1e-6 mm apart end that far apart), and no step of the differences gets below 1.3e-6 --
    0.01 px leaves that stopping error, larger steps the loss's curvature.  The device S itself equals the
    reference's to 1e-12, and the reference's S equals differences of polished scipy re-solves to 1e-6 for every
    loss (test_reference_sensitivity_is_the_derivative_of_the_minimiser)."""
    uvs, ext, intr, truth = scene(300, sigma=0.0, p_missing=0.0, seed=9)
    X = mcc.refine_points(uvs, ext, intr, truth, loss=loss, **TIGHT).points

    def solve(e, i):
        return mcc.refine_points(uvs, e, i, X, loss=loss, ftol=1e-15, xtol=1e-15, gtol=0.0, max_iter=1000).points
    cams = (0, 2)
    fd = fd_sensitivity(solve, ext, intr, cams, len(X))
    cov = pcr.random_camera_covariance(6)
    S = mcc.point_covariance(uvs, ext, intr, X, cov, loss=loss, sensitivity=True).sensitivity
    err = weighted_error(S.reshape(len(X), 3, 6, 12)[:, :, list(cams)], fd).max()
    print(f"{loss}: largest gap of the device S to device re-solves {err:.2g} of S diag(STD)")
    assert err <= (1e-5 if loss == "soft_l1" else 1e-6)


@gpu
def test_predicts_the_scatter_of_points_through_noisy_calibrations():
    """6 cameras x 300 frames, sigma = 0.5 px, camera 0's extrinsics pinned at the truth, 256 noisy
    calibrations (the engine of bundle_adjust(fixed=...) and calibration_covariance(reference_camera=None,
    fixed=..., sigma=0.5)).  Per draw, 2,000 fixed keypoints projected through the true cameras are refined with
    the estimated cameras, from noise-free pixels and from fresh 0.5 px noise.  The mean Mahalanobis^2 per
    dimension of (points - truth) is 1 under pc.calibration for the former and under pc.total for the latter.

    Spread of the statistic: a draw's calibration error is shared by its 2,000 points, so a draw contributes one
    correlated sample.  If the points' errors were fully correlated the per-draw mean would be chi2_3 / 3 with
    variance 2/3, and the mean over 256 draws would have standard deviation sqrt(2 / (3 * 256)) = 0.051; the
    band [0.9, 1.1] is then two of those.  The measured per-draw spread, printed, is below that bound."""
    C, F, sigma, n_draws, P = 6, 300, 0.5, 256, 2000
    sc = make_scene(C, F, sigma=sigma, p_missing_view=0.2, seed=11)
    x_true = np.concatenate([sc.true_cams.ravel(), sc.true_poses.ravel()])
    clean = forward_model(sc.true_cams, sc.true_poses, sc.objpoints)
    miss = np.isnan(sc.uvs)
    fixed = np.zeros((C, 12), dtype=bool)
    fixed[0, 6:] = True
    rng = np.random.default_rng(13)
    truth = rng.normal(0, 80, (P, 3))
    ext_t, intr_t = sc._split(sc.true_cams)
    kp = np.stack([orc.project_points(truth, ext_t[c], intr_t[c][0], intr_t[c][1][:2]) for c in range(C)])
    prob = mcc.BAProblem(np.where(miss, np.nan, clean), sc.objpoints)
    stat = {"calibration": [], "total": [], "measurement": [], "measurement_clean": []}
    for _ in range(n_draws):
        prob.set_observations(np.where(miss, np.nan, clean + rng.normal(0, sigma, clean.shape)))
        x, _ = prob.solve(x_true, fixed=fixed, loss="linear", ftol=1e-14, xtol=1e-14, gtol=1e-12, max_nfev=100,
                          verbose=0)
        cam, _, _ = prob.covariance(x, reference_camera=None, loss="linear", sigma=sigma, fixed=fixed, poses=False)
        ext, intr = sc._split(x[:12 * C].reshape(C, 12))
        for uvs, key in ((kp, "calibration"), (kp + rng.normal(0, sigma, kp.shape), "total")):
            res = mcc.refine_points(uvs, ext, intr, truth, sigma=sigma, **TIGHT)
            pc = mcc.point_covariance(uvs, ext, intr, res.points, cam, sigma=sigma)
            e = res.points - truth
            m = lambda A: float(np.einsum("pi,pi->p", e, np.linalg.solve(A, e[..., None])[..., 0]).mean() / 3)  # noqa
            stat[key].append(m(getattr(pc, key)))
            stat["measurement" if key == "total" else "measurement_clean"].append(m(pc.measurement))
    mean = {k: float(np.mean(v)) for k, v in stat.items()}
    spread = {k: float(np.std(v) / np.sqrt(n_draws)) for k, v in stat.items()}
    print(f"\nMahalanobis^2 per dimension over {n_draws} draws x {P} points: "
          + ", ".join(f"{k} {mean[k]:.4f} (+- {spread[k]:.4f})" for k in stat)
          + f"; fully correlated bound of the spread {np.sqrt(2 / (3 * n_draws)):.4f}")
    assert 0.9 <= mean["calibration"] <= 1.1
    assert 0.9 <= mean["total"] <= 1.1
    assert mean["measurement"] > mean["total"]    # the pixel noise alone understates the error


@gpu
def test_edge_cases():
    uvs, ext, intr, _ = scene(2000, seed=15)
    uvs[:, :10] = np.nan
    uvs[1:, 10:20] = np.nan                         # one view: status -1
    res = mcc.refine_points(uvs, ext, intr)
    assert (res.status[:20] == -1).all()
    held = np.zeros((6, 12), dtype=bool)
    held[0, 6:] = True
    held[:, :2] = True                               # focal lengths held
    held[4] = True                                   # a camera held entirely
    cov = pcr.random_camera_covariance(6, seed=16, held=held, nan_cameras=(2,))
    pc = mcc.point_covariance(uvs, ext, intr, res.points, cov, sensitivity=True)
    for a in (pc.total, pc.measurement, pc.calibration, pc.sensitivity):
        assert np.isnan(a[:20]).all()
    seen2 = ~np.isnan(uvs[2]).any(-1)
    live = res.status > 0
    assert np.isnan(pc.calibration[live & seen2]).all() and np.isnan(pc.total[live & seen2]).all()
    assert np.isfinite(pc.calibration[live & ~seen2]).all() and np.isfinite(pc.measurement[live]).all()
    assert np.isfinite(pc.sensitivity[live]).all()
    check_against_reference(pc, uvs, ext, intr, res.points, cov)
    S = pc.sensitivity.reshape(-1, 3, 6, 12)
    assert (S[live & np.isnan(uvs[3]).any(-1)][:, :, 3] == 0).all()      # unseen camera: zero columns
    again = mcc.point_covariance(uvs, ext, intr, res.points, cov, sensitivity=True)
    for a, b in zip((pc.total, pc.measurement, pc.calibration, pc.sensitivity),
                    (again.total, again.measurement, again.calibration, again.sensitivity)):
        assert np.array_equal(a, b, equal_nan=True)
    cc = mcc.CalibrationCovariance(camera=cov, camera_std=None, poses=None, pose_std=None, sigma2=1.0, dof=1.0,
                                   n_residuals=1, cost=0.0)
    assert np.array_equal(mcc.point_covariance(uvs, ext, intr, res.points, cc).calibration, pc.calibration,
                          equal_nan=True)
    empty = mcc.point_covariance(uvs[:, :0], ext, intr, np.zeros((0, 3)), cov, sensitivity=True)
    assert empty.total.shape == (0, 3, 3) and empty.sensitivity.shape == (0, 3, 72)


@gpu
def test_configs4_in_full():
    """configs[4]: 1 M keypoints x 6 cameras, sigma 0.3 px, 20 % missing views."""
    uvs, ext, intr, _ = scene(1_000_000, seed=0)
    res = mcc.refine_points(uvs, ext, intr)
    cov = pcr.random_camera_covariance(6, seed=1)
    pc = mcc.point_covariance(uvs, ext, intr, res.points, cov, sensitivity=True)
    assert np.array_equal(pc.measurement, res.covariance, equal_nan=True)
    live = res.status > 0
    assert np.isfinite(pc.total[live]).all() and np.isfinite(pc.sensitivity[live]).all()
    sub = np.arange(0, len(res.points), 100)
    sub_pc = mcc.PointCovariance(pc.total[sub], pc.measurement[sub], pc.calibration[sub], pc.sensitivity[sub])
    e = check_against_reference(sub_pc, uvs[:, sub], ext, intr, res.points[sub], cov)
    print(f"configs[4]: {live.sum()} refined points, every 100th: calibration {e[0]:.2g}, sensitivity {e[1]:.2g}")
