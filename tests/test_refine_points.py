"""refine_points: per-point least-squares refinement of triangulated points (k9_refine.cu).

CPU: the numpy reference (``tests/refine_reference.py``) against scipy -- its losses against scipy's loss
functions, its minimiser against per-point ``least_squares(method="trf")`` with the analytic Jacobian, its
covariance against ``sigma^2 inv(res.jac.T res.jac)`` -- and the argument validation of the public call.
GPU: the engine against the reference at production size (configs[4]), with planted outliers for every
robust loss, at every template instantiation, on near-degenerate rigs and non-finite pixels, and the
covariance element-wise and statistically.
"""
import numpy as np
import pytest
from scipy.optimize import least_squares
from scipy.optimize._lsq.least_squares import construct_loss_function

from oracle import np_oracle as orc
import refine_reference as rr
import multicam_calibration_b200 as mcc
from multicam_calibration_b200.synthetic import make_keypoints

gpu = pytest.mark.gpu
F_SCALES = (0.5, 1.0, 3.0)
TIGHT = dict(ftol=1e-15, xtol=1e-15, gtol=1e-10, max_iter=1000)   # engine and reference run to the minimum


def scene(n, C=6, sigma=0.3, p_missing=0.2, seed=0):
    all_uvs, ext, intr, truth = make_keypoints(n, C, sigma=sigma, p_missing=p_missing, seed=seed)
    return np.stack(all_uvs), ext, intr, truth


def plant_outliers(uvs, frac=0.1, shift=30.0, seed=7):
    """Displace one seen view of ``frac`` of the points by ``shift`` px; returns (uvs, points, cameras)."""
    rng = np.random.default_rng(seed)
    uvs = uvs.copy()
    seen = ~np.isnan(uvs).any(-1)
    pts = np.flatnonzero((rng.random(uvs.shape[1]) < frac) & (seen.sum(0) >= 3))
    cams = np.array([rng.choice(np.flatnonzero(seen[:, p])) for p in pts], dtype=int)
    ang = rng.uniform(0, 2 * np.pi, pts.size)
    uvs[cams, pts] += shift * np.stack([np.cos(ang), np.sin(ang)], -1)
    return uvs, pts, cams


def point_problem(uvs, ext, Ks, dists, seen, p):
    """scipy's view of point p: residual and analytic Jacobian of its seen views."""
    s = seen[:, p]
    u = uvs[s][:, p:p + 1]

    def fun(x):
        return rr.residuals(x[None], u, ext[s], Ks[s], dists[s])[0][:, 0].ravel()

    def jac(x):
        return -rr.residuals(x[None], u, ext[s], Ks[s], dists[s])[1][:, 0].reshape(-1, 3)
    return fun, jac


def match_or_better(X, cost, X_ref, cost_ref, rel=None, atol=None, H=None, px=1e-6):
    """Per point: X matches X_ref (relative to |X_ref| or absolutely, or -- given H = J~^T J~ at X_ref -- moves the
    scaled residuals by at most ``px`` pixels, sqrt(d^T H d): where the cost surface is flat, two fp64 runs whose
    starts differ by 1e-15 relative already stop up to ~1e-7 mm and ~3e-7 px apart), or X ends at a different
    local minimum whose cost is not above cost_ref.  Returns (ok mask, mask of points beyond the tolerance in mm,
    largest difference within it, largest residual change of the points judged the same)."""
    d = X - X_ref
    dm = np.abs(d).max(1)
    tol = rel * np.abs(X_ref).max(1) if rel is not None else atol
    same = dm <= tol
    move = np.zeros(len(X)) if H is None else np.sqrt(np.abs(np.einsum("pi,pij,pj->p", d, H, d)))
    if H is not None:
        same |= move <= px
    better = cost <= cost_ref * (1 + 1e-12) + 1e-300
    return same | better, dm > tol, float(dm[dm <= tol].max(initial=0.0)), float(move[same].max(initial=0.0))


# ------------------------------------------------------------------ CPU: reference against scipy
@pytest.mark.parametrize("loss", rr.LOSSES)
@pytest.mark.parametrize("f_scale", F_SCALES)
def test_reference_losses_match_scipy(loss, f_scale):
    f = np.concatenate([np.linspace(-40, 40, 801), [0.0, 1e-8, f_scale, -f_scale, 1e4]])
    rho, r1, r2 = rr.loss_rho(f, loss, f_scale)
    if loss == "linear":
        np.testing.assert_allclose(rho, f * f, rtol=4e-16)   # scipy's linear loss is rho(z) = z
        np.testing.assert_array_equal(r1, 1.0)
        np.testing.assert_array_equal(r2, 0.0)
        return
    ref = construct_loss_function(f.size, loss, f_scale)(f)
    for mine, theirs in zip((rho, r1, r2), ref):
        np.testing.assert_allclose(mine, theirs, rtol=4e-16, atol=1e-300)


@pytest.mark.parametrize("loss", rr.LOSSES)
def test_reference_minimiser_matches_scipy(loss):
    """~300 points x f_scale 0.5 / 1 / 3: the reference's minimiser against per-point trf with the
    analytic Jacobian, both at tight tolerances; 1e-9 relative where they end at the same minimum, and the
    reference's cost not above scipy's where they end at different ones."""
    uvs, ext, intr, _ = scene(300, seed=11)
    E, Ks, D = rr.rig(ext, intr)
    seen = rr.seen_views(uvs, Ks, D)
    X0 = orc.triangulate(list(uvs), list(ext), intr)
    tight = dict(ftol=1e-15, xtol=1e-15, gtol=1e-13)
    for f_scale in F_SCALES:
        X, status, iters, cost = rr.refine(uvs, ext, intr, X0, loss=loss, f_scale=f_scale, max_iter=1000, **tight)
        live = status >= 0
        assert np.array_equal(live, seen.sum(0) >= 2) and (status[live] > 0).all()
        Xs = np.full_like(X, np.nan)
        cs = np.full(len(X), np.nan)
        conv = np.zeros(len(X), dtype=bool)
        for p in np.flatnonzero(live):
            fun, jac = point_problem(uvs, E, Ks, D, seen, p)
            r = least_squares(fun, X0[p], jac=jac, method="trf", loss=loss, f_scale=f_scale, max_nfev=2000, **tight)
            Xs[p], cs[p], conv[p] = r.x, r.cost, r.status > 0
        ok, differ, worst, _ = match_or_better(X[conv], cost[conv], Xs[conv], cs[conv], rel=1e-9)
        print(f"{loss} f_scale {f_scale}: {conv.sum()} points, largest matched difference {worst:.2g} mm (tolerance "
              f"1e-9 |x|), {differ.sum()} beyond it (a different minimum, cost not above scipy's), "
              f"mean / max iterations "
              f"{iters[live].mean():.1f} / {iters.max()}")
        assert ok.all(), np.flatnonzero(conv)[~ok]


@pytest.mark.parametrize("loss", rr.LOSSES)
def test_reference_covariance_matches_scipy_jac(loss):
    uvs, ext, intr, _ = scene(60, seed=12)
    uvs, _, _ = plant_outliers(uvs, frac=0.3)
    E, Ks, D = rr.rig(ext, intr)
    seen = rr.seen_views(uvs, Ks, D)
    X0 = orc.triangulate(list(uvs), list(ext), intr)
    worst = 0.0
    for p in np.flatnonzero(seen.sum(0) >= 2):
        fun, jac = point_problem(uvs, E, Ks, D, seen, p)
        r = least_squares(fun, X0[p], jac=jac, method="trf", loss=loss, f_scale=1.5)
        ref = 0.49 * np.linalg.inv(r.jac.T @ r.jac)
        mine = rr.covariance(r.x[None], uvs[:, p:p + 1], seen[:, p:p + 1], E, Ks, D, loss, 1.5, sigma=0.7)[0]
        worst = max(worst, np.abs(mine - ref).max() / np.abs(ref).max())
    print(f"{loss}: largest covariance difference {worst:.2g} relative")
    assert worst <= 1e-10


# ------------------------------------------------------------------ CPU: argument validation
def _args(C=3, P=4):
    uvs, ext, intr, _ = scene(P, C=C, p_missing=0.0, seed=1)
    return uvs, ext, intr


@pytest.mark.parametrize("kwargs, match", [
    (dict(loss="l2"), "loss"), (dict(loss=lambda z: z), "loss"), (dict(loss=None), "loss"),
    (dict(f_scale=0.0), "f_scale"), (dict(f_scale=-1.0), "f_scale"), (dict(f_scale=np.nan), "f_scale"),
    (dict(sigma=0.0), "sigma"), (dict(sigma=np.inf), "sigma"),
    (dict(max_iter=0), "max_iter"), (dict(max_iter=2.5), "max_iter"), (dict(max_iter=40000), "max_iter"),
    (dict(ftol=-1.0), "ftol"), (dict(xtol=np.nan), "xtol"), (dict(gtol="1"), "gtol"),
])
def test_refine_points_rejects_bad_options(kwargs, match):
    uvs, ext, intr = _args()
    with pytest.raises(ValueError, match=match):
        mcc.refine_points(uvs, ext, intr, **kwargs)


def test_refine_points_rejects_bad_shapes():
    uvs, ext, intr = _args()
    bad = [
        ((uvs[..., :1], ext, intr), "all_uvs"),
        ((uvs[0], ext, intr), "all_uvs"),
        ((uvs.astype(complex), ext, intr), "real"),
        ((uvs, ext[:2], intr), "all_extrinsics"),
        ((uvs, ext, intr[:2]), "all_intrinsics"),
        ((uvs, ext, [(np.eye(2), d) for _, d in intr]), "camera_matrix"),
        ((uvs, ext, [(K, np.zeros(1)) for K, _ in intr]), "dist_coefs"),
        ((uvs, ext, intr, np.zeros((3, 3))), "points"),
        ((uvs, ext, intr, np.zeros((4, 2))), "points"),
        ((np.zeros((0, 4, 2)), ext[:0], []), "n_cameras"),
    ]
    for args, match in bad:
        with pytest.raises(ValueError, match=match):
            mcc.refine_points(*args)
    uvs33, ext33, intr33 = _args(C=33, P=2)
    with pytest.raises(ValueError, match="n_cameras"):
        mcc.refine_points(uvs33, ext33, intr33)


def test_refine_points_without_cuda_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    uvs, ext, intr = _args()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mcc.refine_points(uvs, ext, intr)


# ------------------------------------------------------------------ GPU
def _ref_at(uvs, ext, intr, X0, idx, **kw):
    return rr.refine(uvs[:, idx], ext, intr, X0[idx], **kw)


@gpu
def test_noise_free_recovers_truth():
    uvs, ext, intr, truth = scene(20000, sigma=0.0, seed=21)
    res = mcc.refine_points(uvs, ext, intr)
    live = res.status >= 0
    assert np.array_equal(live, res.n_views >= 2)
    err = np.abs(res.points[live] - truth[live]).max()
    rng = np.random.default_rng(3)
    start = truth + rng.normal(0, 5 / np.sqrt(3), truth.shape)
    res2 = mcc.refine_points(uvs, ext, intr, start)
    err2 = np.abs(res2.points[live] - truth[live]).max()
    print(f"sigma = 0: largest error {err:.2g} mm from the triangulation, {err2:.2g} mm from 5 mm starts")
    assert err <= 1e-9 and err2 <= 1e-9
    assert (res.status[live] > 0).all() and (res2.status[live] > 0).all()


@gpu
def test_configs4_full_workload_linear():
    """1 M points x 6 cameras, sigma 0.3 px, 20 % missing views: the benchmark's triangulation workload."""
    all_uvs, ext, intr, truth = make_keypoints(1_000_000, 6, sigma=0.3, p_missing=0.2, seed=0)
    uvs = np.stack(all_uvs)
    tri = mcc.triangulate(all_uvs, list(ext), intr)
    res = mcc.refine_points(all_uvs, ext, intr, view_errors=True)
    assert np.array_equal(res.status == -1, np.isnan(tri).any(1))
    assert np.isnan(res.points[res.status == -1]).all()
    live = res.status >= 0
    E, Ks, D = rr.rig(ext, intr)
    seen = rr.seen_views(uvs, Ks, D)
    assert np.array_equal(res.n_views, seen.sum(0))
    assert np.array_equal(np.isnan(res.view_errors), ~seen | ~live[None])
    # cost at the DLT median, by the reference
    c0 = np.full(len(tri), np.nan)
    c0[live] = rr.cost_only(tri[live], uvs[:, live], seen[:, live], E, Ks, D, "linear", 1.0)
    assert (res.cost[live] <= c0[live] * (1 + 1e-12)).all()
    rms0 = np.sqrt(2 * c0[live] / (2 * res.n_views[live]))
    # every 10th point against the reference, both run to the minimum (TIGHT): with the default ftol the two
    # may stop one step apart, which moves a point by up to ~1e-7 mm while its cost differs by < ftol * cost
    idx = np.flatnonzero(live)[::10]
    tight = mcc.refine_points(all_uvs, ext, intr, covariance=False, **TIGHT)
    Xr, sr, ir, cr = _ref_at(uvs, ext, intr, tri, idx, **TIGHT)
    _, _, Hr = rr.normal_equations(Xr, uvs[:, idx], seen[:, idx], E, Ks, D, "linear", 1.0)
    ok, differ, worst, move = match_or_better(tight.points[idx], tight.cost[idx], Xr, cr, atol=1e-8, H=Hr)
    # the gradient at the result, by the reference
    _, g, _ = rr.normal_equations(tight.points[idx], uvs[:, idx], seen[:, idx], E, Ks, D, "linear", 1.0)
    gmax = np.abs(g).max(1)
    g1 = tight.status[idx] == 1
    hist = {int(k): int(v) for k, v in zip(*np.unique(res.status, return_counts=True))}
    hist_t = {int(k): int(v) for k, v in zip(*np.unique(tight.status, return_counts=True))}
    print(f"configs[4]: status histogram {hist}; mean RMS {rms0.mean():.6f} px at the DLT median -> "
          f"{res.rms[live].mean():.6f} px refined; iterations mean {res.iterations[live].mean():.2f} max "
          f"{res.iterations.max()}; tight run: status histogram {hist_t}, largest matched difference to the "
          f"reference {worst:.2g} mm on {idx.size} points, {differ.sum()} beyond 1e-8 mm, residual change "
          f"up to {move:.2g} px, {(~ok).sum()} failing; largest |g| "
          f"{gmax[g1].max(initial=0):.2g} where gtol ended the iteration, {gmax[~g1].max(initial=0):.2g} elsewhere")
    assert ok.all()
    assert gmax[g1].max(initial=0) <= 2 * TIGHT["gtol"]


@gpu
@pytest.mark.parametrize("loss", rr.LOSSES[1:])
def test_planted_outliers_robust_losses(loss):
    uvs, ext, intr, truth = scene(20000, seed=31)
    uvs, pts, cams = plant_outliers(uvs)
    tri = mcc.triangulate(list(uvs), list(ext), intr)
    res = mcc.refine_points(uvs, ext, intr, loss=loss, view_errors=True)
    lin = mcc.refine_points(uvs, ext, intr, loss="linear")
    live = res.status >= 0
    idx = np.flatnonzero(live)[::4]
    tight = mcc.refine_points(uvs, ext, intr, loss=loss, covariance=False, **TIGHT)
    Xr, sr, ir, cr = _ref_at(uvs, ext, intr, tri, idx, loss=loss, **TIGHT)
    E, Ks, D = rr.rig(ext, intr)
    seen = rr.seen_views(uvs, Ks, D)
    _, _, Hr = rr.normal_equations(Xr, uvs[:, idx], seen[:, idx], E, Ks, D, loss, 1.0)
    ok, differ, worst, move = match_or_better(tight.points[idx], tight.cost[idx], Xr, cr, atol=1e-8, H=Hr)
    err = np.linalg.norm(res.points[pts] - truth[pts], axis=1)
    err_lin = np.linalg.norm(lin.points[pts] - truth[pts], axis=1)
    single = np.mean(np.nanargmax(res.view_errors[:, pts], axis=0) == cams)
    print(f"{loss}: {idx.size} points against the reference, largest matched difference {worst:.2g} mm, "
          f"{differ.sum()} beyond 1e-8 mm (residual change up to {move:.2g} px, {(~ok).sum()} failing); median "
          f"distance to the truth on the {pts.size} displaced "
          f"points {np.median(err):.4f} mm ({np.median(err_lin):.4f} linear); displaced view singled out on "
          f"{single:.1%}; iterations mean {res.iterations[live].mean():.2f} max {res.iterations.max()}")
    assert ok.all()
    if loss in ("huber", "soft_l1", "cauchy"):
        assert np.median(err) < np.median(err_lin)
    if loss == "cauchy":
        assert single >= 0.95


@gpu
@pytest.mark.parametrize("C", [2, 3, 8, 9, 16, 17, 32])
def test_camera_counts(C):
    """C <= 8 runs refine_points_kernel<8> (observations in registers), 9..32 refine_points_kernel<32>."""
    n = 4000 if C >= 16 else 10000
    uvs, ext, intr, _ = scene(n, C=C, p_missing=0.3, seed=40 + C)
    res = mcc.refine_points(uvs, ext, intr, loss="soft_l1", covariance=True, **TIGHT)
    tri = mcc.triangulate(list(uvs), list(ext), intr)
    Xr, sr, ir, cr = rr.refine(uvs, ext, intr, tri, loss="soft_l1", **TIGHT)
    live = sr >= 0
    assert np.array_equal(res.status < 0, sr < 0)
    E, Ks, D = rr.rig(ext, intr)
    seen = rr.seen_views(uvs, Ks, D)
    _, _, Hr = rr.normal_equations(Xr[live], uvs[:, live], seen[:, live], E, Ks, D, "soft_l1", 1.0)
    ok, differ, worst, move = match_or_better(res.points[live], res.cost[live], Xr[live], cr[live], atol=1e-8, H=Hr)
    cov = rr.covariance(res.points[live], uvs[:, live], seen[:, live], E, Ks, D, "soft_l1", 1.0)
    dc = np.abs(res.covariance[live] - cov).max((1, 2)) / np.abs(cov).max((1, 2))
    print(f"{C} cameras: largest matched difference {worst:.2g} mm, {differ.sum()} of {live.sum()} beyond 1e-8 mm "
          f"(residual change up to {move:.2g} px, {(~ok).sum()} failing), covariance {dc.max():.2g} relative")
    assert ok.all() and dc.max() <= 1e-10


@gpu
def test_rejects_33_cameras():
    uvs, ext, intr, _ = scene(10, C=33, p_missing=0.0, seed=1)
    with pytest.raises(ValueError, match="n_cameras"):
        mcc.refine_points(uvs, ext, intr)


@gpu
def test_short_baseline_pair():
    """Two cameras 0.5 mm apart: a nearly singular depth.  No NaN where the start is finite, and a point
    that cannot be refined reports -2 with its start."""
    uvs, ext, intr, _ = scene(20000, C=2, p_missing=0.0, seed=50)
    ext = ext.copy()
    ext[1] = ext[0]
    ext[1, 3] += 0.5
    rng = np.random.default_rng(5)
    pts = rng.normal(0, 80, (20000, 3))
    uvs = np.stack([orc.project_points(pts, ext[c], intr[c][0], intr[c][1][:2]) for c in range(2)])
    uvs += rng.normal(0, 0.3, uvs.shape)
    tri = mcc.triangulate(list(uvs), list(ext), intr)
    res = mcc.refine_points(uvs, ext, intr)
    fin = np.isfinite(tri).all(1)
    assert not np.isnan(res.points[fin]).any()
    assert np.isin(res.status, [-2, 0, 1, 2, 3, 4]).all()
    m2 = res.status == -2
    np.testing.assert_array_equal(res.points[m2], tri[m2])
    print(f"0.5 mm baseline: status {dict(zip(*np.unique(res.status, return_counts=True)))}")


@gpu
def test_non_finite_pixels_are_unseen():
    uvs, ext, intr, _ = scene(3000, C=4, p_missing=0.0, seed=60)
    rng = np.random.default_rng(1)
    bad = rng.random(uvs.shape[:2]) < 0.25
    vals = rng.choice([np.inf, -np.inf, 1e300, np.nan], size=bad.sum())
    coord = rng.integers(0, 2, bad.sum())
    c_idx, p_idx = np.nonzero(bad)
    uvs[c_idx, p_idx, coord] = vals
    res = mcc.refine_points(uvs, ext, intr, view_errors=True)
    clean = uvs.copy()
    clean[bad] = np.nan
    ref = mcc.refine_points(clean, ext, intr, view_errors=True)
    assert np.array_equal(res.n_views, (~bad).sum(0))
    np.testing.assert_array_equal(res.points, ref.points)
    np.testing.assert_array_equal(res.status, ref.status)
    np.testing.assert_array_equal(res.view_errors, ref.view_errors)


@gpu
def test_given_triangulation_and_repeat_are_bit_identical():
    uvs, ext, intr, _ = scene(50000, seed=70)
    a = mcc.refine_points(uvs, ext, intr, loss="cauchy", view_errors=True)
    b = mcc.refine_points(uvs, ext, intr, mcc.triangulate(list(uvs), list(ext), intr), loss="cauchy",
                          view_errors=True)
    c = mcc.refine_points(list(uvs), ext, intr, loss="cauchy", view_errors=True)
    for x, y in ((a, b), (a, c)):
        for f in a._fields:
            np.testing.assert_array_equal(getattr(x, f), getattr(y, f), err_msg=f)


@gpu
def test_covariance_against_reference_and_scatter():
    """Element-wise against the reference; then 64 noise draws on 2,000 fixed points: the mean Mahalanobis^2
    per dimension of the refined points about the truth, with the linear loss and the true sigma."""
    uvs, ext, intr, truth = scene(2000, sigma=0.0, p_missing=0.0, seed=80)
    E, Ks, D = rr.rig(ext, intr)
    rng = np.random.default_rng(9)
    sigma = 0.5
    m2 = []
    worst = 0.0
    for draw in range(64):
        noisy = uvs + rng.normal(0, sigma, uvs.shape)
        res = mcc.refine_points(noisy, ext, intr, sigma=sigma)
        assert (res.status > 0).all()
        if draw < 2:
            for loss in ("linear", "arctan"):
                r = res if loss == "linear" else mcc.refine_points(noisy, ext, intr, loss=loss, sigma=sigma)
                seen = np.ones(noisy.shape[:2], bool)
                cov = rr.covariance(r.points, noisy, seen, E, Ks, D, loss, 1.0, sigma=sigma)
                worst = max(worst, float((np.abs(r.covariance - cov).max((1, 2)) / np.abs(cov).max((1, 2))).max()))
        e = res.points - truth
        m2.append(np.einsum("pi,pij,pj->p", e, np.linalg.inv(res.covariance), e))
    per_dim = np.mean(m2) / 3
    print(f"covariance: largest element-wise difference {worst:.2g} relative; mean Mahalanobis^2 per "
          f"dimension over 64 x 2000 refined points {per_dim:.4f}")
    assert worst <= 1e-10
    assert 0.95 <= per_dim <= 1.05
