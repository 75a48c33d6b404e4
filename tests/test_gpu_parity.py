"""GPU parity tests: every call goes through the C ABI (libmcba.so) and is
checked against the numpy oracle and the committed fixtures generated from the
unmodified reference.  Tolerances are the ones BASELINE.json's north_star states:
residuals 1e-10 relative, Jacobians 1e-5 relative to the reference's finite
differences (norm-wise per column block), converged RMS within 1e-6 px and
camera parameters within 1e-6 relative (gauge-normalised, SURVEY.md H1)."""
import numpy as np
import pytest
from scipy.sparse import csr_matrix

from conftest import load_golden, split_cams
from oracle import np_oracle as orc
import multicam_calibration_b200 as mcc
from multicam_calibration_b200.synthetic import make_scene, make_keypoints

pytestmark = pytest.mark.gpu


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300)


# ------------------------------------------------------------------ geometry / config 5
def test_project_points_matches_reference():
    g = load_golden("geometry")
    uv = mcc.project_points(g["pts"], g["ext"], g["K"], g["dist"])
    assert uv.shape == g["uv_dist"].shape
    np.testing.assert_allclose(uv, g["uv_dist"], rtol=1e-12)
    np.testing.assert_allclose(mcc.project_points(g["pts"], g["ext"], g["K"], None), g["uv_nodist"], rtol=1e-12)


def test_undistort_points_matches_reference_cv2():
    g = load_golden("geometry")
    out = mcc.undistort_points(g["uv_in"], g["K"], g["dist"])
    assert np.array_equal(np.isnan(out), np.isnan(g["uv_undist"]))
    np.testing.assert_allclose(out, g["uv_undist"], rtol=0, atol=1e-9)


def test_triangulate_matches_reference():
    g = load_golden("triangulate")
    intr = list(zip(g["Ks"], g["dists"]))
    out = mcc.triangulate(list(g["all_uvs"]), list(g["extrinsics"]), intr)
    assert np.array_equal(np.isnan(out), np.isnan(g["points"]))
    np.testing.assert_allclose(out, g["points"], rtol=1e-8, atol=1e-8)


def test_triangulate_large_against_oracle_and_truth():
    all_uvs, ext, intr, pts = make_keypoints(20000, 6, sigma=0.0, p_missing=0.2, seed=2)
    out = mcc.triangulate(all_uvs, list(ext), intr)
    ref = orc.triangulate(all_uvs, list(ext), intr)
    assert np.array_equal(np.isnan(out), np.isnan(ref))
    ok = ~np.isnan(ref).any(1)
    np.testing.assert_allclose(out[ok], ref[ok], rtol=1e-8, atol=1e-8)
    # noise-free projections of (k1,k2)-distorted cameras: the 5-step undistortion is accurate to ~1e-6 px
    assert np.abs(out[ok] - pts[ok]).max() < 1e-2
    # round trip: project the triangulated points back
    uv = mcc.project_points(out[ok], ext[0], *intr[0])
    seen = ~np.isnan(all_uvs[0][ok]).any(1)
    assert np.abs(uv[seen] - all_uvs[0][ok][seen]).max() < 1e-2


# ------------------------------------------------------------------ per-call operators
def test_residuals_match_reference_fixture():
    g = load_golden("ba_small")
    r = mcc.residuals(g["x0"], g["uvs"], g["objpoints"])
    assert r.shape == g["residuals"].shape
    assert rel(r, g["residuals"]) < 1e-10
    assert np.abs(r - g["residuals"]).max() < 1e-10 * np.abs(g["residuals"]).max()


def test_predict_and_embed_match_reference_fixture():
    g = load_golden("ba_small")
    ext, intr, poses = mcc.deserialize_params(g["x0"], g["uvs"].shape[0])
    np.testing.assert_allclose(mcc.embed_calib_objpoints(g["objpoints"], poses), g["world"], rtol=1e-12, atol=1e-11)
    np.testing.assert_allclose(mcc.predict_calib_uvs(ext, intr, g["objpoints"], poses), g["predicted"], rtol=1e-11)
    prob = mcc.BAProblem(g["uvs"], g["objpoints"])
    np.testing.assert_allclose(prob.predict(g["x0"]), g["predicted"], rtol=1e-11)
    assert prob.n_residuals == g["residuals"].size


@pytest.mark.parametrize("shape", [(1, 1, 1), (2, 33, 4), (3, 64, 35), (9, 70, 6), (16, 40, 35)])
def test_residuals_ragged_shapes_against_oracle(shape):
    C, F, N = shape
    sc = make_scene(C, F, board=(1, N) if N != 35 else (5, 7), sigma=0.5, p_missing_view=0.3,
                    p_missing_corner=0.15, seed=C * 100 + F)
    uvs = sc.uvs.copy()
    if uvs.size > 8:
        uvs[0, 0, 0, 1] = np.nan
    x = sc.x0()
    ref = orc.residuals(x, uvs, sc.objpoints)
    out = mcc.residuals(x, uvs, sc.objpoints)
    assert out.shape == ref.shape
    if ref.size:
        assert np.abs(out - ref).max() <= 1e-10 * max(np.abs(ref).max(), 1.0)


def test_residuals_all_missing_is_empty():
    sc = make_scene(2, 5, sigma=0.1, seed=1)
    uvs = np.full_like(sc.uvs, np.nan)
    assert mcc.residuals(sc.x0(), uvs, sc.objpoints).shape == (0,)


def test_jacobian_blocks_match_oracle_and_reference_fd():
    g = load_golden("ba_small")
    uvs, obj, x0 = g["uvs"], g["objpoints"], g["x0"]
    C, F, N, _ = uvs.shape
    prob = mcc.BAProblem(uvs, obj)
    Jc, Jp = prob.jacobian_blocks(x0)
    Jc_o, Jp_o, _ = orc.jacobian_blocks(x0, C, obj)
    assert rel(Jc, -Jc_o) < 1e-11 and rel(Jp, -Jp_o) < 1e-11
    # assemble in the reference row order and compare with ITS finite differences
    ci, fi, ni, ui = np.nonzero(~np.isnan(uvs))
    J = np.zeros((ci.size, 12 * C + 6 * F))
    rows = np.arange(ci.size)
    for s in range(12):
        J[rows, ci * 12 + s] = Jc[ci, fi, ni, ui, s]
    for s in range(6):
        J[rows, 12 * C + fi * 6 + s] = Jp[ci, fi, ni, ui, s]
    J2 = csr_matrix((g["J2_data"], g["J2_indices"], g["J2_indptr"]), shape=J.shape).toarray()
    J3 = csr_matrix((g["J3_data"], g["J3_indices"], g["J3_indptr"]), shape=J.shape).toarray()
    assert rel(J, J3) < 1e-8
    for s in range(12):
        cols = np.arange(C) * 12 + s
        assert rel(J[:, cols], J2[:, cols]) < 1e-5
    for s in range(6):
        cols = 12 * C + np.arange(F) * 6 + s
        assert rel(J[:, cols], J2[:, cols]) < 1e-5


@pytest.mark.parametrize("loss", ["soft_l1", "linear", "soft_l1_irls"])
@pytest.mark.parametrize("lam", [0.0, 1e-2])
def test_reduced_camera_system_matches_oracle(loss, lam):
    g = load_golden("ba_small")
    uvs, obj, x0 = g["uvs"], g["objpoints"], g["x0"]
    C = uvs.shape[0]
    prob = mcc.BAProblem(uvs, obj)
    S, b, gcam, cost = prob.build_reduced(x0, lam=lam, loss=loss)
    hessian = "irls" if loss.endswith("irls") else "triggs"
    loss = loss.replace("_irls", "")
    H, grad, cost_o = orc.normal_equations(x0, uvs, obj, loss=loss, hessian=hessian)
    D2 = np.diag(H).copy()
    D2[:12 * C] = 0.0                    # camera damping is added by the solve, not by K2
    S_o, b_o = orc.reduced_camera_system(H, grad, C, lam, D2)
    assert cost == pytest.approx(cost_o, rel=1e-12)
    assert rel(gcam, grad[:12 * C]) < 1e-10
    assert np.abs(S - S_o).max() < 1e-9 * np.abs(S_o).max()
    assert np.abs(b - b_o).max() < 1e-9 * np.abs(b_o).max()
    assert np.abs(S - S.T).max() == 0.0
    assert rel(prob.gradient(), grad) < 1e-10
    c2, sumsq, cnt = prob.cost(x0, loss=loss)
    assert c2 == pytest.approx(cost_o, rel=1e-12) and cnt == g["residuals"].size
    assert sumsq == pytest.approx(float((g["residuals"] ** 2).sum()), rel=1e-11)


def test_damped_step_matches_oracle():
    g = load_golden("ba_small")
    uvs, obj, x0 = g["uvs"], g["objpoints"], g["x0"]
    C = uvs.shape[0]
    lam = 1e-3
    prob = mcc.BAProblem(uvs, obj)
    prob.build_reduced(x0, lam=lam)
    x1 = prob.solve_step(lam)
    H, grad, _ = orc.normal_equations(x0, uvs, obj)
    step = orc.lm_step(H, grad, C, lam, np.diag(H).copy())
    assert np.abs((x1 - x0) - step).max() < 1e-7 * np.abs(step).max()


def test_many_cameras_reduced_system_matches_oracle():
    # 9 and 16 cameras exercise the camera-group path (more cameras than warps per CTA)
    for C, F in ((9, 37), (16, 33)):
        sc = make_scene(C, F, sigma=0.4, p_missing_view=0.3, seed=C)
        x0 = sc.x0()
        prob = mcc.BAProblem(sc.uvs, sc.objpoints)
        lam = 1e-3
        S, b, gcam, cost = prob.build_reduced(x0, lam=lam)
        H, grad, cost_o = orc.normal_equations(x0, sc.uvs, sc.objpoints)
        D2 = np.diag(H).copy()
        D2[:12 * C] = 0.0
        S_o, b_o = orc.reduced_camera_system(H, grad, C, lam, D2)
        assert cost == pytest.approx(cost_o, rel=1e-12)
        assert np.abs(S - S_o).max() < 1e-9 * np.abs(S_o).max()
        assert np.abs(b - b_o).max() < 1e-9 * np.abs(b_o).max()
        x1 = prob.solve_step(lam)
        step = orc.lm_step(H, grad, C, lam, np.diag(H).copy())
        assert np.abs((x1 - x0) - step).max() < 1e-6 * np.abs(step).max()


@pytest.mark.parametrize("C,F", [(1, 40), (2, 31), (3, 65), (5, 33), (7, 96), (12, 40)])
def test_camera_count_sweep_step_and_solve(C, F):
    """Every camera count takes its own variants of K2c (ring 2-6 cameras / streamed), of the SYRK tile
    lists, of the finalize grid and of the solve kernel (12 C not a multiple of 8: partial last panel;
    3 / 8 register tiles per warp, 19 in shared memory): reduced system and damped step against the dense oracle, then
    the LM loop down to the oracle's own minimum."""
    sc = make_scene(C, F, sigma=0.3, p_missing_view=0.25 if C > 2 else 0.0, p_missing_corner=0.05, seed=40 + C)
    x0 = sc.x0()
    prob = mcc.BAProblem(sc.uvs, sc.objpoints)
    lam = 1e-3
    S, b, gcam, cost = prob.build_reduced(x0, lam=lam)
    H, grad, cost_o = orc.normal_equations(x0, sc.uvs, sc.objpoints)
    D2 = np.diag(H).copy()
    D2[:12 * C] = 0.0
    S_o, b_o = orc.reduced_camera_system(H, grad, C, lam, D2)
    assert cost == pytest.approx(cost_o, rel=1e-12)
    assert np.abs(S - S_o).max() < 1e-9 * np.abs(S_o).max()
    assert np.abs(b - b_o).max() < 1e-9 * np.abs(b_o).max()
    assert np.array_equal(S, S.T)
    x1 = prob.solve_step(lam)
    step = orc.lm_step(H, grad, C, lam, np.diag(H).copy())
    assert np.abs((x1 - x0) - step).max() < 1e-6 * np.abs(step).max()
    x, res = prob.solve(x0, ftol=1e-12, xtol=1e-12, verbose=0)
    assert res.success
    assert res.cost == pytest.approx(orc.robust_cost(x, sc.uvs, sc.objpoints), rel=1e-11)
    assert res.cost < cost and res.rms < 0.4


# ------------------------------------------------------------------ convergence
@pytest.mark.parametrize("hessian", ["auto", "triggs", "irls"])
def test_lm_loop_follows_the_dense_mirror(hessian):
    """The device LM loop and its dense numpy restatement (oracle.lm_solve) take the same
    path: same number of accepted steps / evaluations and the same final cost."""
    sc = make_scene(4, 24, sigma=0.4, p_missing_view=0.2, seed=21)
    x0 = sc.x0()
    x, res = mcc.BAProblem(sc.uvs, sc.objpoints).solve(x0, ftol=1e-9, xtol=1e-9, hessian=hessian, verbose=0)
    xo, info = orc.lm_solve(x0, sc.uvs, sc.objpoints, ftol=1e-9, xtol=1e-9, hessian=hessian)
    assert res.status == info["status"]
    assert abs(res.iterations - info["iterations"]) <= 1 and abs(res.nfev - info["nfev"]) <= 1
    assert res.cost == pytest.approx(info["cost"], rel=1e-9)
    assert orc.reprojection_rms(x, sc.uvs, sc.objpoints) == pytest.approx(
        orc.reprojection_rms(xo, sc.uvs, sc.objpoints), abs=1e-7)


def gauge_free(x, C):
    cams = x[:12 * C].reshape(C, 12)
    return cams[:, :6].copy(), orc.relative_camera_transforms(cams[:, 6:])


def assert_cameras_match(x, x_ref, C, rtol=1e-6):
    """north_star: camera parameters within 1e-6 relative -- all six intrinsics (k1, k2 included),
    element-wise, and the gauge-normalised camera transforms T_c T_0^-1 (SURVEY.md H1)."""
    intr_a, T_a = gauge_free(x, C)
    intr_b, T_b = gauge_free(x_ref, C)
    np.testing.assert_allclose(intr_a, intr_b, rtol=rtol, atol=0)
    assert np.abs(T_a - T_b).max() < rtol * np.abs(T_b).max()


def test_converges_to_the_reference_minimum():
    """6 x 40 frames: the fixture's x_tight is scipy least_squares on the UNMODIFIED reference residual
    function (trf, exact solve, tolerances 1e-15), polished to |g| ~ 5e-8; nothing in it comes from the engine."""
    g = load_golden("convergence")
    use = g["use_frames"]
    uv, obj = g["uvs"][:, use], g["objpoints"]
    C = uv.shape[0]
    x0 = np.concatenate([g["init_cams"].ravel(), g["init_poses"][use].ravel()])
    prob = mcc.BAProblem(uv, obj)
    x, res = prob.solve(x0, ftol=1e-15, xtol=1e-15, gtol=1e-9, max_nfev=300, verbose=0)
    rms = orc.reprojection_rms(x, uv, obj)
    assert res.cost <= float(g["cost_tight"]) * (1 + 1e-10)
    assert abs(rms - float(g["rms_tight"])) < 1e-6          # north_star: RMS within 1e-6 px of scipy
    assert abs(res.rms - rms) < 1e-9
    assert res.optimality < 1e-6
    assert_cameras_match(x, g["x_tight"], C)                 # polished scipy solution
    assert_cameras_match(x, g["x_scipy_tight"], C)           # scipy's own stopping point (optimality 8e-4)


def test_cfg1_converges_to_the_reference_minimum():
    """BASELINE configs[0] (6 cameras x 500 frames x 35 corners, sigma = 0.3 px): same inputs and
    initialisation as the reference run recorded in tests/golden/ba_cfg1.npz."""
    g = load_golden("ba_cfg1")
    use = g["use_frames"]
    uv, obj = g["uvs"][:, use], g["objpoints"]
    C = uv.shape[0]
    prob = mcc.BAProblem(uv, obj)
    # (1) tight tolerances: the minimum of the reference's objective
    x, res = prob.solve(g["x0"], ftol=1e-15, xtol=1e-15, gtol=1e-9, max_nfev=300, verbose=0)
    rms = orc.reprojection_rms(x, uv, obj)
    assert res.cost <= float(g["cost_tight"]) * (1 + 1e-11)
    assert abs(rms - float(g["rms_tight"])) < 1e-6
    assert res.optimality < 1e-5
    assert_cameras_match(x, g["x_tight"], C)
    # (2) reference defaults (ftol = 1e-4): at least as low as where scipy stopped, in far fewer evaluations
    xd, rd = prob.solve(g["x0"], verbose=0)
    assert rd.success and rd.cost <= float(g["cost_default"]) * (1 + 1e-9)
    assert rd.nfev <= int(g["nfev_default"])
    assert abs(orc.reprojection_rms(xd, uv, obj) - float(g["rms_tight"])) < 1e-5
    # (3) the public call: same frames, same message, and the same minimum under tight tolerances
    ext, intr = split_cams(g["init_cams"])
    np.random.seed(0)
    e, i, p, use_b, rb = mcc.bundle_adjust(g["uvs"], ext, intr, obj, g["init_poses"], n_frames=None,
                                           ftol=1e-15, xtol=1e-15, gtol=1e-9, max_nfev=300, verbose=0)
    assert np.array_equal(use_b, use)
    assert_cameras_match(rb.x, g["x_tight"], C)
    np.testing.assert_allclose(np.stack([k[[0, 1, 0, 1], [0, 1, 2, 2]] for k, _ in i]), rb.x[:72].reshape(6, 12)[:, :4])
    assert rb.fun.shape == (uv.size,) and abs(np.sqrt(np.mean(rb.fun ** 2)) - float(g["rms_tight"])) < 1e-6


def test_default_tolerances_reach_at_least_the_reference_cost():
    g = load_golden("convergence")
    use = g["use_frames"]
    uv, obj = g["uvs"][:, use], g["objpoints"]
    x0 = np.concatenate([g["init_cams"].ravel(), g["init_poses"][use].ravel()])
    x, res = mcc.BAProblem(uv, obj).solve(x0, verbose=0)
    assert res.status in (1, 2, 3, 4) and res.success
    assert res.cost <= float(g["cost_default"]) * (1 + 1e-6)
    assert res.fun.shape == ((~np.isnan(uv)).sum(),)
    assert res.cost == pytest.approx(orc.robust_cost(x, uv, obj), rel=1e-10)
    np.testing.assert_allclose(res.grad, orc.normal_equations(x, uv, obj)[1], atol=1e-7 * np.abs(res.grad).max() + 1e-9)


def test_bundle_adjust_api_matches_reference_front_end(capsys):
    g = load_golden("frontend")
    ext, intr = split_cams(g["init_cams"])
    for tag, nf in (("all", None), ("sub", 20)):
        np.random.seed(0)
        e, i, p, use, result = mcc.bundle_adjust(g["uvs"], ext, intr, g["objpoints"], g["init_poses"],
                                                 n_frames=nf, verbose=0)
        out = capsys.readouterr().out
        assert np.array_equal(use, g[f"use_{tag}"])
        # same sentence and counts as the reference; the threshold (5 * nanmedian of the device-computed
        # errors) may differ from numpy's in the last bits
        got, ref = out.strip().splitlines()[0].split(), str(g[f"msg_{tag}"]).strip().split()
        assert got[:-1] == ref[:-1] and float(got[-1]) == pytest.approx(float(ref[-1]), rel=1e-12)
        assert e.shape == (5, 6) and p.shape == (len(use), 6) and len(i) == 5
        assert i[0][0].shape == (3, 3) and i[0][1].shape == (5,)
        assert result.x.shape == (60 + 6 * len(use),) and result.success


def test_bundle_adjust_verbose_table_and_nonfinite_x0(capsys):
    sc = make_scene(3, 12, sigma=0.2, seed=4)
    args = sc.init_args()
    mcc.bundle_adjust(*args, n_frames=None, max_nfev=5)
    out = capsys.readouterr().out
    assert "Iteration" in out and "Total nfev" in out and "Optimality" in out
    bad = args[4].copy()
    bad[3, 0] = np.nan
    with pytest.raises(ValueError, match="not finite"):
        mcc.BAProblem(sc.uvs, sc.objpoints).solve(np.concatenate([sc.init_cams.ravel(), bad.ravel()]), verbose=0)


# ------------------------------------------------------------------ full-size properties
def test_full_size_properties_cfg2():
    """6 cams x 5000 frames: size-independent checks (no oracle at this size)."""
    sc = make_scene(6, 5000, sigma=0.3, p_missing_view=0.2, seed=0)
    prob = mcc.BAProblem(sc.uvs, sc.objpoints)
    x0 = sc.x0()
    # (1) cost from K2, from the cost kernel and from the materialised residual vector agree
    r = prob.residuals(x0)
    cost_r = float((2 * (np.sqrt(1 + r * r) - 1)).sum() * 0.5)
    S, b, gcam, cost = prob.build_reduced(x0, lam=1e-3)
    assert cost == pytest.approx(cost_r, rel=1e-11)
    assert prob.cost(x0)[0] == pytest.approx(cost_r, rel=1e-11)
    assert r.size == (~np.isnan(sc.uvs)).sum()
    # (2) sharding additivity: S, b of two halves (same camera block) sum to the whole
    halves = []
    for a, bnd in ((0, 2500), (2500, 5000)):
        p2 = mcc.BAProblem(sc.uvs[:, a:bnd], sc.objpoints)
        xl = np.concatenate([x0[:72], x0[72 + 6 * a:72 + 6 * bnd]])
        halves.append(p2.build_reduced(xl, lam=1e-3))
    S2 = halves[0][0] + halves[1][0]
    b2 = halves[0][1] + halves[1][1]
    assert np.abs(S2 - S).max() < 1e-11 * np.abs(S).max()
    assert np.abs(b2 - b).max() < 1e-10 * np.abs(b).max()
    # (3) the solve reduces the cost monotonically to the noise floor and is a stationary point
    x, res = prob.solve(x0, ftol=1e-10, verbose=0)
    assert res.cost < cost and res.success
    assert 0.28 < res.rms < 0.32          # sigma = 0.3 px
    assert res.optimality < 1e-2 * np.abs(gcam).max()


def test_full_size_properties_cfg3():
    """BASELINE configs[2] at full size (6 cams x 50,000 frames, 20 % missing views, 0.5 px noise):
    size-independent properties, no oracle at this size."""
    C, F = 6, 50000
    sc = make_scene(C, F, sigma=0.5, p_missing_view=0.2, seed=0)
    prob = mcc.BAProblem(sc.uvs, sc.objpoints)
    x0 = sc.x0()
    nc = 12 * C
    # (1) checksum of checksums: the cost accumulated inside K2p, the cost kernel and the robust
    #     cost of the materialised residual vector agree; the vector has one entry per finite scalar
    r = prob.residuals(x0)
    assert r.size == (~np.isnan(sc.uvs)).sum() == prob.n_residuals
    cost_r = float((2 * (np.sqrt(1 + r * r) - 1)).sum() * 0.5)
    S, b, gcam, cost = prob.build_reduced(x0, lam=1e-3)
    assert cost == pytest.approx(cost_r, rel=1e-11)
    assert prob.cost(x0)[0] == pytest.approx(cost_r, rel=1e-11)
    assert np.abs(S - S.T).max() <= 1e-12 * np.abs(S).max()
    # (2) residuals = observed - predicted on the finite entries, in the reference's order
    pred = prob.predict(x0)
    assert pred.shape == sc.uvs.shape and not np.isnan(pred).any()
    ok = ~np.isnan(sc.uvs)
    assert np.abs((sc.uvs - pred)[ok] - r).max() <= 1e-10 * np.abs(r).max()
    # (3) frame order does not matter: a random permutation of the frames (observations and
    #     poses together) gives the same reduced camera system up to summation order
    perm = np.random.default_rng(5).permutation(F)
    xp = np.concatenate([x0[:nc], x0[nc:].reshape(F, 6)[perm].ravel()])
    Sp, bp, gp_, costp = mcc.BAProblem(np.ascontiguousarray(sc.uvs[:, perm]), sc.objpoints).build_reduced(xp, lam=1e-3)
    assert costp == pytest.approx(cost, rel=1e-12)
    assert np.abs(Sp - S).max() <= 1e-10 * np.abs(S).max()
    assert np.abs(bp - b).max() <= 1e-9 * np.abs(b).max()
    # (4) additivity over frame shards (what the multi-GPU path relies on): four uneven shards
    bounds = [0, 7, 12501, 31000, F]
    Ssum, bsum, csum = 0.0, 0.0, 0.0
    for a, e in zip(bounds[:-1], bounds[1:]):
        xl = np.concatenate([x0[:nc], x0[nc + 6 * a:nc + 6 * e]])
        Sl, bl, _, cl = mcc.BAProblem(sc.uvs[:, a:e], sc.objpoints).build_reduced(xl, lam=1e-3)
        Ssum, bsum, csum = Ssum + Sl, bsum + bl, csum + cl
    assert csum == pytest.approx(cost, rel=1e-12)
    assert np.abs(Ssum - S).max() <= 1e-10 * np.abs(S).max()
    assert np.abs(bsum - b).max() <= 1e-9 * np.abs(b).max()
    # (5) the solve ends at a stationary point at the noise floor, and solving again from there is idempotent
    x, res = prob.solve(x0, ftol=1e-10, xtol=1e-10, verbose=0)
    assert res.success and res.cost < cost
    assert 0.48 < res.rms < 0.52          # sigma = 0.5 px
    assert res.optimality < 1e-6 * np.abs(gcam).max()
    x2, res2 = prob.solve(x, ftol=1e-10, xtol=1e-10, verbose=0)
    assert res2.iterations <= 2 and abs(res2.cost - res.cost) <= 1e-9 * res.cost
    assert np.abs(x2 - x).max() <= 1e-4   # the 6-D rigid gauge is free (as in the reference): a restart may drift along it


# ------------------------------------------------------------------ device front end (SURVEY 8(f) N1)
@pytest.mark.parametrize("threshold", [None, 2.5])
def test_select_frames_device_matches_oracle(threshold, capsys):
    """mcba_select_frames (eligibility, per-frame worst mean error, exact nanmedian threshold,
    exclusion) against the numpy restatement of bundle_adjustment.py:265-296, on a scene with
    missing views, per-corner dropouts, gross outlier frames, a NaN pose in an ineligible frame
    and one in an eligible frame."""
    sc = make_scene(5, 211, sigma=0.4, p_missing_view=0.35, p_missing_corner=0.03, seed=17)
    uvs = sc.uvs.copy()
    rng = np.random.default_rng(3)
    bad = rng.choice(211, 12, replace=False)
    uvs[:, bad] += rng.normal(0, 40.0, uvs[:, bad].shape)          # gross outliers
    ext, intr, _, obj, poses = sc.init_args()[1], sc.init_args()[2], None, sc.objpoints, sc.init_args()[4].copy()
    complete = (~np.isnan(uvs).any((-1, -2))).sum(0)
    poses[np.nonzero(complete <= 1)[0][0]] = np.nan                 # never looked at
    poses[np.nonzero(complete > 1)[0][5], 0] = np.nan               # eligible: all its errors are NaN
    for nf in (None, 40):
        np.random.seed(1)
        use = mcc.select_frames(uvs, ext, intr, obj, poses, n_frames=nf, outlier_threshold=threshold)
        msg = capsys.readouterr().out.strip().splitlines()[0].split()
        np.random.seed(1)
        use_o, thr_o = orc.select_frames(uvs, ext, intr, obj, poses, n_frames=nf, outlier_threshold=threshold,
                                         verbose=False)
        assert np.array_equal(use, use_o)
        assert float(msg[-1]) == pytest.approx(float(thr_o), rel=1e-12)


def test_sharded_front_end_equals_the_single_device_front_end(capsys):
    """The staged front end of frame-sharded runs (mcba_frame_errors + radix-selection median through
    mcba_key_histogram + mcba_apply_threshold; one rank here) keeps exactly the frames, prints exactly
    the threshold and consumes the RNG exactly like the single-device front end and the oracle."""
    import torch
    from multicam_calibration_b200 import bundle_adjustment as ba
    sc = make_scene(5, 211, sigma=0.4, p_missing_view=0.35, p_missing_corner=0.03, seed=17)
    uvs = sc.uvs.copy()
    rng = np.random.default_rng(3)
    bad = rng.choice(211, 12, replace=False)
    uvs[:, bad] += rng.normal(0, 40.0, uvs[:, bad].shape)
    _, ext, intr, obj, poses = sc.init_args()
    for nf, thr in ((None, None), (40, None), (None, 2.5)):
        np.random.seed(1)
        use_a = mcc.select_frames(uvs, ext, intr, obj, poses, n_frames=nf, outlier_threshold=thr)
        msg_a = capsys.readouterr().out.strip().splitlines()[0]
        np.random.seed(1)
        use_b, d_local, counts = ba._select_frames_sharded(uvs, ext, intr, obj, poses, nf, thr)
        assert counts.tolist() == [len(use_b)]
        msg_b = capsys.readouterr().out.strip().splitlines()[0]
        assert np.array_equal(use_a, use_b) and msg_a == msg_b
        assert np.array_equal(d_local.cpu().numpy(), uvs[:, use_b], equal_nan=True)
    # the histogram kernel against numpy on the raw bit patterns
    import ctypes
    from multicam_calibration_b200 import _native
    vals = np.abs(rng.normal(0, 3, 100003))
    vals[::5] = np.nan
    vals[7] = 0.0
    d_vals = _native.to_device(vals)
    d_hist = torch.empty(256, dtype=torch.int64, device="cuda")
    keys = vals[~np.isnan(vals)].view(np.uint64)
    top = int(np.bincount((keys >> np.uint64(56)).astype(np.int64)).argmax())
    for prefix, bits in ((0, 0), (top, 8)):
        _native.check(_native.load().mcba_key_histogram(torch.cuda.current_device(), ctypes.c_void_p(
            torch.cuda.current_stream().cuda_stream), ctypes.c_void_p(d_vals.data_ptr()), vals.size,
            ctypes.c_uint64(prefix), bits, ctypes.c_void_p(d_hist.data_ptr())))
        k = keys if bits == 0 else keys[(keys >> np.uint64(64 - bits)) == np.uint64(prefix)]
        ref = np.bincount(((k >> np.uint64(64 - bits - 8)) & np.uint64(0xff)).astype(np.int64), minlength=256)
        assert np.array_equal(d_hist.cpu().numpy(), ref)


def test_repeated_bundle_adjust_on_the_cached_problem_orders_gather_before_solve():
    """Two calls of the same shape at a size where the device gather of the kept frames outlasts the
    host: the second call reuses the cached problem (no allocation in between), so the solve must be
    ordered after the gather kernel on the caller's stream (the problem runs on its own stream)."""
    sc = make_scene(6, 20000, sigma=0.5, p_missing_view=0.2, seed=3)
    args = sc.init_args()
    outs = []
    for _ in range(2):
        np.random.seed(0)
        e, i, p, use, res = mcc.bundle_adjust(*args, n_frames=None, verbose=0)
        outs.append((use, res.x, res.cost, res.nfev))
    x0 = mcc.serialize_params(args[1], args[2], args[4][outs[0][0]])
    x, r = mcc.BAProblem(args[0][:, outs[0][0]], sc.objpoints).solve(x0, verbose=0)      # host-array path
    for use, xs, cost, nfev in outs:
        assert np.array_equal(use, outs[0][0]) and nfev == r.nfev
        assert cost == pytest.approx(r.cost, rel=1e-12) and np.allclose(xs, x, rtol=0, atol=1e-9)
    mcc.release_device_memory()


def test_handwritten_reduced_solve_matches_the_library_path():
    """The one-CTA shared-memory Cholesky (k3_solve.cu) against cuSOLVER potrf/potrs on the same
    damped systems (MCBA_CUSOLVER=1 in a child process), 6 / 9 / 16 cameras; and a non-positive
    pivot is reported, not propagated silently."""
    import subprocess
    import sys
    import json
    from conftest import ROOT
    code = (
        "import sys, json, numpy as np\n"
        "sys.path.insert(0, %r)\n"
        "import multicam_calibration_b200 as mcc\n"
        "from multicam_calibration_b200.synthetic import make_scene\n"
        "out = {}\n"
        "for C, F in ((6, 64), (9, 37), (16, 33)):\n"
        "    sc = make_scene(C, F, sigma=0.4, p_missing_view=0.3, seed=C)\n"
        "    prob = mcc.BAProblem(sc.uvs, sc.objpoints)\n"
        "    prob.build_reduced(sc.x0(), lam=1e-3)\n"
        "    out[str(C)] = prob.solve_step(1e-3).tolist()\n"
        "print(json.dumps(out))\n" % ROOT)
    import os
    steps = {}
    for tag, env in (("own", {}), ("lib", {"MCBA_CUSOLVER": "1"})):
        e = dict(os.environ)
        e.update(env)
        run = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=e)
        assert run.returncode == 0, run.stderr[-2000:]
        steps[tag] = json.loads(run.stdout.strip().splitlines()[-1])
    for C in ("6", "9", "16"):
        a, b = np.array(steps["own"][C]), np.array(steps["lib"][C])
        assert np.abs(a - b).max() <= 1e-9 * np.abs(b).max(), C
    # lambda = 0: the undamped reduced system is singular along the rigid gauge -> rejected loudly
    sc = make_scene(3, 12, sigma=0.2, seed=4)
    prob = mcc.BAProblem(sc.uvs, sc.objpoints)
    prob.build_reduced(sc.x0(), lam=0.0)
    try:
        x1 = prob.solve_step(0.0)
        assert np.isfinite(x1).all()          # rounding can leave the tiny pivots positive
    except Exception as err:
        assert "not positive definite" in str(err)


def test_bundle_adjust_device_gather_equals_host_slicing():
    """bundle_adjust (device front end + device gather of the kept frames) ends where a BAProblem
    built from the host-sliced observations ends."""
    sc = make_scene(4, 150, sigma=0.3, p_missing_view=0.25, seed=8)
    args = sc.init_args()
    np.random.seed(2)
    e, i, p, use, res = mcc.bundle_adjust(*args, n_frames=60, ftol=1e-10, xtol=1e-10, verbose=0)
    x0 = mcc.serialize_params(args[1], args[2], args[4][use])
    x, r = mcc.BAProblem(args[0][:, use], sc.objpoints).solve(x0, ftol=1e-10, xtol=1e-10, verbose=0)
    assert res.cost == pytest.approx(r.cost, rel=1e-12) and res.nfev == r.nfev
    assert np.allclose(res.x, x, rtol=0, atol=1e-9)


# ------------------------------------------------------------------ host <-> device staging, lazy result fields
@pytest.mark.parametrize("n", [0, 1, 1000, (8 << 20) // 8 - 3, 5 * (4 << 20) // 8 + 7, 29 * (4 << 20) // 8 + 12345])
def test_staged_upload_download_round_trip(n):
    """mcba_upload / mcba_download move pageable numpy buffers bit-exactly (sizes below the staging
    threshold, an exact multiple of the chunk, ragged tails, more chunks than worker threads)."""
    import torch
    from multicam_calibration_b200 import _native
    rng = np.random.default_rng(n)
    a = rng.standard_normal(n)
    d = _native.to_device(a)
    assert d.shape == (n,) and d.dtype == torch.float64
    assert np.array_equal(d.cpu().numpy(), a)
    d2 = d * 2.0 + 1.0                       # produced on the stream the download is ordered after
    assert np.array_equal(_native.to_host(d2), a * 2.0 + 1.0)
    pinned = torch.from_numpy(a.copy()).pin_memory()
    assert np.array_equal(_native.to_device(pinned.numpy()).cpu().numpy(), a)


def test_result_fun_is_lazy_and_matches_residuals():
    g = load_golden("frontend")
    ext, intr = split_cams(g["init_cams"])
    np.random.seed(0)
    e, i, p, use, result = mcc.bundle_adjust(g["uvs"], ext, intr, g["objpoints"], g["init_poses"],
                                             n_frames=None, verbose=0)
    assert not dict.__contains__(result, "fun") and "fun" in result and "fun" in result.keys()
    r_ref = orc.residuals(result.x, g["uvs"][:, use], g["objpoints"])
    fun = result.fun
    assert dict.__contains__(result, "fun") and result["fun"] is fun
    assert fun.shape == r_ref.shape and np.abs(fun - r_ref).max() <= 1e-10 * np.abs(r_ref).max()
    # a result whose cached problem has been reused still produces fun (rebuilt from the caller's arrays)
    np.random.seed(0)
    *_, result2 = mcc.bundle_adjust(g["uvs"], ext, intr, g["objpoints"], g["init_poses"], n_frames=None, verbose=0)
    mcc.residuals(result2.x, g["uvs"][:, use] + 1.0, g["objpoints"])
    assert np.abs(result2.fun - r_ref).max() <= 1e-10 * np.abs(r_ref).max()
    with pytest.raises(AttributeError):       # like scipy's OptimizeResult
        result2.missing_field
    assert not hasattr(result2, "missing_field") and hasattr(result2, "fun")


# ------------------------------------------------------------------ initialisation algebra (SURVEY 8(f) N2)
@pytest.mark.parametrize("tag", ["a", "b"])
def test_initialisation_algebra_matches_reference_fixture(tag):
    g = load_golden("init")
    poses = g[f"{tag}_poses"]
    pair = mcc.estimate_pairwise_camera_transform(poses[0], poses[1])
    np.testing.assert_allclose(pair, g[f"{tag}_pair01"], rtol=0, atol=1e-9)
    for root, key in ((0, ""), (2, "_root2")):
        ext, tree = mcc.estimate_all_extrinsics(poses, root=root)
        assert tree == [tuple(int(v) for v in e) for e in g[f"{tag}_tree{key}"]]
        np.testing.assert_allclose(ext, g[f"{tag}_ext{key}"], rtol=0, atol=1e-9)
    cons = mcc.consensus_calib_poses(poses, g[f"{tag}_ext"])
    assert np.array_equal(np.isnan(cons), np.isnan(g[f"{tag}_consensus"]))
    np.testing.assert_allclose(cons, g[f"{tag}_consensus"], rtol=0, atol=1e-9)


def test_initialisation_algebra_large_against_oracle_and_truth():
    from multicam_calibration_b200.synthetic import make_camera_poses
    poses, ext_true, board_true = make_camera_poses(7, 20000, p_missing=0.3, seed=5)
    poses[:, 11] = np.nan
    ext, tree = mcc.estimate_all_extrinsics(poses, root=0)
    ext_o, tree_o = orc.estimate_all_extrinsics(poses, root=0)
    assert tree == [tuple(int(v) for v in e) for e in tree_o]
    np.testing.assert_allclose(ext, ext_o, rtol=0, atol=1e-9)
    cons = mcc.consensus_calib_poses(poses, ext)
    cons_o = orc.consensus_calib_poses(poses, ext)
    assert np.array_equal(np.isnan(cons), np.isnan(cons_o)) and np.isnan(cons[11]).all()
    np.testing.assert_allclose(cons, cons_o, rtol=0, atol=1e-9)
    dT = orc.transformation_matrix(ext) - orc.transformation_matrix(ext_true)
    assert np.abs(dT[:, :3, :3]).max() < 0.01 and np.abs(dT[:, :3, 3]).max() < 5.0
    # no common frame: NaN like np.median of an empty selection; wrong shapes raise
    a, b = poses[0].copy(), poses[1].copy()
    a[::2], b[1::2] = np.nan, np.nan
    assert np.isnan(mcc.estimate_pairwise_camera_transform(a, b)).all()
    with pytest.raises(ValueError):
        mcc.estimate_pairwise_camera_transform(poses[0], poses[1][:-1])
    with pytest.raises(ValueError):
        mcc.consensus_calib_poses(poses, ext[:-1])


def test_device_transformation_vectors_match_reference():
    import ctypes
    import torch
    from multicam_calibration_b200 import _native
    g = load_golden("init")
    lib = _native.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for key, dim, width in (("R", 3, 3), ("T", 4, 6)):
        d_in = _native.to_device(g[key])
        d_out = torch.empty((len(g[key]), width), dtype=torch.float64, device="cuda")
        _native.check(lib.mcba_transformation_vectors(torch.cuda.current_device(), stream, ctypes.c_void_p(d_in.data_ptr()),
                                                      len(g[key]), dim, ctypes.c_void_p(d_out.data_ptr())))
        np.testing.assert_allclose(_native.to_host(d_out), g[f"{key}_vec"], rtol=0, atol=1e-12)


def test_project_points_multi_matches_per_camera_projection():
    g = load_golden("triangulate")
    intr = list(zip(g["Ks"], g["dists"]))
    rng = np.random.default_rng(4)
    pts = rng.normal(0, 80, (3, 1001, 3))                       # leading dims, ragged against the 256-point blocks
    both = mcc.project_points_multi(pts, list(g["extrinsics"]), intr)
    assert both.shape == (len(intr), 3, 1001, 2)
    for c, (ext, (K, dist)) in enumerate(zip(g["extrinsics"], intr)):
        np.testing.assert_allclose(both[c], orc.project_points(pts, ext, K, dist), rtol=1e-12)
        np.testing.assert_allclose(both[c], mcc.project_points(pts, ext, K, dist), rtol=1e-14)
    nodist = mcc.project_points_multi(pts, list(g["extrinsics"]), [(K, None) for K, _ in intr])
    np.testing.assert_allclose(nodist[2], orc.project_points(pts, g["extrinsics"][2], intr[2][0], None), rtol=1e-12)
    with pytest.raises(ValueError):
        mcc.project_points_multi(pts, list(g["extrinsics"]), [(K, None if c else d) for c, (K, d) in enumerate(intr)])


# ------------------------------------------------------------------ N3: reprojection-error QC (viz.py:155-177)
def test_reprojection_residuals_vs_reference_and_oracle():
    """mcba_homography_transfer against the output of the UNMODIFIED viz.plot_residuals (cv2.findHomography
    per frame; tests/golden/qc.npz) and against the oracle's restatement of the same algorithm."""
    from test_io_qc_cpu import compare_transfer, qc_fixture
    d, intr = qc_fixture()
    med, rep, tr = mcc.reprojection_residuals(d["uvs"], d["ext"], intr, d["objpoints"], d["poses"])
    np.testing.assert_allclose(rep, d["reprojections"], rtol=1e-12)
    # reference: transferred corners within 1e-5 board units (mm) on >= 95 % of the frames cv2 fitted (its
    # binary-only LM ends elsewhere on the few grazing-angle frames), medians over those frames to 1e-6
    good, valid = compare_transfer(tr, med, d, frame_tol=1e-5, frac_required=0.95, median_rtol=1e-6)
    assert valid >= 100
    # oracle: the same arithmetic up to the eigen-solver and FMA contraction
    med_o, _, tr_o = orc.reprojection_transfer(d["uvs"], d["ext"], intr, d["objpoints"], d["poses"])
    assert np.array_equal(np.isnan(tr), np.isnan(tr_o))
    ok = ~np.isnan(tr_o).any((-1, -2))
    diff = np.abs(np.where(ok[..., None, None], tr - tr_o, 0.0)).max((-1, -2))
    # (whether the refinement takes one more step when its last step is within rounding of FLT_EPSILON
    # is decided differently on a few frames: those differ by the size of that last step)
    assert (diff[ok] <= 1e-6).mean() >= 0.97 and diff[ok].max() <= 1e-4, np.sort(diff[ok])[-8:]
    np.testing.assert_allclose(med, med_o, rtol=1e-3)
    # frames with a missing corner stay NaN; nothing else does
    missing = np.isnan(d["uvs"]).any((-1, -2))
    assert np.array_equal(np.isnan(tr).all((-1, -2)), missing)


def test_reprojection_residuals_exact_homography():
    """Noise-free detections of a distortion-free rig: every transferred corner lands on its board corner
    (float32 rounding of the inputs inside findHomography bounds the error) and the medians are ~0."""
    sc = make_scene(4, 64, sigma=0.0, seed=2)
    cams = sc.true_cams.copy()
    cams[:, 4:6] = 0.0
    from multicam_calibration_b200.synthetic import forward_model
    uvs = forward_model(cams, sc.true_poses, sc.objpoints)
    ext, intr = split_cams(cams)
    med, rep, tr = mcc.reprojection_residuals(uvs, ext, intr, sc.objpoints, sc.true_poses)
    np.testing.assert_allclose(rep, uvs, rtol=1e-11)
    err = np.linalg.norm(tr - sc.objpoints[:, :2], axis=-1)
    assert np.nanmax(err) < 5e-3 and np.all(med < 1e-3)


def test_host_buffer_call_pipelined_equals_plain_and_leaves_the_problem_usable(monkeypatch):
    """mcba_build_reduced_host with page-locked buffers and >= 16384 frames streams the observations in
    frame ranges that are tiled, evaluated and reduced while the next range is in flight: S, b and the
    cost must equal the plain path's (one upload, one evaluation) and the device-resident evaluation,
    and the handle must be left as after mcba_set_observations."""
    import ctypes
    import torch
    from multicam_calibration_b200 import _native
    lib = _native.load()
    sc = make_scene(6, 20011, sigma=0.5, p_missing_view=0.2, seed=5)     # not a multiple of the tile or chunk size
    x0 = sc.x0()
    prob = mcc.BAProblem(sc.uvs, sc.objpoints)
    S0, b0, g0, cost0 = prob.build_reduced(x0, lam=1e-3)
    C = 6
    keep = [torch.from_numpy(np.ascontiguousarray(sc.uvs)).pin_memory(),
            torch.from_numpy(np.ascontiguousarray(sc.objpoints, dtype=np.float64)).pin_memory(),
            torch.from_numpy(x0.copy()).pin_memory(), torch.empty(144 * C * C, dtype=torch.float64).pin_memory(),
            torch.empty(12 * C, dtype=torch.float64).pin_memory(), torch.empty(1, dtype=torch.float64).pin_memory()]
    ptrs = [ctypes.c_void_p(t.data_ptr()) for t in keep]

    def call(lam=1e-3):
        _native.check(lib.mcba_build_reduced_host(prob._h, ptrs[0], ptrs[1], ptrs[2], lam, _native.LOSSES["soft_l1"], 1.0,
                                                  ptrs[3], ptrs[4], ptrs[5]))
        return keep[3].numpy().reshape(12 * C, 12 * C).copy(), keep[4].numpy().copy(), float(keep[5][0])

    n0 = prob.kernel_launches
    Sp, bp, cp = call()                                   # pipelined
    n_pipe = prob.kernel_launches - n0
    monkeypatch.setenv("MCBA_NO_HOST_PIPELINE", "1")
    Sq, bq, cq = call()                                   # plain
    monkeypatch.delenv("MCBA_NO_HOST_PIPELINE")
    for S, b, c in ((Sp, bp, cp), (Sq, bq, cq)):
        assert np.abs(S - S0).max() < 1e-11 * np.abs(S0).max()
        assert np.abs(b - b0).max() < 1e-10 * np.abs(b0).max()
        assert c == pytest.approx(cost0, rel=1e-12)
    assert n_pipe <= 20                                   # the chunks ran on the children, not on this handle
    # twice in a row (the children's buffers are reused), then the handle itself is still a full problem
    Sp2, bp2, cp2 = call()
    assert np.array_equal(Sp2, Sp) and np.array_equal(bp2, bp) and cp2 == cp
    fresh = mcc.BAProblem(sc.uvs, sc.objpoints)
    # a third call with the same arguments replays the ranges' CUDA graphs; a different damping drops them
    Sp3, bp3, cp3 = call()
    assert np.array_equal(Sp3, Sp) and np.array_equal(bp3, bp) and cp3 == cp
    S1, b1, g1, cost1 = fresh.build_reduced(x0, lam=1e-1)
    for _ in range(3):
        Sl, bl, cl = call(1e-1)
        assert np.abs(Sl - S1).max() < 1e-11 * np.abs(S1).max() and np.abs(bl - b1).max() < 1e-10 * np.abs(b1).max()
    assert np.abs(S1 - S0).max() > 1e-6 * np.abs(S0).max()      # the damping did change the system
    Sp4, bp4, cp4 = call()
    assert np.array_equal(Sp4, Sp) and np.array_equal(bp4, bp)
    fresh.build_reduced(x0, lam=1e-3)
    assert np.allclose(prob.solve_step(1e-3), fresh.solve_step(1e-3), rtol=0, atol=1e-9)   # the damped step of the system just built
    assert np.allclose(prob.gradient(), fresh.gradient(), rtol=1e-10, atol=1e-9)
    x, res = prob.solve(x0, verbose=0)
    x_ref, res_ref = fresh.solve(x0, verbose=0)
    assert res.cost == pytest.approx(res_ref.cost, rel=1e-12) and res.nfev == res_ref.nfev
