"""CPU: the numpy oracle reproduces the outputs of the unmodified reference
(fixtures written by tests/golden/make_golden.py in the build container)."""
import numpy as np
import pytest
from scipy.sparse import csr_matrix

from conftest import load_golden, split_cams
from oracle import np_oracle as orc


def test_geometry_matches_reference():
    g = load_golden("geometry")
    assert np.array_equal(orc.rodrigues(g["r"]), g["R"])
    np.testing.assert_allclose(orc.rodrigues_inv(g["R"]), g["r_back"], rtol=0, atol=1e-14)
    assert np.array_equal(orc.transformation_matrix(g["t6"]), g["T"])
    np.testing.assert_allclose(orc.transformation_vector(g["T"]), g["t6_back"], rtol=0, atol=1e-12)
    ext, K, dist, pts = g["ext"], g["K"], g["dist"], g["pts"]
    assert np.array_equal(orc.apply_rigid_transform(ext, pts), g["pts_rigid_vec"])
    assert np.array_equal(orc.apply_rigid_transform(orc.transformation_matrix(ext), pts), g["pts_rigid_mat"])
    np.testing.assert_allclose(orc.project_points(pts, ext, K, dist), g["uv_dist"], rtol=1e-14)
    np.testing.assert_allclose(orc.project_points(pts, ext, K, None), g["uv_nodist"], rtol=1e-14)
    np.testing.assert_allclose(orc.projection_matrix(ext, (K, dist)), g["P"], rtol=1e-15)
    und = orc.undistort_points(g["uv_in"], K, dist)
    assert np.array_equal(np.isnan(und), np.isnan(g["uv_undist"]))
    np.testing.assert_allclose(und, g["uv_undist"], rtol=0, atol=1e-9)


def test_rodrigues_theta_zero_is_identity():
    assert np.array_equal(orc.rodrigues(np.zeros(3)), np.eye(3))


def test_triangulate_matches_reference():
    g = load_golden("triangulate")
    intr = list(zip(g["Ks"], g["dists"]))
    out = orc.triangulate(list(g["all_uvs"]), list(g["extrinsics"]), intr)
    assert np.array_equal(np.isnan(out), np.isnan(g["points"]))
    assert np.isnan(g["points"][:4]).all()          # < 2 views
    np.testing.assert_allclose(out, g["points"], rtol=1e-9, atol=1e-9)


def test_residuals_and_layout_match_reference():
    g = load_golden("ba_small")
    uvs, obj, x0 = g["uvs"], g["objpoints"], g["x0"]
    r = orc.residuals(x0, uvs, obj)
    assert r.shape == g["residuals"].shape == ((~np.isnan(uvs)).sum(),)
    np.testing.assert_allclose(r, g["residuals"], rtol=0, atol=1e-12)
    ext, intr, poses = orc.deserialize_params(x0, uvs.shape[0])
    np.testing.assert_allclose(orc.predict_calib_uvs(ext, intr, obj, poses), g["predicted"], rtol=1e-14)
    np.testing.assert_allclose(orc.embed_calib_objpoints(obj, poses), g["world"], rtol=1e-14, atol=1e-13)
    assert np.array_equal(orc.serialize_params(ext, intr, poses), x0)
    A = orc.sparsity_pattern(uvs)
    assert np.array_equal(A.indices, g["A_indices"]) and np.array_equal(A.indptr, g["A_indptr"])


def test_analytic_jacobian_matches_reference_finite_differences():
    g = load_golden("ba_small")
    uvs, obj, x0 = g["uvs"], g["objpoints"], g["x0"]
    J = orc.dense_residual_jacobian(x0, uvs, obj)
    shape = J.shape
    J3 = csr_matrix((g["J3_data"], g["J3_indices"], g["J3_indptr"]), shape=shape).toarray()
    J2 = csr_matrix((g["J2_data"], g["J2_indices"], g["J2_indptr"]), shape=shape).toarray()
    assert np.linalg.norm(J - J3) / np.linalg.norm(J3) < 1e-8
    C = uvs.shape[0]
    # 1e-5 relative, norm-wise per parameter column block (SURVEY.md H3)
    for s in range(12):
        cols = np.arange(C) * 12 + s
        assert np.linalg.norm(J[:, cols] - J2[:, cols]) <= 1e-5 * np.linalg.norm(J2[:, cols])
    for s in range(6):
        cols = 12 * C + np.arange((shape[1] - 12 * C) // 6) * 6 + s
        assert np.linalg.norm(J[:, cols] - J2[:, cols]) <= 1e-5 * np.linalg.norm(J2[:, cols])


def test_frame_selection_matches_reference(capsys):
    g = load_golden("frontend")
    ext, intr = split_cams(g["init_cams"])
    for tag, nf in (("all", None), ("sub", 20)):
        np.random.seed(0)
        use, _ = orc.select_frames(g["uvs"], ext, intr, g["objpoints"], g["init_poses"], n_frames=nf)
        assert np.array_equal(use, g[f"use_{tag}"])
        assert capsys.readouterr().out.strip() == str(g[f"msg_{tag}"]).strip()
    assert 17 not in g["use_all"]


def test_schur_step_equals_dense_step():
    g = load_golden("ba_small")
    uvs, obj, x0 = g["uvs"], g["objpoints"], g["x0"]
    C = uvs.shape[0]
    H, grad, cost = orc.normal_equations(x0, uvs, obj)
    D2 = np.diag(H).copy()
    lam = 1e-3
    step = orc.lm_step(H, grad, C, lam, D2)
    dense = -np.linalg.solve(H + lam * np.diag(D2), grad)
    np.testing.assert_allclose(step, dense, rtol=1e-7, atol=1e-9 * np.abs(dense).max())
    assert cost == pytest.approx(orc.robust_cost(x0, uvs, obj))


def test_convergence_fixture_is_a_stationary_point():
    g = load_golden("convergence")
    uv = g["uvs"][:, g["use_frames"]]
    H, grad, cost = orc.normal_equations(g["x_tight"], uv, g["objpoints"])
    assert cost == pytest.approx(float(g["cost_tight"]), rel=1e-12)
    assert float(g["cost_tight"]) <= float(g["cost_default"])
    assert orc.reprojection_rms(g["x_tight"], uv, g["objpoints"]) == pytest.approx(float(g["rms_tight"]), rel=1e-12)


def _sparse_gradient(x, uv, obj):
    f = orc.residuals(x, uv, obj)
    return orc.analytic_jac_for_scipy(x, uv, obj).T @ (orc.loss_rho(f)[1] * f)


def test_cfg1_fixture_pins_the_reference_run_and_its_minimum():
    """BASELINE configs[0] (6 x 500 x 35): the reference's default bundle_adjust run (cost, nfev,
    use_frames, wall time recorded in the build container) and the tight minimum of the same objective.
    The oracle reproduces the reference's cost at both points; x_tight is stationary."""
    g = load_golden("ba_cfg1")
    use = g["use_frames"]
    uv, obj = g["uvs"][:, use], g["objpoints"]
    assert uv.shape == (6, 500, 35, 2) and not np.isnan(uv).any()
    assert int(g["nfev_default"]) > 5 and int(g["status_default"]) == 2 and float(g["wall_s_default"]) > 1.0
    ext, intr = split_cams(g["init_cams"])
    np.random.seed(0)
    use_o, _ = orc.select_frames(g["uvs"], ext, intr, obj, g["init_poses"], n_frames=None, verbose=False)
    assert np.array_equal(use_o, use)
    assert np.array_equal(orc.serialize_params(ext, intr, g["init_poses"][use]), g["x0"])
    assert orc.robust_cost(g["x_default"], uv, obj) == pytest.approx(float(g["cost_default"]), rel=1e-13)
    assert orc.robust_cost(g["x_tight"], uv, obj) == pytest.approx(float(g["cost_tight"]), rel=1e-13)
    assert float(g["cost_tight"]) < float(g["cost_default"])
    assert orc.reprojection_rms(g["x_tight"], uv, obj) == pytest.approx(float(g["rms_tight"]), rel=1e-12)
    assert np.abs(_sparse_gradient(g["x_tight"], uv, obj)).max() < 1e-6
    assert np.abs(_sparse_gradient(g["x_default"], uv, obj)).max() > 1.0      # ftol = 1e-4 stops early (SURVEY H2)
    # the default stop is within 1e-6 px RMS of the minimum at this size, but not in the parameters
    assert abs(float(g["rms_default"]) - float(g["rms_tight"])) < 1e-6


def test_sparse_polish_reaches_the_dense_minimum():
    """oracle.sparse_gauss_newton_polish (what pins x_tight at 6 x 500) against scipy's exact-solve trf
    result on the 6 x 40 fixture, from the reference's default stop."""
    g = load_golden("convergence")
    uv, obj = g["uvs"][:, g["use_frames"]], g["objpoints"]
    x, cost, gnorm = orc.sparse_gauss_newton_polish(g["x_default"], uv, obj)
    assert gnorm < 1e-5 and cost == pytest.approx(float(g["cost_tight"]), rel=1e-13)   # |g| starts at ~6e2
    a, b = x[:72].reshape(6, 12), g["x_scipy_tight"][:72].reshape(6, 12)
    np.testing.assert_allclose(a[:, :6], b[:, :6], rtol=1e-6)
    Ta, Tb = orc.relative_camera_transforms(a[:, 6:]), orc.relative_camera_transforms(b[:, 6:])
    assert np.abs(Ta - Tb).max() < 1e-6 * np.abs(Tb).max()


@pytest.mark.parametrize("name,kw", [
    ("ba_small", dict(n_cameras=4, n_frames=12, sigma=0.3, p_missing_view=0.2, p_missing_corner=0.1, seed=7)),
    ("frontend", dict(n_cameras=5, n_frames=60, sigma=0.3, p_missing_view=0.45, p_missing_corner=0.02, seed=11)),
    ("convergence", dict(n_cameras=6, n_frames=40, sigma=0.3, p_missing_view=0.15, seed=5)),
    ("ba_cfg1", dict(n_cameras=6, n_frames=500, sigma=0.3, seed=0)),
])
def test_scene_generator_has_not_drifted_from_the_fixtures(name, kw):
    """tests/golden/make_golden.py builds its scenes with synthetic.make_scene; if the generator
    changes, the committed fixtures can no longer be regenerated (`make_golden.py --check`).  The
    fixtures store their inputs, so parity would stay green -- this test is what turns red."""
    from multicam_calibration_b200.synthetic import make_scene
    g = load_golden(name)
    sc = make_scene(**kw)
    touched = {"ba_small": [(0, 0, 0, 0), (2, 5, 3, 1)], "frontend": "frame17"}.get(name)
    uvs = sc.uvs.copy()
    if name == "ba_small":
        for idx in touched:
            uvs[idx] = np.nan
    if name == "frontend":
        uvs[:, 17] += 40.0
    assert np.array_equal(uvs, g["uvs"], equal_nan=True)
    assert np.array_equal(sc.objpoints, g["objpoints"])
    if "init_cams" in g.files:
        assert np.array_equal(sc.init_cams, g["init_cams"]) and np.array_equal(sc.init_poses, g["init_poses"])
    else:
        assert np.array_equal(sc.x0(), g["x0"])


# ------------------------------------------------------------------ initialisation algebra (calibration.py)
def _tree(a):
    return [tuple(int(v) for v in e) for e in a]


@pytest.mark.parametrize("tag", ["a", "b"])
def test_initialisation_algebra_matches_reference(tag):
    g = load_golden("init")
    poses = g[f"{tag}_poses"]
    np.testing.assert_allclose(orc.estimate_pairwise_camera_transform(poses[0], poses[1]), g[f"{tag}_pair01"],
                               rtol=0, atol=1e-12)
    ext, tree = orc.estimate_all_extrinsics(poses, root=0)
    assert _tree(tree) == _tree(g[f"{tag}_tree"])
    np.testing.assert_allclose(ext, g[f"{tag}_ext"], rtol=0, atol=1e-10)
    ext2, tree2 = orc.estimate_all_extrinsics(poses, root=2)
    assert _tree(tree2) == _tree(g[f"{tag}_tree_root2"])
    np.testing.assert_allclose(ext2, g[f"{tag}_ext_root2"], rtol=0, atol=1e-10)
    cons = orc.consensus_calib_poses(poses, g[f"{tag}_ext"])
    assert np.array_equal(np.isnan(cons), np.isnan(g[f"{tag}_consensus"]))
    assert np.isnan(cons[5]).all()                                     # a frame no camera saw
    assert np.isnan(cons[6]).any() == np.isnan(poses[0, 6]).any()      # a frame only camera 0 can have seen
    np.testing.assert_allclose(cons, g[f"{tag}_consensus"], rtol=0, atol=1e-10)


def test_host_spanning_tree_orders_edges_like_the_reference():
    """The package's networkx-free spanning tree against the reference fixtures and, under heavy
    ties, against the oracle's networkx version (what the reference calls)."""
    from multicam_calibration_b200.calibration import get_camera_spanning_tree
    g = load_golden("init")
    for tag in ("a", "b"):
        assert get_camera_spanning_tree(g[f"{tag}_poses"], root=0) == _tree(g[f"{tag}_tree"])
        assert get_camera_spanning_tree(g[f"{tag}_poses"], root=2) == _tree(g[f"{tag}_tree_root2"])
    pytest.importorskip("networkx")
    rng = np.random.default_rng(1)
    for _ in range(60):
        C, F = int(rng.integers(2, 9)), int(rng.integers(1, 6))
        poses = rng.normal(size=(C, F, 6))
        poses[rng.random((C, F)) < 0.5] = np.nan
        root = int(rng.integers(0, C))
        assert get_camera_spanning_tree(poses, root=root) == _tree(orc.camera_spanning_tree(poses, root=root))


def test_transformation_vectors_match_reference():
    g = load_golden("init")
    np.testing.assert_allclose(orc.rodrigues_inv(g["R"]), g["R_vec"], rtol=0, atol=1e-15)
    np.testing.assert_allclose(orc.transformation_vector(g["T"]), g["T_vec"], rtol=0, atol=1e-15)


# ------------------------------------------------------------------ blockwise reference at scale (oracle/blockwise.py)
def _pinning_scene(lam):
    """4 cameras x 30 frames with every irregular input the blockwise reference must handle: camera 2 sees
    nothing, frames 3 and 17 are seen by no camera, a few corners are half observed (u without v), two
    frames are gross outliers (shifted by 1e3 / 1e5 px) and one pose has rotation norm 0.  At lam = 0 the
    outlier frames are left unobserved instead: their pose blocks (robust weights down to the EPS clamp)
    are too ill-conditioned for two elimination orders to agree to 1e-12 without damping."""
    from multicam_calibration_b200.synthetic import make_scene
    sc = make_scene(4, 30, sigma=0.4, p_missing_view=0.2, p_missing_corner=0.05, seed=12)
    uvs = sc.uvs.copy()
    uvs[2] = np.nan
    uvs[:, [3, 17]] = np.nan
    uvs[0, 5, 3, 1] = np.nan
    uvs[1, 6, 10, 0] = np.nan
    uvs[3, 8, 0, 1] = np.nan
    uvs[:, 11] += 1e3
    uvs[:, 23, :, 0] += 1e5
    if lam == 0.0:
        uvs[:, [11, 23]] = np.nan
    x = sc.x0()
    x[48 + 6 * 9:48 + 6 * 9 + 3] = 0.0
    return uvs, sc.objpoints, x


@pytest.mark.parametrize("loss,hessian,f_scale,lam", [
    ("linear", "triggs", 1.0, 0.0), ("linear", "triggs", 0.25, 1e-2), ("soft_l1", "triggs", 1.0, 1e-2),
    ("soft_l1", "triggs", 0.25, 0.0), ("soft_l1", "triggs", 4.0, 1e-2), ("soft_l1", "irls", 0.25, 1e-2),
    ("soft_l1", "irls", 4.0, 0.0)])
def test_blockwise_reference_matches_the_dense_oracle(loss, hessian, f_scale, lam):
    """oracle.blockwise (what the GPU tests at 50,000 frames compare the kernels with) against the dense
    normal equations of np_oracle: S, b, both gradients and the cost to 1e-12, the damped step to 1e-10.
    Chunks of 7 frames (the last one short) run the chunked accumulation."""
    from oracle import blockwise
    uvs, obj, x = _pinning_scene(lam)
    C, F = uvs.shape[:2]
    nc = 12 * C
    ev = blockwise.BlockwiseEvaluation(x, uvs, obj, lam=lam, loss=loss, f_scale=f_scale, hessian=hessian, chunk=7)
    assert np.array_equal(ev.empty, np.isnan(uvs).all((0, 2, 3))) and ev.empty[[3, 17]].all()
    H, g, cost = orc.normal_equations(x, uvs, obj, loss=loss, f_scale=f_scale, hessian=hessian)
    D2 = np.diag(H).copy()
    D2[D2 == 0.0] = 1.0
    if lam == 0.0:   # frames nobody sees contribute nothing; the dense elimination would invert their zero blocks
        keep = np.r_[np.arange(nc), nc + (np.nonzero(~ev.empty)[0][:, None] * 6 + np.arange(6)).ravel()]
        S_o, b_o = orc.reduced_camera_system(H[np.ix_(keep, keep)], g[keep], C, 0.0)
    else:
        S_o, b_o = orc.reduced_camera_system(H, g, C, lam, np.r_[np.zeros(nc), D2[nc:]])
    assert ev.cost == pytest.approx(cost, rel=1e-12)
    assert np.abs(ev.g_cam - g[:nc]).max() <= 1e-12 * np.abs(g).max()
    assert np.abs(ev.g_pose.ravel() - g[nc:]).max() <= 1e-12 * np.abs(g).max()
    assert np.abs(ev.S - S_o).max() <= 1e-12 * np.abs(S_o).max()
    assert np.abs(ev.b - b_o).max() <= 1e-12 * np.abs(b_o).max()
    assert np.array_equal(ev.diag_U, np.diag(H)[:nc]) or np.abs(ev.diag_U - np.diag(H)[:nc]).max() <= 1e-12 * np.diag(H).max()
    assert (ev.diag_U[24:36] == 0).all() and (ev.g_pose[ev.empty] == 0).all()
    if lam:
        step = ev.step()
        step_o = orc.lm_step(H, g, C, lam, D2)
        assert np.abs(step - step_o).max() <= 1e-10 * np.abs(step_o).max()
        assert (step[nc:].reshape(F, 6)[ev.empty] == 0).all()
        S2, b2, gc2, gp2, c2 = blockwise.reduced_camera_system_blockwise(x, uvs, obj, lam, loss, f_scale, hessian)
        assert np.abs(S2 - ev.S).max() <= 1e-13 * np.abs(S_o).max() and c2 == pytest.approx(ev.cost, rel=1e-14)
