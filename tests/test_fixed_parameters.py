"""Camera parameters held at their initial values (``fixed=`` of ``bundle_adjust`` / ``BAProblem.solve`` /
``calibration_covariance``, ``BAProblem.set_fixed``, ``mcba_set_fixed``).

CPU: the masked blockwise step against the dense damped system restricted to the free columns, the masked
covariance references against each other and against scipy's ``res.jac`` recipe on the sub-problem, and
argument validation.  GPU: a mask that holds nothing changes nothing; a masked solve launches what an unmasked
one does; the masked step of every solve tier against the reference; convergence against scipy on the free
sub-problem; a pinned camera against the gauge-normalised free solve; pose-only refinement; the masked
covariance against its reference and against the scatter of solutions; the error paths; the sharded solve."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import multicam_calibration_b200 as mcc
from conftest import ROOT, load_golden
from multicam_calibration_b200.synthetic import forward_model, make_scene
from oracle import blockwise
from oracle import np_oracle as orc
import fixed_reference as fref
from test_gpu_parity import assert_cameras_match

LAM = 1e-3


def masks(C, seed=0):
    """name -> (C, 12) bool: the masks every step comparison runs."""
    out = {k: np.zeros((C, 12), dtype=bool) for k in ("intrinsics", "k2", "cam0_pinned", "random30", "all")}
    out["intrinsics"][:, :6] = True
    out["k2"][:, 5] = True
    out["cam0_pinned"][0, 6:] = True
    out["random30"] = np.random.default_rng(seed).random((C, 12)) < 0.3
    out["all"][:] = True
    return out


def _normalised_diff(A, B):
    """max |A - B| / sqrt(B_ii B_jj) over the finite entries of B (NaN / zero patterns must match)."""
    assert np.array_equal(np.isnan(A), np.isnan(B))
    d = np.sqrt(np.abs(np.einsum("...ii->...i", np.nan_to_num(B))))
    scale = d[..., :, None] * d[..., None, :]
    fin = ~np.isnan(B) & (scale > 0)
    assert (A[~np.isnan(B) & (scale == 0)] == 0).all()
    return float((np.abs(A - B)[fin] / scale[fin]).max()) if fin.any() else 0.0


def _cond_scaled(camera):
    keep = np.isfinite(np.diag(camera)) & (np.diag(camera) > 0)
    if not keep.any():
        return 1.0
    A = camera[np.ix_(keep, keep)]
    d = np.sqrt(np.diag(A))
    return float(np.linalg.cond(A / d[:, None] / d[None, :]))


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", ["intrinsics", "k2", "cam0_pinned", "random30", "all"])
def test_masked_blockwise_step_is_the_restricted_dense_step(name):
    sc = make_scene(3, 12, sigma=0.4, p_missing_view=0.2, p_missing_corner=0.05, seed=2)
    x, uvs, obj = sc.x0(), sc.uvs, sc.objpoints
    fixed = masks(3, seed=1)[name]
    lam = 1e-2
    H, g, _ = orc.normal_equations(x, uvs, obj)
    D2 = np.diag(H).copy()
    D2[D2 == 0] = 1.0
    free = np.concatenate([~fixed.ravel(), np.ones(H.shape[0] - 36, dtype=bool)])
    want = np.zeros(H.shape[0])
    Hd = H + lam * np.diag(D2)
    want[free] = -np.linalg.solve(Hd[np.ix_(free, free)], g[free])
    got = fref.masked_step(blockwise.BlockwiseEvaluation(x, uvs, obj, lam=lam), fixed)
    assert (got[:36][fixed.ravel()] == 0).all()
    assert np.abs(got - want).max() <= 1e-10 * np.abs(want).max()


@pytest.mark.parametrize("ref,name", [(0, "intrinsics"), (None, "cam0_pinned"), (2, "cam2_pinned"), (None, "all")])
def test_masked_blockwise_covariance_matches_dense(ref, name):
    sc = make_scene(4, 40, sigma=0.4, p_missing_view=0.2, p_missing_corner=0.05, seed=3)
    uvs = sc.uvs.copy()
    uvs[1] = np.nan                                  # held rows win over the NaN of an unobserved camera
    x, obj = sc.x0(), sc.objpoints
    fixed = np.zeros((4, 12), dtype=bool)
    if name == "intrinsics":
        fixed[:, :6] = True
    elif name == "cam0_pinned":
        fixed[0, 6:] = True
        fixed[3, 4:6] = True
    elif name == "cam2_pinned":
        fixed[2, 6:] = True
    else:
        fixed[:] = True
    d = fref.dense_covariance(x, uvs, obj, ref, fixed=fixed)
    b = fref.blockwise_covariance(x, uvs, obj, ref, fixed=fixed)
    assert abs(b["sigma2"] - d["sigma2"]) <= 1e-12 * d["sigma2"] and b["dof"] == d["dof"]
    tol = max(1e-10, 1e-13 * _cond_scaled(d["camera"]))
    assert _normalised_diff(b["camera"], d["camera"]) <= tol
    assert _normalised_diff(b["poses"], d["poses"]) <= tol
    held = fixed.ravel()
    assert (d["camera"][held] == 0).all() and (d["camera"][:, held] == 0).all()
    cam1 = np.repeat(np.arange(4) == 1, 12)
    assert np.isnan(d["camera"][np.ix_(cam1 & ~held, ~held)]).all()


def test_masked_dense_covariance_matches_scipy_result_jac():
    """Intrinsics held and camera 0 pinned: ``inv(J^T J) 2 cost / (m - p)`` from ``least_squares``' ``res.jac`` on
    the free sub-problem."""
    from scipy.optimize import least_squares
    sc = make_scene(3, 25, sigma=0.5, p_missing_view=0.1, seed=5)
    uvs, obj, x0 = sc.uvs, sc.objpoints, sc.x0()
    fixed = np.zeros((3, 12), dtype=bool)
    fixed[:, :6] = True
    fixed[0, 6:] = True
    free = np.concatenate([~fixed.ravel(), np.ones(6 * 25, dtype=bool)])

    def full(z):
        x = x0.copy()
        x[free] = z
        return x
    res = least_squares(lambda z: orc.residuals(full(z), uvs, obj), x0[free],
                        jac=lambda z: orc.analytic_jac_for_scipy(full(z), uvs, obj)[:, free], loss="soft_l1",
                        method="trf", x_scale="jac", ftol=1e-15, xtol=1e-15, gtol=1e-15, max_nfev=200)
    J = res.jac.toarray() if hasattr(res.jac, "toarray") else np.asarray(res.jac)
    m, p = J.shape
    cov = np.linalg.inv(J.T @ J) * 2 * res.cost / (m - p)
    d = fref.dense_covariance(full(res.x), uvs, obj, None, "soft_l1", fixed=fixed)
    want = np.zeros((free.size, free.size))
    want[np.ix_(free, free)] = cov
    assert abs(d["sigma2"] - 2 * res.cost / (m - p)) <= 1e-10 * d["sigma2"]
    assert _normalised_diff(d["camera"], want[:36, :36]) <= 1e-8
    poses = np.stack([want[36 + 6 * i:42 + 6 * i, 36 + 6 * i:42 + 6 * i] for i in range(25)])
    assert _normalised_diff(d["poses"], poses) <= 1e-8


def test_mask_validation_without_cuda():
    sc = make_scene(3, 10, seed=1)
    ext, intr, poses = orc.deserialize_params(sc.x0(), 3)
    args = (sc.uvs, ext, intr, sc.objpoints, poses)
    bad = (np.zeros((3, 11), dtype=bool), np.zeros((2, 12), dtype=bool), np.zeros(36, dtype=bool),
           np.zeros((3, 12), dtype=int), np.zeros((3, 12)), [[0] * 12] * 3)
    for fixed in bad:
        with pytest.raises(ValueError, match="fixed"):
            mcc.calibration_covariance(*args, fixed=fixed)
        with pytest.raises(ValueError, match="fixed"):
            mcc.bundle_adjust(*args, fixed=fixed)
    with pytest.raises(ValueError):
        mcc.calibration_covariance(*args, reference_camera=1.0)
    # the oracle's gauge rule (the engine's is tested on the GPU)
    pin = np.zeros((3, 12), dtype=bool)
    pin[0, 6:] = True
    part = np.zeros((3, 12), dtype=bool)
    part[1, 6:9] = True
    assert fref.gauge(3, None, pin) is None and fref.gauge(3, 0, pin) is None and fref.gauge(3, 2, None) == 2
    for ref, fixed in ((1, pin), (None, None), (None, part), (0, part)):
        with pytest.raises(ValueError):
            fref.gauge(3, ref, fixed)


# ------------------------------------------------------------------ GPU
def _scene(C, F, p=0.2, seed=0, sigma=0.5):
    sc = make_scene(C, F, sigma=sigma, p_missing_view=p, seed=seed)
    return np.ascontiguousarray(sc.uvs), sc.objpoints, sc.x0()


@pytest.mark.gpu
def test_no_mask_is_the_unmasked_solve():
    """``fixed`` omitted, None and all False: bit-identical solve, same evaluations and launches (ba_cfg1)."""
    g = load_golden("ba_cfg1")
    use = g["use_frames"]
    uv, obj = g["uvs"][:, use], g["objpoints"]
    out = []
    for kw in ({}, dict(fixed=None), dict(fixed=np.zeros((6, 12), dtype=bool))):
        prob = mcc.BAProblem(uv, obj)
        x, res = prob.solve(g["x0"], verbose=0, **kw)
        out.append((x, res))
        prob.close()
    for x, res in out[1:]:
        assert np.array_equal(x.view(np.int64), out[0][0].view(np.int64))
        for k in ("cost", "nfev", "njev", "status", "kernel_launches", "optimality"):
            assert res[k] == out[0][1][k], k


@pytest.mark.gpu
def test_masked_solve_adds_no_launches():
    """Same number of evaluations (a fixed budget, Triggs weights throughout): the same kernel launches."""
    g = load_golden("ba_cfg1")
    use = g["use_frames"]
    uv, obj = g["uvs"][:, use], g["objpoints"]
    prob = mcc.BAProblem(uv, obj)
    kw = dict(hessian="triggs", max_nfev=6, ftol=1e-15, xtol=1e-15, gtol=1e-15, verbose=0)
    _, r0 = prob.solve(g["x0"], **kw)
    for name, fixed in masks(6).items():
        _, r = prob.solve(g["x0"], fixed=fixed, **kw)
        assert r.nfev == r0.nfev == 6 and r.kernel_launches == r0.kernel_launches, name


# masked damped step against the reference, every solve tier: name -> (builder, expected tier, environment)
TIERS = {
    "6x50000": (lambda: _scene(6, 50000), "regs3", None),
    "10x8000": (lambda: _scene(10, 8000, seed=11), "regs8", None),
    "16x8000": (lambda: _scene(16, 8000, seed=16), "smem19", None),
    "6x8000_cusolver": (lambda: _scene(6, 8000, seed=1), "cusolver", {"MCBA_CUSOLVER": "1"}),
    "20x2000": (lambda: _scene(20, 2000, seed=20), "cusolver", None),
}


def tier_scene(name):
    """The scene with camera 0's k2 set to -0.0 (held by the "k2" mask: it must come back as -0.0)."""
    uvs, obj, x0 = TIERS[name][0]()
    x0 = x0.copy()
    x0[5] = -0.0
    return uvs, obj, x0


def engine_masked_steps(name):
    """``{mask: x_new}`` and the plan from ``build_reduced`` + ``set_fixed`` + ``solve_step`` in this process."""
    uvs, obj, x0 = tier_scene(name)
    prob = mcc.BAProblem(uvs, obj)
    prob.build_reduced(x0, lam=LAM)
    steps = {}
    for k, fixed in masks(prob.C).items():
        prob.set_fixed(fixed)
        steps[k] = prob.solve_step(LAM)
    prob.set_fixed(None)
    plan = prob.plan_info()
    prob.close()
    return steps, plan["solve"]


_CHILD = r"""
import sys, json, numpy as np
sys.path.insert(0, {root!r})
sys.path.insert(0, {tests!r})
import test_fixed_parameters as t
steps, tier = t.engine_masked_steps({name!r})
np.savez({out!r}, **steps)
print(json.dumps(tier))
"""


def compare_masked_step(tag, ref_step, x_new, x0, fixed, empty):
    nc = fixed.size
    held = fixed.ravel()
    d = x_new - x0
    dc, dc_ref = d[:nc], ref_step[:nc]
    assert np.array_equal(x_new[:nc][held].view(np.int64), x0[:nc][held].view(np.int64)), f"{tag}: held entries moved"
    assert (dc_ref[held] == 0).all()
    err_c = np.abs(dc - dc_ref)[~held].max() / np.abs(dc_ref).max() if (~held).any() else 0.0
    dp, dp_ref = d[nc:].reshape(-1, 6), ref_step[nc:].reshape(-1, 6)
    tol_p = 1e-6 * np.abs(dp_ref).max(1) + 1e-9 * np.abs(dp_ref).max()
    err_p = (np.abs(dp - dp_ref).max(1) / (np.abs(dp_ref).max(1) + 1e-3 * np.abs(dp_ref).max())).max()
    print(f"\n[{tag}] step_cam {err_c:.1e}  step_pose {err_p:.1e}")
    assert err_c <= 1e-6, tag
    assert (np.abs(dp - dp_ref).max(1) <= tol_p).all(), tag
    assert np.array_equal(x_new[nc:].reshape(-1, 6)[empty], x0[nc:].reshape(-1, 6)[empty])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TIERS))
def test_masked_step_matches_the_reference(name, tmp_path):
    _, tier, env = TIERS[name]
    if env is None:
        steps, got_tier = engine_masked_steps(name)
    else:
        out = str(tmp_path / "steps.npz")
        code = _CHILD.format(root=ROOT, tests=os.path.join(ROOT, "tests"), name=name, out=out)
        run = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900,
                             env=dict(os.environ, **env))
        assert run.returncode == 0, run.stderr[-3000:]
        got_tier = json.loads(run.stdout.strip().splitlines()[-1])
        steps = dict(np.load(out))
    assert got_tier == tier
    uvs, obj, x0 = tier_scene(name)
    ev = blockwise.BlockwiseEvaluation(x0, uvs, obj, lam=LAM)
    for k, fixed in masks(ev.C).items():
        compare_masked_step(f"{name} {k}", fref.masked_step(ev, fixed), steps[k], x0, fixed, ev.empty)
    assert np.signbit(steps["k2"][5]) and np.signbit(steps["all"][5])


def _solve_free_with_scipy(x0, uvs, obj, fixed):
    from scipy.optimize import least_squares
    nc = fixed.size
    free = np.concatenate([~fixed.ravel(), np.ones(x0.size - nc, dtype=bool)])

    def full(z):
        x = x0.copy()
        x[free] = z
        return x
    res = least_squares(lambda z: orc.residuals(full(z), uvs, obj), x0[free],
                        jac=lambda z: orc.analytic_jac_for_scipy(full(z), uvs, obj)[:, free].toarray(),   # dense: exact solve
                        loss="soft_l1", method="trf", x_scale="jac", ftol=1e-15, xtol=1e-15, gtol=1e-15, max_nfev=300)
    return full(res.x), res.cost


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["intrinsics_at_truth", "cam0_pinned"])
def test_masked_solve_converges_to_scipy_on_the_sub_problem(case):
    sc = make_scene(4, 40, sigma=0.3, p_missing_view=0.15, seed=5)
    uvs, obj, x0 = sc.uvs, sc.objpoints, sc.x0()
    fixed = np.zeros((4, 12), dtype=bool)
    if case == "intrinsics_at_truth":
        x0[:48].reshape(4, 12)[:, :6] = sc.true_cams[:, :6]
        fixed[:, :6] = True
    else:
        fixed[0, 6:] = True
    xs, cost_s = _solve_free_with_scipy(x0, uvs, obj, fixed)
    x, res = mcc.BAProblem(uvs, obj).solve(x0, fixed=fixed, ftol=1e-15, xtol=1e-15, gtol=1e-9, max_nfev=300,
                                           verbose=0)
    held = fixed.ravel()
    print(f"\n[{case}] cost {res.cost:.12e} scipy {cost_s:.12e} nfev {res.nfev} optimality {res.optimality:.1e}")
    assert np.array_equal(x[:48][held], x0[:48][held])
    assert res.cost <= cost_s * (1 + 1e-10)
    assert abs(res.cost - orc.robust_cost(x, uvs, obj)) <= 1e-10 * res.cost
    assert res.optimality < 1e-6
    assert_cameras_match(x, xs, 4)
    if case == "cam0_pinned":                                # no gauge left: the same point, not only the same shape
        cams, cams_s = x[:48].reshape(4, 12), xs[:48].reshape(4, 12)
        assert (np.abs(cams - cams_s) <= 1e-6 * np.abs(cams_s).max(axis=0)).all()
    assert res.grad.shape == x.shape and np.abs(res.grad[:48][held]).max() > 0    # the full gradient


def _align_to_reference(x, x_ref, C, ref=0):
    """Rigid change of world frame that puts camera ``ref`` at its extrinsics in ``x_ref``."""
    cams = x[:12 * C].reshape(C, 12).copy()
    poses = x[12 * C:].reshape(-1, 6).copy()
    tc = x_ref[:12 * C].reshape(C, 12)[ref]
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
def test_pinned_camera_is_the_free_solve_in_its_frame():
    """6 x 50,000: camera 0's extrinsics held remove the gauge -- same minimum, the free solution moved into
    camera 0's initial frame, camera 0 untouched."""
    uvs, obj, x0 = _scene(6, 50000)
    prob = mcc.BAProblem(uvs, obj)
    kw = dict(ftol=1e-12, xtol=1e-15, gtol=1e-12, verbose=0)
    xf, rf = prob.solve(x0, **kw)
    fixed = np.zeros((6, 12), dtype=bool)
    fixed[0, 6:] = True
    xp, rp = prob.solve(x0, fixed=fixed, **kw)
    print(f"\ncost free {rf.cost:.12e} ({rf.nfev} nfev)  pinned {rp.cost:.12e} ({rp.nfev} nfev)")
    assert np.array_equal(xp[6:12].view(np.int64), x0[6:12].view(np.int64))
    assert abs(rp.cost - rf.cost) <= 1e-10 * rf.cost
    xa = _align_to_reference(xf, x0, 6)
    cams, cams_a = xp[:72].reshape(6, 12), xa[:72].reshape(6, 12)
    err_c = (np.abs(cams - cams_a) / np.abs(cams_a).max(axis=0)).max()
    # frames without observations keep their initial pose in either world frame: not comparable; rotations as
    # matrices (an rvec near pi has two representations)
    seen = ~np.isnan(uvs).all(axis=(0, 2, 3))
    poses, poses_a = xp[72:].reshape(-1, 6)[seen], xa[72:].reshape(-1, 6)[seen]
    err_r = np.abs(orc.rodrigues(poses[:, :3]) - orc.rodrigues(poses_a[:, :3])).max()
    err_t = (np.abs(poses[:, 3:] - poses_a[:, 3:]) / np.abs(poses_a[:, 3:]).max(axis=0)).max()
    print(f"aligned free solution against the pinned one: cameras {err_c:.1e}  pose rotations {err_r:.1e}  "
          f"translations {err_t:.1e} ({int((~seen).sum())} frames without observations left out)")
    assert err_c <= 1e-6 and err_r <= 1e-6 and err_t <= 1e-6


@pytest.mark.gpu
def test_pose_only_refinement():
    """6 x 50,000, every camera parameter held: cameras bit-identical, poses equal per-frame scipy solves."""
    from scipy.optimize import least_squares
    uvs, obj, x0 = _scene(6, 50000)
    fixed = np.ones((6, 12), dtype=bool)
    x, res = mcc.BAProblem(uvs, obj).solve(x0, fixed=fixed, ftol=1e-12, xtol=1e-15, gtol=1e-12, verbose=0)
    assert np.array_equal(x[:72].view(np.int64), x0[:72].view(np.int64))
    assert res.success and res.cost < res.initial_cost
    rng = np.random.default_rng(7)
    worst = 0.0
    for f in rng.choice(50000, 24, replace=False):
        if np.isnan(uvs[:, f]).all():
            continue
        u = uvs[:, f:f + 1]

        def full(z):
            return np.concatenate([x0[:72], z])
        r = least_squares(lambda z: orc.residuals(full(z), u, obj), x0[72 + 6 * f:78 + 6 * f],
                          jac=lambda z: orc.analytic_jac_for_scipy(full(z), u, obj)[:, 72:], loss="soft_l1",
                          x_scale="jac", ftol=1e-15, xtol=1e-15, gtol=1e-15, max_nfev=200)
        p = x[72 + 6 * f:78 + 6 * f]
        worst = max(worst, float((np.abs(p - r.x) / np.array([1, 1, 1, 100, 100, 100.0])).max()))
    print(f"\npose-only: {res.nfev} nfev, worst pose difference (rad, 100 mm units) {worst:.1e}")
    assert worst <= 1e-7


COV = {"intrinsics": 0, "cam0_pinned": None, "all": None}   # mask name -> reference_camera


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(COV))
def test_masked_covariance_matches_the_reference(name):
    uvs, obj, x = _scene(6, 50000)
    ref, fixed = COV[name], masks(6)[name]
    cam, poses, info = mcc.BAProblem(uvs, obj).covariance(x, reference_camera=ref, fixed=fixed)
    want = fref.blockwise_covariance(x, uvs, obj, ref, fixed=fixed)
    e_cam, e_pose = _normalised_diff(cam, want["camera"]), _normalised_diff(poses, want["poses"])
    print(f"\n[{name}] camera {e_cam:.2e}  poses {e_pose:.2e}  s2 {info['sigma2']:.6g}  dof {info['dof']:.0f}  "
          f"device ms eval {info['eval_ms']:.3f} camera {info['camera_ms']:.3f} poses {info['pose_ms']:.3f}")
    tol = max(1e-7, 1e-13 * _cond_scaled(want["camera"]))
    assert e_cam <= tol and e_pose <= tol
    assert abs(info["sigma2"] - want["sigma2"]) <= 1e-12 * want["sigma2"] and info["dof"] == want["dof"]
    held = fixed.ravel()
    assert (cam[held] == 0).all() and (cam[:, held] == 0).all()


@pytest.mark.gpu
def test_masked_covariance_predicts_the_scatter_of_solutions():
    """Linear loss, 6 x 300, sigma = 0.5 px, intrinsics and camera 0 held at the truth, 32 noisy solves."""
    C, F, sigma = 6, 300, 0.5
    sc = make_scene(C, F, sigma=sigma, p_missing_view=0.2, seed=11)
    x_true = np.concatenate([sc.true_cams.ravel(), sc.true_poses.ravel()])
    clean = forward_model(sc.true_cams, sc.true_poses, sc.objpoints)
    miss = np.isnan(sc.uvs)
    fixed = np.zeros((C, 12), dtype=bool)
    fixed[:, :6] = True
    fixed[0, 6:] = True
    prob = mcc.BAProblem(np.where(miss, np.nan, clean), sc.objpoints)
    cam, poses, _ = prob.covariance(x_true, reference_camera=None, loss="linear", sigma=sigma, fixed=fixed)
    free = ~fixed.ravel()
    cam_inv = np.linalg.inv(cam[np.ix_(free, free)])
    pose_inv = np.linalg.inv(poses)
    d_cam, d_pose = [], []
    rng = np.random.default_rng(12)
    for _ in range(32):
        prob.set_observations(np.where(miss, np.nan, clean + rng.normal(0, sigma, clean.shape)))
        x, res = prob.solve(x_true, fixed=fixed, loss="linear", ftol=1e-14, xtol=1e-14, gtol=1e-12, max_nfev=100,
                            verbose=0)
        e = (x - x_true)[:12 * C][free]
        d_cam.append(e @ cam_inv @ e / free.sum())
        ep = (x - x_true)[12 * C:].reshape(F, 6)
        d_pose.append(np.einsum("fi,fij,fj->", ep, pose_inv, ep) / (6 * F))
    print(f"\nMahalanobis^2 per dimension: cameras {np.mean(d_cam):.4f} ({free.sum()} parameters), "
          f"poses {np.mean(d_pose):.4f}")
    assert free.sum() == 30
    assert 0.8 <= np.mean(d_cam) <= 1.2
    assert 0.9 <= np.mean(d_pose) <= 1.1


@pytest.mark.gpu
def test_mask_errors():
    import ctypes
    from multicam_calibration_b200 import _native
    uvs, obj, x = _scene(4, 200, seed=4, p=0.0)
    prob = mcc.BAProblem(uvs, obj)
    pin = np.zeros((4, 12), dtype=bool)
    pin[0, 6:] = True
    part = np.zeros((4, 12), dtype=bool)
    part[2, 9:] = True
    with pytest.raises(ValueError, match="reference_camera 1 is not such a camera"):
        prob.covariance(x, reference_camera=1, fixed=pin)
    with pytest.raises(ValueError, match="gauge is not fixed"):
        prob.covariance(x, reference_camera=None)
    with pytest.raises(ValueError, match="some extrinsic parameters"):
        prob.covariance(x, reference_camera=0, fixed=part)
    with pytest.raises(ValueError, match="fixed must have shape"):
        prob.solve(x, fixed=pin[:3], verbose=0)
    with pytest.raises(ValueError, match="boolean"):
        prob.set_fixed(pin.astype(np.uint8))
    two = np.zeros(48, dtype=np.uint8)
    two[7] = 2
    assert prob.lib.mcba_set_fixed(prob._h, two.ctypes.data_as(ctypes.c_void_p)) == _native.ERR_ARG
    assert "0 (free) or 1 (held)" in prob.lib.mcba_last_error().decode()
    cam, _, _ = prob.covariance(x, reference_camera=0, fixed=pin)      # a pinned reference camera is accepted
    cam2, _, _ = prob.covariance(x, reference_camera=None, fixed=pin)
    assert np.array_equal(cam, cam2)
    # each call sets its own mask: nothing is inherited from the previous one
    _, r1 = prob.solve(x, verbose=0)
    prob.solve(x, fixed=pin, verbose=0)
    _, r2 = prob.solve(x, verbose=0)
    assert r1.cost == r2.cost and r1.nfev == r2.nfev


@pytest.mark.gpu
def test_bundle_adjust_and_calibration_covariance_take_the_mask():
    sc = make_scene(6, 500, sigma=0.3, p_missing_view=0.2, seed=7)
    ext, intr, poses = orc.deserialize_params(sc.x0(), 6)
    fixed = np.zeros((6, 12), dtype=bool)
    fixed[:, :6] = True
    fixed[2, 6:] = True
    np.random.seed(0)
    e, i, p, use, res = mcc.bundle_adjust(sc.uvs, ext, intr, sc.objpoints, poses, n_frames=None, verbose=0, fixed=fixed)
    x0 = mcc.serialize_params(ext, intr, poses[use])
    assert np.array_equal(res.x[:72][fixed.ravel()], x0[:72][fixed.ravel()])
    assert np.array_equal(e[2], np.asarray(ext[2]))
    cov = mcc.calibration_covariance(sc.uvs[:, use], e, i, sc.objpoints, p, reference_camera=None, fixed=fixed)
    assert (cov.camera_std[fixed] == 0).all() and (cov.camera_std[~fixed] > 0).all()
    assert np.isfinite(cov.pose_std).all()


@pytest.mark.gpu
def test_sharded_masked_solve_matches_single_gpu():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29617",
           os.path.join(ROOT, "scripts", "fixed_params_multigpu_check.py"), "997"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "FIXED_MULTIGPU_OK" in out.stdout
