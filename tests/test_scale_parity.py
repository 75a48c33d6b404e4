"""GPU: the reduced camera system, gradient, damped step and predictions at production sizes and for every
kernel variant, against the blockwise fp64 reference (oracle/blockwise.py, pinned to the dense oracle by
tests/test_oracle_golden.py).

The dense oracle stops at a few hundred frames, where K2p runs with 1-4 warps per CTA and K2c, the SYRK,
finalize and the back-substitution see a handful of tiles.  Each scenario below is chosen for the branch
of the launch heuristics it reaches (K2p width, rounds of the static schedule and the split half-unit
tail; K2c ring / streamed pair; static or run-time SYRK tile lists and their CTA rows; the solve tier);
``mcba_plan_info`` reports what the handle actually chose and the last test asserts that the scenario set
reached every branch, so a changed heuristic shows up as lost coverage instead of a quiet pass.

Comparisons are element-wise and scaled so that one wrong frame out of 50,000 cannot hide in a norm; the
measured maxima are printed (``pytest -s``) to show the margin the tolerances leave."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import blockwise
import multicam_calibration_b200 as mcc
from multicam_calibration_b200.synthetic import forward_model, make_scene

pytestmark = pytest.mark.gpu

LAM = 1e-3


# ------------------------------------------------------------------ scenarios
def _rotation_scene():
    """6 x 3000: camera 0 at rvec = 0 exactly (what estimate_all_extrinsics gives the root camera) and
    board rotations of norm 0, 1e-9, 0.0999, 0.1001 (either side of the series switch of
    so3_left_jacobian) and 3.1415 (near pi), 40 frames each."""
    sc = make_scene(6, 3000, sigma=0.4, p_missing_view=0.2, seed=31)
    cams, poses = sc.true_cams.copy(), sc.true_poses.copy()
    cams[0, 6:9] = 0.0
    cams[0, 9:12] = [0.0, 0.0, 600.0]
    rng = np.random.default_rng(31)
    axes = rng.normal(size=(200, 3))
    axes /= np.linalg.norm(axes, axis=1, keepdims=True)
    norms = np.repeat([0.0, 1e-9, 0.0999, 0.1001, 3.1415], 40)
    poses[:200, :3] = axes * norms[:, None]
    uvs = forward_model(cams, poses, sc.objpoints) + rng.normal(0, 0.4, (6, 3000, 35, 2))
    uvs[np.isnan(sc.uvs)] = np.nan
    init_cams = sc.init_cams.copy()
    init_cams[0, 6:9] = 0.0
    init_cams[0, 9:12] = cams[0, 9:12] + rng.normal(0, 2, 3)
    init_poses = sc.init_poses.copy()
    init_poses[:200, :3] = poses[:200, :3]
    return uvs, sc.objpoints, np.concatenate([init_cams.ravel(), init_poses.ravel()])


def _outlier_scene():
    """6 x 3000 with 2 % of the frames shifted by 1e3 - 1e5 px: the robust weights reach the EPS clamp."""
    sc = make_scene(6, 3000, sigma=0.4, p_missing_view=0.2, seed=32)
    uvs = sc.uvs.copy()
    rng = np.random.default_rng(32)
    bad = rng.choice(3000, 60, replace=False)
    uvs[:, bad] += (10.0 ** rng.uniform(3, 5, 60))[None, :, None, None] * rng.choice([-1.0, 1.0], (1, 60, 1, 2))
    return uvs, sc.objpoints, sc.x0()


def _scene(C, F, p=0.2, board=(5, 7), seed=0, sigma=0.5):
    sc = make_scene(C, F, board=board, sigma=sigma, p_missing_view=p, seed=seed)
    return sc.uvs, sc.objpoints, sc.x0()


def _without_camera(c):
    def build():
        uvs, obj, x = _scene(6, 50000)
        uvs[c] = np.nan
        return uvs, obj, x
    return build


# name -> (builder, loss, f_scale); the bench scene is BASELINE configs[2] as bench.py builds it
SCENARIOS = {
    "bench_6x50000": (lambda: _scene(6, 50000), "soft_l1", 1.0),
    "6x8000": (lambda: _scene(6, 8000, seed=1), "soft_l1", 1.0),
    "2x30000": (lambda: _scene(2, 30000, p=0.0, seed=2), "soft_l1", 1.0),
    "3x20000": (lambda: _scene(3, 20000, seed=3), "soft_l1", 1.0),
    "6x12000": (lambda: _scene(6, 12000, seed=4), "soft_l1", 1.0),
    "6x6400": (lambda: _scene(6, 6400, seed=5), "soft_l1", 1.0),
    "6x50000_no_cam2": (_without_camera(2), "soft_l1", 1.0),
    "6x50000_no_cam5": (_without_camera(5), "soft_l1", 1.0),
    "6x50000_all_views": (lambda: _scene(6, 50000, p=0.0, seed=6), "soft_l1", 1.0),
    "6x50000_70pc_missing": (lambda: _scene(6, 50000, p=0.7, seed=7), "soft_l1", 1.0),
    "1x40000": (lambda: _scene(1, 40000, p=0.0, seed=8), "soft_l1", 1.0),
    "8x4000": (lambda: _scene(8, 4000, seed=9), "soft_l1", 1.0),
    "9x4000": (lambda: _scene(9, 4000, seed=10), "soft_l1", 1.0),
    "10x4000": (lambda: _scene(10, 4000, seed=11), "soft_l1", 1.0),
    "11x4000": (lambda: _scene(11, 4000, seed=12), "soft_l1", 1.0),
    "13x6000": (lambda: _scene(13, 6000, seed=13), "soft_l1", 1.0),
    "14x3000": (lambda: _scene(14, 3000, seed=14), "soft_l1", 1.0),
    "15x3000": (lambda: _scene(15, 3000, seed=15), "soft_l1", 1.0),
    "16x8000": (lambda: _scene(16, 8000, seed=16), "soft_l1", 1.0),
    "17x2000": (lambda: _scene(17, 2000, seed=17), "soft_l1", 1.0),
    "24x2000": (lambda: _scene(24, 2000, seed=18), "soft_l1", 1.0),
    "32x2000": (lambda: _scene(32, 2000, seed=19), "soft_l1", 1.0),
    "6x8000_n36": (lambda: _scene(6, 8000, board=(6, 6), seed=20), "soft_l1", 1.0),
    "6x8000_n99": (lambda: _scene(6, 8000, board=(9, 11), seed=21), "soft_l1", 1.0),
    "6x2000_n1": (lambda: _scene(6, 2000, board=(1, 1), seed=22), "soft_l1", 1.0),
    "6x2000_n2": (lambda: _scene(6, 2000, board=(1, 2), seed=23), "soft_l1", 1.0),
    "6x2000_n140": (lambda: _scene(6, 2000, board=(10, 14), seed=24), "soft_l1", 1.0),
    "6x3000_rotations": (_rotation_scene, "soft_l1", 1.0),
    "6x3000_outliers_fs0.25": (_outlier_scene, "soft_l1", 0.25),
    "6x3000_outliers_fs4": (_outlier_scene, "soft_l1", 4.0),
    "6x3000_outliers_linear": (_outlier_scene, "linear", 1.0),
    "6x3000_outliers_irls": (_outlier_scene, "soft_l1_irls", 1.0),
}

# One- and two-corner boards leave part of every pose block without information (a rotation about the board
# origin, resp. about the line through both corners).  The engine's pose blocks carry rounding there, where the
# reference has exact zeros (damping D^2 = 1), so the damped pose steps of those frames differ along that null
# direction; everything else of these scenes -- S, b, gradients, cost and the camera step -- is compared.
RANK_DEFICIENT_POSES = {"6x2000_n1", "6x2000_n2"}

_REFS = {}      # name -> compact reference at x0 (module-wide: the forced variants and the solves reuse it)
_PLANS = {}     # name -> launch choices reported by mcba_plan_info + the K2p schedule derived from them


def build(name):
    fn, loss, f_scale = SCENARIOS[name]
    uvs, obj, x = fn()
    return np.ascontiguousarray(uvs), obj, x, loss, f_scale


def _hessian(loss):
    return ("irls" if loss.endswith("_irls") else "triggs"), loss.replace("_irls", "")


def evaluate_reference(uvs, obj, x, lam, loss, f_scale):
    hessian, base = _hessian(loss)
    return blockwise.BlockwiseEvaluation(x, uvs, obj, lam=lam, loss=base, f_scale=f_scale, hessian=hessian)


def reference(name, uvs=None, obj=None, x=None):
    """Compact reference of a scenario at x0 and LAM (computed once per module)."""
    if name not in _REFS:
        if uvs is None:
            uvs, obj, x, _, _ = build(name)
        _, loss, f_scale = SCENARIOS[name]
        ev = evaluate_reference(uvs, obj, x, LAM, loss, f_scale)
        _REFS[name] = dict(S=ev.S, b=ev.b, g_cam=ev.g_cam, g_pose=ev.g_pose, cost=ev.cost, step=ev.step(),
                           empty=ev.empty, C=ev.C)
    return _REFS[name]


def k2p_schedule(plan):
    """Rounds, leftover groups and the split-tail predicate of the K2p schedule, with the kernel's own
    formula (csrc/k2_producer.cuh) applied to the live units per camera the handle reports."""
    C, w, grid, units = plan["cameras"], plan["k2p_warps"], plan["k2p_grid"], plan["units"]
    gp = np.r_[0, np.cumsum([(u + w - 1) // w for u in units])]
    n_groups = int(gp[-1])
    rounds, left = n_groups // grid, n_groups % grid
    tc = 0
    while tc + 1 < C and gp[tc + 1] <= rounds * grid:
        tc += 1
    tail_units = units[tc] - (rounds * grid - gp[tc]) * w if left > 0 else 0
    per_cta = (2 * tail_units + grid - 1) // grid
    split = w == 8 and rounds >= 1 and left > 0 and per_cta <= w and gp[tc + 1] >= n_groups
    return dict(rounds=int(rounds), left=int(left), split_tail=bool(split), tail_units=int(tail_units))


def record_plan(name, prob):
    plan = prob.plan_info()
    plan.update(k2p_schedule(plan))
    plan["N"] = prob.N
    _PLANS[name] = plan
    return plan


# ------------------------------------------------------------------ comparisons
def compare_system(tag, ref, S, b, g_cam, cost, grad=None, x_new=None, x0=None, pose_step=True):
    """Element-wise comparison with the reference; returns the measured maxima (printed)."""
    nc = 12 * ref["C"]
    err = {}
    err["cost"] = abs(cost - ref["cost"]) / ref["cost"]
    err["g_cam"] = np.abs(g_cam - ref["g_cam"]).max() / np.abs(ref["g_cam"]).max()
    err["S"] = np.abs(S - ref["S"]).max() / np.abs(ref["S"]).max()
    err["b"] = np.abs(b - ref["b"]).max() / np.abs(ref["b"]).max()
    ok = {"cost": err["cost"] <= 1e-12, "g_cam": err["g_cam"] <= 1e-10, "S": err["S"] <= 1e-9, "b": err["b"] <= 1e-9}
    empty = ref["empty"]
    if grad is not None:
        gp, gp_ref = grad[nc:].reshape(-1, 6), ref["g_pose"]
        gmax = max(np.abs(gp_ref).max(), np.abs(ref["g_cam"]).max())
        scale = np.abs(gp_ref).max(1) + 1e-3 * gmax
        err["g_pose"] = (np.abs(gp - gp_ref).max(1) / scale).max()
        ok["g_pose"] = (np.abs(gp - gp_ref).max(1) <= 1e-9 * np.abs(gp_ref).max(1) + 1e-12 * gmax).all()
        ok["g_empty"] = (gp[empty] == 0.0).all()
        ok["g_head"] = np.array_equal(grad[:nc], g_cam)
    if x_new is not None:
        d = x_new - x0
        dc, dc_ref = d[:nc], ref["step"][:nc]
        dp, dp_ref = d[nc:].reshape(-1, 6), ref["step"][nc:].reshape(-1, 6)
        err["step_cam"] = np.abs(dc - dc_ref).max() / np.abs(dc_ref).max()
        tol_p = 1e-6 * np.abs(dp_ref).max(1) + 1e-9 * np.abs(dp_ref).max()
        err["step_pose"] = (np.abs(dp - dp_ref).max(1) / (np.abs(dp_ref).max(1) + 1e-3 * np.abs(dp_ref).max())).max()
        ok["step_cam"] = err["step_cam"] <= 1e-6
        ok["step_pose"] = (np.abs(dp - dp_ref).max(1) <= tol_p).all() or not pose_step
        ok["step_empty"] = np.array_equal(x_new[nc:].reshape(-1, 6)[empty], x0[nc:].reshape(-1, 6)[empty])
    print(f"\n[{tag}] " + "  ".join(f"{k} {v:.1e}" for k, v in err.items()) + f"  empty frames {int(empty.sum())}")
    failed = [k for k, v in ok.items() if not v]
    assert not failed, f"{tag}: {failed} out of tolerance ({err})"
    return err


# ------------------------------------------------------------------ 1. every scenario against the reference
@pytest.mark.parametrize("name", list(SCENARIOS))
def test_scenario_matches_the_blockwise_reference(name):
    uvs, obj, x0, loss, f_scale = build(name)
    prob = mcc.BAProblem(uvs, obj)
    plan = record_plan(name, prob)
    print(f"\n[{name}] plan " + json.dumps({k: v for k, v in plan.items() if k != "units"}) + f" units {plan['units']}")
    ev = evaluate_reference(uvs, obj, x0, LAM, loss, f_scale)
    _REFS[name] = dict(S=ev.S, b=ev.b, g_cam=ev.g_cam, g_pose=ev.g_pose, cost=ev.cost, step=ev.step(),
                       empty=ev.empty, C=ev.C)
    ref = _REFS[name]
    S, b, g_cam, cost = prob.build_reduced(x0, lam=LAM, loss=loss, f_scale=f_scale)
    grad = prob.gradient()
    x1 = prob.solve_step(LAM)
    compare_system(name, ref, S, b, g_cam, cost, grad, x1, x0, pose_step=name not in RANK_DEFICIENT_POSES)
    pred = prob.predict(x0)
    err_pred = np.abs(pred - ev.pred).max() / np.abs(ev.pred).max()
    print(f"[{name}] predict {err_pred:.1e}")
    assert err_pred <= 1e-10
    r_ref = (uvs - ev.pred)[~np.isnan(uvs)]
    r = prob.residuals(x0)
    assert r.shape == r_ref.shape and np.abs(r - r_ref).max() <= 1e-10 * np.abs(ev.pred).max()
    assert np.array_equal(S, S.T)


def test_undamped_system_matches_the_reference_at_full_rank():
    """lam = 0 (no pose damping): every non-empty pose block of these scenes has full rank."""
    for name in ("17x2000", "6x8000_n99"):
        uvs, obj, x0, loss, f_scale = build(name)
        ev = evaluate_reference(uvs, obj, x0, 0.0, loss, f_scale)
        S, b, g_cam, cost = mcc.BAProblem(uvs, obj).build_reduced(x0, lam=0.0, loss=loss, f_scale=f_scale)
        compare_system(name + " lam=0", dict(S=ev.S, b=ev.b, g_cam=ev.g_cam, cost=ev.cost, empty=ev.empty, C=ev.C),
                       S, b, g_cam, cost)


# ------------------------------------------------------------------ 2. the pipelined host-buffer call
@pytest.mark.parametrize("C", [6, 16])
def test_pipelined_host_call_matches_the_reference(C):
    """mcba_build_reduced_host with page-locked buffers splits the frames into eight child problems; their
    sums, and the parent rebuilt from them afterwards (gradient, damped step), against the reference."""
    import ctypes
    import torch
    from multicam_calibration_b200 import _native
    sc = make_scene(C, 20011, sigma=0.5, p_missing_view=0.2, seed=40 + C)
    uvs, obj, x0 = sc.uvs, sc.objpoints, sc.x0()
    ev = evaluate_reference(uvs, obj, x0, LAM, "soft_l1", 1.0)
    ref = dict(S=ev.S, b=ev.b, g_cam=ev.g_cam, g_pose=ev.g_pose, cost=ev.cost, step=ev.step(), empty=ev.empty, C=C)
    prob = mcc.BAProblem(uvs, obj)
    keep = [torch.from_numpy(np.ascontiguousarray(uvs)).pin_memory(),
            torch.from_numpy(np.ascontiguousarray(obj, dtype=np.float64)).pin_memory(),
            torch.from_numpy(x0.copy()).pin_memory(), torch.empty(144 * C * C, dtype=torch.float64).pin_memory(),
            torch.empty(12 * C, dtype=torch.float64).pin_memory(), torch.empty(1, dtype=torch.float64).pin_memory()]
    ptrs = [ctypes.c_void_p(t.data_ptr()) for t in keep]
    n0 = prob.kernel_launches
    _native.check(prob.lib.mcba_build_reduced_host(prob._h, ptrs[0], ptrs[1], ptrs[2], LAM, _native.LOSSES["soft_l1"], 1.0,
                                                   ptrs[3], ptrs[4], ptrs[5]))
    assert prob.kernel_launches - n0 <= 20            # the ranges ran on the child problems
    S = keep[3].numpy().reshape(12 * C, 12 * C).copy()
    b = keep[4].numpy().copy()
    cost = float(keep[5][0])
    prob._x_last = prob._x(x0)
    grad = prob.gradient()
    x1 = prob.solve_step(LAM)
    compare_system(f"host pipeline {C}x20011", ref, S, b, grad[:12 * C], cost, grad, x1, x0)


# ------------------------------------------------------------------ 3. forced kernel variants (one child process each)
_CHILD = r"""
import sys, json, numpy as np
sys.path.insert(0, {root!r})
sys.path.insert(0, {tests!r})
import multicam_calibration_b200 as mcc
import test_scale_parity as t
out = {{}}
for name in {names!r}:
    uvs, obj, x0, loss, f_scale = t.build(name)
    prob = mcc.BAProblem(uvs, obj)
    plan = prob.plan_info()
    S, b, g, cost = prob.build_reduced(x0, lam=t.LAM, loss=loss, f_scale=f_scale)
    grad = prob.gradient()
    x1 = prob.solve_step(t.LAM)
    np.savez({out_dir!r} + "/" + name + ".npz", S=S, b=b, g=g, cost=cost, grad=grad, x1=x1)
    out[name] = plan
print(json.dumps(out))
"""


def _run_child(env, names, tmp_path):
    code = _CHILD.format(root=ROOT, tests=os.path.join(ROOT, "tests"), names=list(names), out_dir=str(tmp_path))
    e = dict(os.environ)
    e.update(env)
    run = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, env=e)
    assert run.returncode == 0, run.stderr[-3000:]
    return json.loads(run.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("env,names,check", [
    ({"MCBA_SYRK_RUNTIME": "1"}, ("bench_6x50000", "16x8000", "8x4000", "17x2000"),
     lambda p: p["syrk_static_nb"] == 0),
], ids=["syrk_runtime"])
def test_forced_kernel_variants_match_the_reference(env, names, check, tmp_path):
    """MCBA_SYRK_RUNTIME (read once per process) selects the run-time SYRK tile lists, which the heuristics
    pick only for widths without a compiled list, for these shapes: against the same reference."""
    plans = _run_child(env, names, tmp_path)
    for name in names:
        assert check(plans[name]), (name, plans[name])
        ref = reference(name)
        _, _, x0, _, _ = build(name)
        d = np.load(tmp_path / (name + ".npz"))
        compare_system(f"{name} {env}", ref, d["S"], d["b"], d["g"], float(d["cost"]), d["grad"], d["x1"], x0)


# ------------------------------------------------------------------ 4. the end of a solve
def check_solve_end(tag, uvs, obj, x, grad, cost, optimality, g0_scale):
    """res.cost, res.grad (the gradient kernel of the closing evaluation) and res.optimality against the
    reference at res.x.  The gradient is near zero there, so its tolerance is scaled by the gradient at
    x0: a frame that the closing evaluation dropped or counted twice moves it by far more."""
    ev = evaluate_reference(uvs, obj, x, 0.0, "soft_l1", 1.0)
    g_ref = np.r_[ev.g_cam, ev.g_pose.ravel()]
    err_cost = abs(cost - ev.cost) / ev.cost
    err_g = np.abs(grad - g_ref).max() / g0_scale
    print(f"\n[solve {tag}] cost {err_cost:.1e}  grad {err_g:.1e} of max|g(x0)|  optimality {optimality:.3e} "
          f"reference {np.abs(g_ref).max():.3e}")
    assert err_cost <= 1e-12
    assert err_g <= 1e-10
    assert optimality == np.abs(grad).max()
    assert abs(optimality - np.abs(g_ref).max()) <= 1e-10 * g0_scale
    assert (grad[12 * ev.C:].reshape(-1, 6)[ev.empty] == 0.0).all()


@pytest.mark.parametrize("name", ["bench_6x50000", "16x8000"])
def test_solve_ends_at_the_reference_gradient(name):
    uvs, obj, x0, loss, f_scale = build(name)
    x, res = mcc.BAProblem(uvs, obj).solve(x0, ftol=1e-10, verbose=0)
    assert res.success
    ref = reference(name, uvs, obj, x0)
    check_solve_end(name, uvs, obj, x, res.grad, res.cost, res.optimality,
                    max(np.abs(ref["g_cam"]).max(), np.abs(ref["g_pose"]).max()))


# ------------------------------------------------------------------ 5. large boards
def test_large_board_goes_through_bundle_adjust():
    """A 9 x 11 board (99 corners): the observation transpose needs more than 48 KB of shared memory."""
    sc = make_scene(4, 300, board=(9, 11), sigma=0.3, p_missing_view=0.2, seed=50)
    np.random.seed(0)
    e, i, p, use, res = mcc.bundle_adjust(*sc.init_args(), n_frames=None, ftol=1e-10, verbose=0)
    assert res.success and len(use) > 200
    uv = sc.uvs[:, use]
    ev0 = evaluate_reference(uv, sc.objpoints, mcc.serialize_params(*sc.init_args()[1:3], sc.init_poses[use]), 0.0,
                             "soft_l1", 1.0)
    check_solve_end("bundle_adjust 99 corners", uv, sc.objpoints, res.x, res.grad, res.cost, res.optimality,
                    max(np.abs(ev0.g_cam).max(), np.abs(ev0.g_pose).max()))
    assert 0.28 < res.rms < 0.32


def test_board_beyond_the_shared_memory_limit_is_rejected():
    sc = make_scene(2, 3, board=(20, 25), sigma=0.3, seed=51)
    with pytest.raises(mcc._native.McbaError, match="shared memory"):
        mcc.BAProblem(sc.uvs, sc.objpoints)


# ------------------------------------------------------------------ 6. coverage of the launch heuristics
def _plan(name):
    if name not in _PLANS:
        uvs, obj, _, _, _ = build(name)
        record_plan(name, mcc.BAProblem(uvs, obj))
    return _PLANS[name]


COVERAGE = [
    ("K2p 8 warps, 6 full rounds + split tail", lambda p: p["k2p_warps"] == 8 and p["rounds"] == 6 and p["split_tail"]),
    ("K2p split tail after 1 round", lambda p: p["rounds"] == 1 and p["split_tail"]),
    ("K2p split tail, even corner count", lambda p: p["split_tail"] and p["N"] % 2 == 0 and p["N"] != 35),
    ("K2p split tail, odd corner count > 35", lambda p: p["split_tail"] and p["N"] % 2 == 1 and p["N"] > 35),
    ("K2p 8 warps, no full round", lambda p: p["k2p_warps"] == 8 and p["rounds"] == 0),
    ("K2p 8 warps, leftover too large to split", lambda p: p["k2p_warps"] == 8 and p["rounds"] >= 1 and p["left"] > 0
     and not p["split_tail"]),
    ("K2p 4 warps", lambda p: p["k2p_warps"] == 4),
    ("K2c ring, 6 cameras, >= 5 tiles per CTA", lambda p: p["k2c_mode"] == "ring" and p["cameras"] == 6
     and p["tiles"] >= 5 * p["k2c_parts"]),
    ("K2c ring, 2 cameras", lambda p: p["k2c_mode"] == "ring" and p["cameras"] == 2),
    ("K2c ring, 3 cameras", lambda p: p["k2c_mode"] == "ring" and p["cameras"] == 3),
    ("K2c streamed, 1 camera", lambda p: p["k2c_mode"] == "stream" and p["cameras"] == 1),
    ("K2c streamed, 12 warps", lambda p: p["k2c_mode"] == "stream" and p["k2c_warps"] == 12),
    ("K2c streamed, fewer than 12 warps", lambda p: p["k2c_mode"] == "stream" and 0 < p["k2c_warps"] < 12),
    ("SYRK 8 warps, static NB 9", lambda p: p["syrk_warps"] == 8 and p["syrk_static_nb"] == 9),
    ("SYRK 8 warps, static NB 12", lambda p: p["syrk_warps"] == 8 and p["syrk_static_nb"] == 12),
    ("SYRK 15 warps, run-time list", lambda p: p["syrk_warps"] == 15 and p["syrk_gy"] == 1 and p["syrk_static_nb"] == 0),
    ("SYRK 15 warps, static NB 24", lambda p: p["syrk_warps"] == 15 and p["syrk_static_nb"] == 24),
    ("SYRK gy = 2", lambda p: p["syrk_gy"] == 2),
    ("SYRK gy = 3", lambda p: p["syrk_gy"] == 3),
    ("SYRK gy = 4", lambda p: p["syrk_gy"] == 4),
    ("solve regs3", lambda p: p["solve"] == "regs3"),
    ("solve regs8", lambda p: p["solve"] == "regs8"),
    ("solve smem19", lambda p: p["solve"] == "smem19"),
    ("solve cuSOLVER", lambda p: p["solve"] == "cusolver"),
    ("empty camera inside the group prefix", lambda p: any(u == 0 for u in p["units"][1:-1])),
    ("empty camera at the end of the group prefix", lambda p: p["cameras"] > 1 and p["units"][-1] == 0),
    ("every unit live", lambda p: p["cameras"] == 6 and sum(p["units"]) == 6 * p["tiles"] and p["tiles"] > 1000),
    ("most units dead", lambda p: p["cameras"] == 6 and 0 < sum(p["units"]) < 0.75 * 6 * p["tiles"]),
]


def test_scenarios_reach_every_kernel_branch():
    plans = {name: _plan(name) for name in SCENARIOS}
    missing = [what for what, pred in COVERAGE if not any(pred(p) for p in plans.values())]
    for what, pred in COVERAGE:
        print(f"{what}: {[n for n, p in plans.items() if pred(p)]}")
    assert not missing, f"no scenario reaches: {missing}"
