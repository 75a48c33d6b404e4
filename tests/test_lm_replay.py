"""The Levenberg-Marquardt loop of ``mcba_lm_run``, decision by decision, at production sizes.

End points (final cost, gradient, RMS) cannot show a wrong loop: a wrong step is rejected and retried, a wrong
scaling or damping rule only changes how many evaluations a solve takes.  So the device solve is replayed: the loop's
path does not depend on ``max_nfev`` until the budget test and the solve is deterministic, so a run with ``max_nfev =
k`` returns the state after exactly k evaluations.  ``lm_reference.check_replay`` checks every transition k -> k+1
from the state the engine was in (step, reported cost / reduction / step norm / gradient, accept, ftol, xtol, the
IRLS -> Triggs switch through the next step, lambda, lambda_max, gtol, budget) against the blockwise fp64 reference;
it never follows a path of its own, so a near-tie in rounding cannot send it elsewhere.

CPU tests pin the reference to ``oracle.lm_solve`` and show that the checker rejects loops with one rule changed.
The GPU scenarios print the accepted (A) / rejected (r) pattern, the largest error per quantity and the ties
(``pytest -s``); the last GPU test asserts that some scenario reaches every path of the loop."""
import ctypes

import numpy as np
import pytest

import lm_reference as lmr
from oracle import np_oracle as orc
from multicam_calibration_b200.synthetic import make_scene


def small_scene(C=3, F=12, seed=5, sigma=0.4):
    sc = make_scene(C, F, sigma=sigma, p_missing_view=0.2, seed=seed)
    return sc.uvs, sc.objpoints, sc.x0()


# ------------------------------------------------------------------ CPU: the reference against oracle.lm_solve
def lm_solve_run(x0, uvs, obj, o):
    """``oracle.lm_solve`` in the form :func:`lm_reference.replay` takes."""
    def run(max_nfev):
        trace = []
        kw = {k: o[k] for k in ("ftol", "xtol", "gtol", "loss", "f_scale", "hessian", "lambda0", "lambda_min",
                                "lambda_max")}
        x, info = orc.lm_solve(x0, uvs, obj, max_nfev=o["max_nfev"] if max_nfev is None else max_nfev,
                               trace=trace, **kw)
        g0 = orc.normal_equations(x0, uvs, obj, o["loss"], o["f_scale"])[1]
        records = [(0, 1, orc.robust_cost(x0, uvs, obj, o["loss"], o["f_scale"]), np.nan, np.nan, np.abs(g0).max())]
        records += [(it, nfev, cost, actual, sn, gnorm) for it, nfev, cost, actual, sn, gnorm, _, _ in trace]
        state = dict(x=x, lam=info["lam"], nfev=info["nfev"], njev=info["njev"], iterations=info["iterations"],
                     status=info["status"], cost=info["cost"], optimality=info["optimality"],
                     step_norm=trace[-1][4] if trace else 0.0, rms=orc.reprojection_rms(x, uvs, obj))
        return state, records
    return run


PIN_CASES = {
    "auto": dict(hessian="auto"),
    "irls": dict(hessian="irls"),
    "triggs": dict(hessian="triggs"),
    "linear": dict(loss="linear"),
    "gtol_after_steps": dict(ftol=0.0, xtol=0.0, gtol=2e-2),
    "lambda_max": dict(ftol=0.0, xtol=0.0, gtol=0.0, lambda0=1e4, lambda_max=1e6),
}


@pytest.mark.parametrize("case", sorted(PIN_CASES))
def test_reference_follows_lm_solve(case):
    """Driven along ``oracle.lm_solve``'s own trajectory, the reference reproduces every step, decision and lambda."""
    uvs, obj, x0 = small_scene()
    o = lmr.options(**dict(dict(ftol=1e-10, xtol=1e-10, max_nfev=60), **PIN_CASES[case]))
    full, records, states = lmr.replay(lm_solve_run(x0, uvs, obj, o))
    rep = lmr.check_replay(states, records, full, x0, uvs, obj, o, log=print)
    assert rep["transitions"] >= 3


def test_reference_with_a_fixed_mask():
    """Intrinsics and camera 0 held: the blockwise loop on the free sub-problem passes its own checker, holds the
    mask exactly and ends at the masked minimum's cost that ``lm_solve`` cannot reach with the mask removed."""
    uvs, obj, x0 = small_scene()
    fixed = np.zeros((3, 12), dtype=bool)
    fixed[:, :6] = True
    fixed[0] = True
    o = lmr.options(ftol=1e-10, xtol=1e-10, max_nfev=40, fixed=fixed)
    full, records, states = lmr.replay(lambda k: lmr.simulate(x0, uvs, obj, o, 40 if k is None else k))
    lmr.check_replay(states, records, full, x0, uvs, obj, o, log=print)
    assert np.array_equal(full["x"][:36][fixed.ravel()], x0[:36][fixed.ravel()])
    _, info = orc.lm_solve(x0, uvs, obj, ftol=1e-10, xtol=1e-10, max_nfev=40)
    assert info["cost"] < full["cost"]


# The IRLS ratios of the default solve exceed 1, where both damping rules give the factor 0.1, and its lambda falls
# by 10 per step, where the scaling hardly matters: the damping and scaling rules are shown on a Triggs solve that
# starts with five rejections and takes steps of every quality.
TRIGGS_CASE = dict(ftol=0.0, xtol=0.0, gtol=2e-2, max_nfev=60, hessian="triggs")
WRONG_CASES = dict(default=dict(ftol=0.0, xtol=0.0, gtol=2e-2, max_nfev=60),
                   damping_1_minus_t2=TRIGGS_CASE, d2_without_running_max=TRIGGS_CASE)


def _wrong_case(wrong):
    return lmr.options(**WRONG_CASES.get(wrong, WRONG_CASES["default"]))


@pytest.mark.parametrize("rules", ["default", "damping_1_minus_t2"])   # the IRLS and the Triggs case
def test_checker_accepts_the_right_loop(rules):
    uvs, obj, x0 = small_scene()
    o = _wrong_case(rules)
    full, records, states = lmr.replay(lambda k: lmr.simulate(x0, uvs, obj, o, 60 if k is None else k))
    rep = lmr.check_replay(states, records, full, x0, uvs, obj, o, log=print)
    assert rep["status"] == 1 and full["status"] == 1


@pytest.mark.parametrize("wrong", lmr.WRONG_RULES)
def test_checker_rejects_a_wrong_loop(wrong):
    """A loop with one rule changed (D^2 without the running maximum, a 10 % switch, ``1 - t^2`` in the damping
    update, the budget before gtol) still converges, but the replay names the transition where it went wrong."""
    uvs, obj, x0 = small_scene()
    o = _wrong_case(wrong)
    full, records, states = lmr.replay(lambda k: lmr.simulate(x0, uvs, obj, o, 60 if k is None else k, wrong))
    with pytest.raises(lmr.ReplayError) as e:
        lmr.check_replay(states, records, full, x0, uvs, obj, o)
    print(f"{wrong}: {e.value}")


# ------------------------------------------------------------------ GPU: the engine's trajectory
def engine_run(prob, x0, o):
    """``mcba_lm_run`` through ctypes as ``BAProblem.solve`` calls it (same options, the problem's stream), with an
    iteration callback that keeps every record at full precision."""
    from multicam_calibration_b200 import _native
    from multicam_calibration_b200.engine import _ptr, parse_options

    kw = {k: o[k] for k in ("ftol", "xtol", "gtol", "loss", "f_scale", "hessian", "lambda0", "lambda_min", "lambda_max")}
    torch = prob.torch

    def run(max_nfev):
        opts = parse_options(dict(kw, verbose=0, max_nfev=o["max_nfev"] if max_nfev is None else max_nfev),
                             prob.n_params)
        records = []
        cb = _native.ITER_CALLBACK(lambda user, it, nfev, cost, red, step, g: records.append((it, nfev, cost, red, step, g)))
        opts.iter_callback = cb
        with torch.cuda.device(prob.device), torch.cuda.stream(prob.stream):
            prob.set_fixed(o["fixed"])
            x = prob._x(x0)
            res = _native.Result()
            _native.check(prob.lib.mcba_lm_run(prob._h, _ptr(x), ctypes.byref(opts), ctypes.byref(res), None))
            xs = _native.to_host(x)
        state = dict(x=xs, lam=res.lambda_, nfev=res.nfev, njev=res.njev, iterations=res.iterations,
                     status=res.status, cost=res.cost, optimality=res.optimality, step_norm=res.step_norm, rms=res.rms)
        return state, records
    return run


def _scene(C, F, seed=0, p=0.2, sigma=0.5):
    sc = make_scene(C, F, sigma=sigma, p_missing_view=p, seed=seed)
    return np.ascontiguousarray(sc.uvs), sc.objpoints, sc.x0()


def _outliers():
    from test_scale_parity import _outlier_scene
    uvs, obj, x0 = _outlier_scene()
    return np.ascontiguousarray(uvs), obj, x0


_CONVERGED = {}


def _converged(C=6, F=2000, seed=40, jitter=0.0):
    """6 x 2000 solved to its minimum on the device (ftol = xtol = 1e-15), optionally moved off it by ``jitter``."""
    import multicam_calibration_b200 as mcc
    if (C, F, seed) not in _CONVERGED:
        uvs, obj, x0 = _scene(C, F, seed)
        prob = mcc.BAProblem(uvs, obj)
        x, _ = prob.solve(x0, ftol=1e-15, xtol=1e-15, gtol=1e-12, max_nfev=200, verbose=0)
        prob.close()
        _CONVERGED[(C, F, seed)] = (uvs, obj, x)
    uvs, obj, x = _CONVERGED[(C, F, seed)]
    rng = np.random.default_rng(1)
    return uvs, obj, x + jitter * rng.normal(size=x.size) * np.maximum(np.abs(x), 1.0), _scene(C, F, seed)[2]


def _held_intrinsics_and_camera0(C):
    fixed = np.zeros((C, 12), dtype=bool)
    fixed[:, :6] = True
    fixed[0] = True
    return fixed


# name -> (builder, options); bundle_adjust's defaults unless given
REPLAYS = {
    "bench_6x50000": (lambda: _scene(6, 50000), {}),
    "16x8000_irls": (lambda: _scene(16, 8000, seed=16), dict(hessian="irls")),
    "32x2000_triggs": (lambda: _scene(32, 2000, seed=19), dict(hessian="triggs")),
    # the same solve starts with six rejections: lambda_max ends it after five, a large xtol on the first
    "32x2000_triggs_lambda_max": (lambda: _scene(32, 2000, seed=19), dict(hessian="triggs", lambda_max=100.0)),
    "32x2000_triggs_xtol_rejected": (lambda: _scene(32, 2000, seed=19), dict(hessian="triggs", xtol=1e3)),
    "6x3000_outliers_fs0.25": (_outliers, dict(f_scale=0.25)),
    "6x2000_linear": (lambda: _scene(6, 2000, seed=41), dict(loss="linear", ftol=1e-10)),
    "6x2000_held": (lambda: _scene(6, 2000, seed=42), dict(fixed=_held_intrinsics_and_camera0(6), ftol=1e-8)),
    "6x2000_gtol_after_steps": (lambda: _scene(6, 2000, seed=43), dict(ftol=0.0, xtol=0.0, gtol=1e-2)),
    "6x2000_clamp_lambda_max": (lambda: _scene(6, 2000, seed=44), dict(ftol=0.0, xtol=0.0, gtol=0.0, lambda_min=3e-4,
                                                                      lambda_max=1e3, max_nfev=80)),
    "6x2000_restart_gtol": (lambda: _converged(), dict(gtol=1e10)),
    "6x2000_restart_zero_tol": (lambda: _converged(), dict(ftol=0.0, xtol=0.0, gtol=0.0, max_nfev=25)),
    "6x2000_near_minimum_ftol_xtol": (lambda: _converged(jitter=1e-7), dict(ftol=1e-4, xtol=1e-4)),
    "6x2000_near_minimum_xtol": (lambda: _converged(jitter=1e-7), dict(ftol=0.0, xtol=1e-4)),
}
_REPORTS = {}


def _replay(name):
    if name not in _REPORTS:
        import time
        import multicam_calibration_b200 as mcc
        build, kw = REPLAYS[name]
        uvs, obj, x0, *start = build()
        o = lmr.options(**kw)
        # a restart from a minimum: gradients are compared on the scale of the problem's unsolved start
        g_scale = lmr.Point(start[0], uvs, obj, o, "triggs").gnorm if start else None
        if o["max_nfev"] is None:
            o["max_nfev"] = 200
        t0 = time.time()
        prob = mcc.BAProblem(uvs, obj)
        full, records, states = lmr.replay(engine_run(prob, x0, o))
        prob.close()
        t1 = time.time()
        print(f"\n{name}: {uvs.shape[0]} x {uvs.shape[1]}, replay {t1 - t0:.1f} s")
        _REPORTS[name] = lmr.check_replay(states, records, full, x0, uvs, obj, o, log=print, g_scale=g_scale)
        print(f"  reference {time.time() - t1:.1f} s")
    return _REPORTS[name]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(REPLAYS))
def test_engine_loop_replays_against_the_reference(name):
    _replay(name)


@pytest.mark.gpu
def test_gtol_on_the_last_evaluation_of_the_budget():
    """A solve that ends on gtol after a step, cut at its own nfev: gtol at the last accepted point still wins over
    the exhausted budget (status 1, success), as in scipy."""
    import multicam_calibration_b200 as mcc
    uvs, obj, x0 = _scene(6, 2000, seed=43)
    prob = mcc.BAProblem(uvs, obj)
    x, res = prob.solve(x0, ftol=0.0, xtol=0.0, gtol=1e-2, verbose=0)
    assert res.status == 1 and res.iterations > 0
    xc, cut = prob.solve(x0, ftol=0.0, xtol=0.0, gtol=1e-2, max_nfev=res.nfev, verbose=0)
    assert cut.status == 1 and cut.success and cut.nfev == res.nfev
    assert np.array_equal(xc, x) and cut.cost == res.cost


# loop path -> predicate on a replay report
COVERAGE = [
    ("rejection", lambda r: "r" in r["pattern"]),
    ("two or more rejections in a row (nu doubles)", lambda r: "rr" in r["pattern"]),
    ("lambda_min clamp", lambda r: "lambda_min clamp" in r["events"]),
    ("IRLS -> Triggs switch, guessed", lambda r: "switch, guessed" in r["events"]),
    ("IRLS -> Triggs switch, re-walk", lambda r: "switch, re-walk" in r["events"] or "no switch, re-walk" in r["events"]),
    ("status 1 at x0", lambda r: r["status"] == 1 and r["transitions"] == 0),
    ("status 1 after a step (and gtol on the last evaluation of the budget)",
     lambda r: r["status"] == 1 and r["transitions"] > 0),
    ("status 2", lambda r: r["status"] == 2),
    ("status 3, accepted step", lambda r: r["status"] == 3 and r["pattern"].endswith("A")),
    ("status 3, rejected step", lambda r: r["status"] == 3 and r["pattern"].endswith("r")),
    ("status 4", lambda r: r["status"] == 4),
    ("status 0 with an evaluation pending", lambda r: r["status"] == 0 and r["pattern"].endswith("A")),
    ("status -1 (lambda_max)", lambda r: r["status"] == -1),
]


@pytest.mark.gpu
def test_scenarios_reach_every_loop_path():
    reports = {name: _replay(name) for name in REPLAYS}
    for what, pred in COVERAGE:
        print(f"{what}: {[n for n, r in reports.items() if pred(r)]}")
    missing = [what for what, pred in COVERAGE if not any(pred(r) for r in reports.values())]
    assert not missing, f"no scenario reaches: {missing}"
