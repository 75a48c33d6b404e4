"""Reference for the Levenberg-Marquardt loop of ``mcba_lm_run``, one transition at a time, and the checker that
replays a solve's trajectory against it (tests/test_lm_replay.py).

A trajectory is what a solver reports after exactly k evaluations, k = 1 .. K (``max_nfev = k``; the loop's path
does not depend on the budget until the budget test): ``x_k``, ``lambda_k``, the counters and the status, plus the
per-iteration records ``(it, nfev, cost, actual reduction, step norm, gnorm)`` of the full run.  The checker never
follows a path of its own: at every transition k -> k+1 it rebuilds the reference at the solver's ``x_k`` and
``lambda_k`` and checks the step, the reported values and every decision against it.

The reference state at an accepted point is a :class:`Point`: the blockwise fp64 evaluation
(``oracle.blockwise.BlockwiseEvaluation``) in the weight mode the loop has there, with the running Marquardt
scaling of the accepted points seen so far (``D2cam``, ``D2pose``: the maximum of ``diag U`` resp. ``diag V_f``).
A rejected step changes only lambda, so the point eliminates the poses again (``redamp``) without walking the
Jacobian again.

Rules (csrc/mcba_api.cu, oracle.np_oracle.lm_solve): ``pred = -0.5 g.d + 0.5 lam d^T D^2 d``, ``ratio = actual /
pred``; a step is accepted iff ``actual > 0``; ftol ``actual < ftol cost and ratio > 0.25``, xtol ``|d| < xtol (xtol +
|x|)`` (status 4 both, 2 ftol, 3 xtol; a rejected step that meets xtol ends with 3); on acceptance ``lam =
max(lambda_min, lam max(0.1, 1 - (2 ratio - 1)^3))``, nu = 2, and IRLS weights switch to Triggs for good when
``actual < 1e-2 cost`` (``hessian='auto'``); on rejection ``lam *= nu, nu *= 2`` and ``lam > lambda_max`` ends with -1.
Precedence: a step that meets ftol / xtol reports that status even where the new point also meets gtol (the
engine's convention, which scipy's trf orders the other way round); otherwise gtol at the new point (status 1) wins
over the evaluation budget (status 0), as in scipy.

Decisions whose deciding quantity is within a rounding margin of its threshold are ties: they are counted and
printed, and the checker follows the solver's choice there."""
import numpy as np

from oracle import blockwise
from oracle import np_oracle as orc

SWITCH = 1e-2          # IRLS -> Triggs once a step reduces the cost by less than 1 %
COST_ULP = 4e-12       # rounding margin of a cost difference, relative to the cost
STEP_RTOL = 1e-6       # step norms (tests/test_scale_parity.compare_system's step tolerance)
# Componentwise backward error of the solver's step in the reference system, beyond the rounding of its inputs
# (Point.backward_error).  What is left is the difference of the two systems -- the engine's agrees with the reference's
# to 1e-9 of the largest entry (tests/test_scale_parity.py) -- and the backward error of the solve itself, fp64
# Cholesky.  1e-6 is compare_system's step tolerance: the measured maxima are 1.9e-11 on the device (outlier scene) and
# 1.5e-13 in the CPU pins, while solving in the wrong weight mode gives 1.7e-3 (the 10 % switch).
BACKWARD_TOL = 1e-6
G_ROUND_ULPS = 4       # gradient rounding in ulps of |J|^T |rho'| (|uv| + |pred|): f = uv - pred rounds by half an ulp
                       # in the engine and in the reference, pred carries a few ulps of the projection chain
EPS = np.finfo(float).eps
PRED_RTOL = 1e-8       # the solver's pred comes from its own g and D^2 and step


def options(ftol=1e-4, xtol=1e-8, gtol=1e-8, loss="soft_l1", f_scale=1.0, hessian="auto", lambda0=1e-3,
            lambda_min=1e-12, lambda_max=1e12, max_nfev=None, fixed=None):
    """The loop's options with ``least_squares``' names and the engine's defaults."""
    return dict(ftol=ftol, xtol=xtol, gtol=gtol, loss=loss, f_scale=f_scale, hessian=hessian, lambda0=lambda0,
                lambda_min=lambda_min, lambda_max=lambda_max, max_nfev=max_nfev, fixed=fixed)


def robust_cost(x, uvs, obj, loss="soft_l1", f_scale=1.0, chunk=4096):
    """``(0.5 sum rho, sum f^2, count)`` at ``x``, frame chunk by frame chunk."""
    C, F = uvs.shape[:2]
    ext, intr, poses = orc.deserialize_params(x, C)
    cost = sumsq = n = 0.0
    for s in range(0, F, chunk):
        f = uvs[:, s:s + chunk] - orc.predict_calib_uvs(ext, intr, obj, poses[s:s + chunk])
        f = f[~np.isnan(f)]
        cost += 0.5 * orc.loss_rho(f, loss, f_scale)[0].sum()
        sumsq += f @ f
        n += f.size
    return cost, sumsq, n


class Point:
    """The reference at an accepted point ``x``: evaluation in weight mode ``mode`` with the running scaling."""

    def __init__(self, x, uvs, obj, o, mode, D2cam=None, D2pose=None, lam=0.0):
        self.x, self.mode = np.asarray(x, dtype=float), mode
        self.ev = blockwise.BlockwiseEvaluation(self.x, uvs, obj, lam=lam, loss=o["loss"], f_scale=o["f_scale"],
                                                hessian=mode, D2pose=D2pose)
        ev = self.ev
        self.D2cam = ev.diag_U.copy() if D2cam is None else np.maximum(D2cam, ev.diag_U)
        self.D2pose = ev.D2pose
        nc = 12 * ev.C
        self.held = np.zeros(nc, dtype=bool) if o["fixed"] is None else np.asarray(o["fixed"], dtype=bool).ravel()
        self.g = np.concatenate([ev.g_cam, ev.g_pose.ravel()])
        self.gnorm = np.abs(np.concatenate([ev.g_cam[~self.held], ev.g_pose.ravel()])).max()
        self.cost = ev.cost
        self.D2 = np.concatenate([self.D2cam, self.D2pose.ravel()])
        self.D2[self.D2 == 0.0] = 1.0

    def step(self, lam):
        """The damped step ``[delta_cam | delta_pose]`` at damping ``lam`` (held entries exactly 0)."""
        ev = self.ev
        if ev.lam != lam:
            ev.redamp(lam)
        free = ~self.held
        dcam = np.zeros(ev.b.size)
        A = ev.S + lam * np.diag(np.where(self.D2cam == 0.0, 1.0, self.D2cam))
        if free.any():
            dcam[free] = -np.linalg.solve(A[np.ix_(free, free)], ev.b[free])
        rhs = ev.g_pose + np.einsum("fai,a->fi", ev.W, dcam)
        dpose = -np.linalg.solve(ev.Vd, rhs[:, :, None])[:, :, 0]
        dpose[ev.empty] = 0.0
        return np.concatenate([dcam, dpose.ravel()])

    def backward_error(self, d, lam, dd=0.0, dg=0.0):
        """Componentwise backward error of a solver's step ``d`` in the damped system ``(H + lam D^2) d = -g`` at this
        point, beyond what the errors of its inputs explain: ``max_i (|r_i| - s_i)^+ / (|H + lam D^2| |d| + |g|)_i`` over
        the free rows, ``r = (H + lam D^2) d + g``, ``s = |H + lam D^2| dd + dg``.

        ``dd`` (per entry) is how well ``d`` is known: a step read back as ``x_{k+1} - x_k`` carries the rounding of
        ``x_k + d``, up to half an ulp of ``x_{k+1}`` -- once lambda is large or the point is a minimum, that is all
        of a 1e-13 step.  ``dg`` (per row) bounds the rounding of the gradient, which near a minimum is all of g.
        The bound is the plain fp64 backward error of a stable solve plus the errors of these two inputs.

        This, not ``d - step(lam)``, is what pins a step down: the cost is invariant under the 6-dimensional rigid
        gauge (the board's object points fix the scale), so once lambda has fallen to 1e-8 .. 1e-12 the step along
        those directions is set by the rounding of g, in the engine and here alike."""
        ev, nc = self.ev, 12 * self.ev.C
        dc, dp = d[:nc], d[nc:].reshape(-1, 6)
        adc, adp = np.abs(dc), np.abs(dp)
        ddv = np.broadcast_to(np.asarray(dd, dtype=float), d.shape)
        ddc, ddp = ddv[:nc], ddv[nc:].reshape(-1, 6)
        Dc, Dp = lam * self.D2[:nc], lam * self.D2[nc:].reshape(-1, 6)
        def abs_cam(vc, vp):     # |U| vc + |W| vp + lam D^2 vc, camera rows
            return (np.einsum("cij,cj->ci", np.abs(ev.U), vc.reshape(-1, 12)).ravel()
                    + np.einsum("fai,fi->a", np.abs(ev.W), vp) + Dc * vc)

        def abs_pose(vc, vp):    # |W|^T vc + |V| vp + lam D^2 vp, pose rows
            return np.einsum("fai,a->fi", np.abs(ev.W), vc) + np.einsum("fij,fj->fi", np.abs(ev.V), vp) + Dp * vp

        r_c = (np.einsum("cij,cj->ci", ev.U, dc.reshape(-1, 12)).ravel() + np.einsum("fai,fi->a", ev.W, dp) + Dc * dc
               + ev.g_cam)
        a_c = abs_cam(adc, adp) + np.abs(ev.g_cam)
        a_s_c = abs_cam(ddc, ddp)
        r_p = np.einsum("fai,a->fi", ev.W, dc) + np.einsum("fij,fj->fi", ev.V, dp) + Dp * dp + ev.g_pose
        a_p = abs_pose(adc, adp) + np.abs(ev.g_pose)
        a_s_p = abs_pose(ddc, ddp)
        # what the two inputs' errors alone can put into r, allowed in full; the solve's own error is relative
        slack = np.concatenate([a_s_c, a_s_p.ravel()]) + dg
        a = np.concatenate([a_c, a_p.ravel()])
        keep = np.concatenate([~self.held, np.ones(a_p.size, dtype=bool)])
        r, a, slack = np.concatenate([r_c, r_p.ravel()])[keep], a[keep], slack[keep]
        excess = np.maximum(np.abs(r) - slack, 0.0)
        live = a > 0
        return float((excess[live] / a[live]).max()) if live.any() else 0.0

    def pred(self, d, lam):
        return -0.5 * self.g @ d + 0.5 * lam * d @ (self.D2 * d)


def damping_update(lam, ratio, lambda_min, cube=True):
    t = 2.0 * ratio - 1.0
    return max(lambda_min, lam * max(0.1, 1.0 - (t ** 3 if cube else t * t)))


# ------------------------------------------------------------------ a blockwise solver with switchable rules
WRONG_RULES = ("d2_without_running_max", "switch_at_10pc", "damping_1_minus_t2", "budget_before_gtol")


def simulate(x0, uvs, obj, o, max_nfev, wrong=None):
    """The loop's rules run on :class:`Point` (the checker's own arithmetic), with one rule of ``WRONG_RULES``
    changed if ``wrong`` is given.  Returns ``(state, records)`` in the form :func:`check_replay` takes."""
    assert wrong in (None,) + WRONG_RULES
    irls = o["hessian"] != "triggs" and o["loss"] != "linear"
    mode = lambda: "irls" if irls else "triggs"
    keep_max = wrong != "d2_without_running_max"
    switch = 0.1 if wrong == "switch_at_10pc" else SWITCH
    P = Point(x0, uvs, obj, o, mode())
    lam, nu, nfev, njev, it, status, sn_last = o["lambda0"], 2.0, 1, 1, 0, None, 0.0
    records = [(0, 1, P.cost, np.nan, np.nan, P.gnorm)]
    if P.gnorm < o["gtol"]:
        status = 1
    while status is None:
        if nfev >= max_nfev:
            status = 0
            break
        d = P.step(lam)
        nfev += 1
        cost_new = robust_cost(P.x + d, uvs, obj, o["loss"], o["f_scale"])[0]
        pred, actual = P.pred(d, lam), P.cost - cost_new
        ratio = actual / pred if pred > 0 else -1.0
        sn, xn = np.linalg.norm(d), np.linalg.norm(P.x)
        f_ok = actual < o["ftol"] * P.cost and ratio > 0.25
        x_ok = sn < o["xtol"] * (o["xtol"] + xn)
        term = 4 if (f_ok and x_ok) else 2 if f_ok else 3 if x_ok else None
        if actual > 0:
            lam = damping_update(lam, ratio, o["lambda_min"], cube=wrong != "damping_1_minus_t2")
            nu, it, njev, sn_last = 2.0, it + 1, njev + 1, sn
            if irls and o["hessian"] == "auto" and actual < switch * P.cost:
                irls = False
            P = Point(P.x + d, uvs, obj, o, mode(), P.D2cam if keep_max else None, P.D2pose if keep_max else None)
            records.append((it, nfev, P.cost, actual, sn, P.gnorm))
            if term is not None:
                status = term
            elif wrong == "budget_before_gtol" and nfev >= max_nfev:
                status = 0
            elif P.gnorm < o["gtol"]:
                status = 1
        else:
            if term in (3, 4):
                status = 3
                break
            lam, nu = lam * nu, nu * 2.0
            if lam > o["lambda_max"]:
                status = -1
    cost, sumsq, n = robust_cost(P.x, uvs, obj, o["loss"], o["f_scale"])
    state = dict(x=P.x, lam=lam, nfev=nfev, njev=njev, iterations=it, status=status, cost=P.cost,
                 optimality=P.gnorm, step_norm=sn_last, rms=np.sqrt(sumsq / n))
    return state, records


def replay(run, K=None):
    """``run(max_nfev) -> (state, records)``: the full run, then the states after k = 1 .. K evaluations.  The
    records of every cut run must be a prefix of the full run's (the solve is deterministic)."""
    full, records = run(None)
    K = full["nfev"] if K is None else K
    states = []
    for k in range(1, K + 1):
        s, rec = run(k)
        assert s["nfev"] == k, f"the run cut at max_nfev={k} made {s['nfev']} evaluations"
        assert np.array_equal(np.array(rec, dtype=float), np.array(records[:len(rec)], dtype=float), equal_nan=True), \
            f"max_nfev={k}: another path"
        states.append(s)
    return full, records, states


# ------------------------------------------------------------------ the checker
class ReplayError(AssertionError):
    pass


def check_replay(states, records, full, x0, uvs, obj, o, log=None, g_scale=None):
    """Check every transition of a replayed trajectory against the reference.  Gradients are compared within
    ``1e-10 g_scale``, by default ``max |g(x0)|``; a solve restarted from a minimum passes the gradient scale of the
    problem (``max |g|`` at its unsolved start), since the gradient's rounding does not shrink with the gradient.  Returns a report dict (pattern,
    largest error per checked quantity, ties); raises :class:`ReplayError` naming the transition and the quantity."""
    uvs = np.asarray(uvs, dtype=float)
    nc = 12 * uvs.shape[0]
    errs, ties = {}, []

    def err(name, v):
        errs[name] = max(errs.get(name, 0.0), float(v))

    def fail(k, what):
        raise ReplayError(f"transition {k} -> {k + 1} (evaluations): {what}")

    def decide(k, name, conds, solver):
        """The AND of the conditions ``value < threshold`` (``conds``: ``(value, threshold, margin)``) as the reference
        sees it; where a condition within its margin of the threshold could give the solver's choice, that choice."""
        ref = all(v < th for v, th, _ in conds)
        if ref == solver:
            return ref
        fixed = [v < th for v, th, m in conds if not abs(v - th) <= m]
        tied = [(float(v), float(th)) for v, th, m in conds if abs(v - th) <= m]
        if tied and (all(fixed) if solver else True):
            ties.append((k, name, tied))
            return solver
        fail(k, f"{name}: the reference says {ref} ({', '.join(f'{v:.17g} < {th:.17g}' for v, th, _ in conds)}), "
                f"the solver {solver}")

    by_nfev = {r[1]: r for r in records if r[0] >= 1}
    irls = o["hessian"] != "triggs" and o["loss"] != "linear"
    P = Point(x0, uvs, obj, o, "irls" if irls else "triggs", lam=o["lambda0"])
    g0 = max(P.gnorm if g_scale is None else g_scale, np.finfo(float).tiny)
    gtol_margin = 1e-10 * g0
    nu, n_acc, pattern, last_sn, last_rel, events = 2.0, 0, [], 0.0, 1.0, set()
    expect_status = None

    def check_point_values(k, s):
        err("cost", abs(s["cost"] - P.cost) / P.cost)
        if abs(s["cost"] - P.cost) > 1e-12 * P.cost:
            fail(k, f"cost at the accepted point {s['cost']!r} vs reference {P.cost!r}")

    check_point_values(0, states[0])
    if states[0]["lam"] != o["lambda0"]:
        fail(0, "lambda at x0")
    if decide(0, "gtol at x0", [(P.gnorm, o["gtol"], gtol_margin)], states[0]["status"] == 1):
        expect_status = 1
        if len(states) > 1:
            fail(0, "gtol holds at x0 but the solver went on")
    for k in range(len(states) - 1):
        s, t = states[k], states[k + 1]
        lam, last = s["lam"], k + 2 == len(states)
        xn = np.linalg.norm(P.x)
        accepted = not np.array_equal(t["x"], s["x"])
        if not np.array_equal(s["x"], P.x):
            fail(k, "the state is not the point the reference stands on")
        if accepted:
            d = t["x"] - s["x"]
            if (d[:nc][P.held] != 0).any():
                fail(k, "a held camera parameter moved")
            if (d[nc:].reshape(-1, 6)[P.ev.empty] != 0).any():
                fail(k, "the pose of a frame without observations moved")
            # d = x_{k+1} - x_k is exact (Sterbenz) but x_{k+1} = fl(x_k + d) rounded by half an ulp of itself
            d_read = 0.5 * EPS * np.abs(t["x"])
            omega = P.backward_error(d, lam, d_read, G_ROUND_ULPS * EPS * P.ev.g_round)
            err("step backward error", omega)
            if not omega <= BACKWARD_TOL:
                fail(k, f"step: backward error {omega:.3g} in the reference's damped system (lambda {lam:.6g})")
            sn = np.linalg.norm(d)
            sn_tol = STEP_RTOL * sn + np.linalg.norm(d_read)      # the read-back step's norm is known to this
            rec = by_nfev.get(k + 2)
            if rec is None or rec[0] != n_acc + 1:
                fail(k, f"no iteration record for the accepted step (iteration {n_acc + 1}, nfev {k + 2})")
            pred = P.pred(d, lam)
            x_ok = decide(k, "xtol", [(sn, o["xtol"] * (o["xtol"] + xn), sn_tol)], last and t["status"] in (3, 4))
            n_acc += 1
            mode = P.mode
            old_cost, old = P.cost, P
            # the weight mode at the new point: decided below from the reduction the reference measures there
            cost_new = robust_cost(t["x"], uvs, obj, o["loss"], o["f_scale"])[0]
            actual = old_cost - cost_new
            margin = COST_ULP * old_cost
            if actual <= -margin:
                fail(k, f"accepted a step that raises the cost by {-actual:.6g}")
            ratio = actual / pred if pred > 0 else -1.0
            d_ratio = margin / abs(pred) + PRED_RTOL * abs(ratio) if pred > 0 else 0.0
            f_ok = decide(k, "ftol", [(actual, o["ftol"] * old_cost, margin), (-ratio, -0.25, d_ratio)],
                          last and t["status"] in (2, 4))
            term = 4 if (f_ok and x_ok) else 2 if f_ok else 3 if x_ok else None
            if mode == "irls" and o["hessian"] == "auto":
                guess = last_rel < 0.1          # the engine walks the trial with Triggs weights already
                if actual < SWITCH * old_cost:
                    mode = "triggs"     # not reported by the solver: checked through the next step's reduced system
                    if guess:
                        events.add("switch, guessed")
                    elif term is None:      # a step that ends the solve needs no new system: no walk at all
                        events.add("switch, re-walk")
                elif guess and term is None:
                    events.add("no switch, re-walk")
            last_rel = actual / old_cost
            if abs(actual - SWITCH * old_cost) <= margin:
                ties.append((k, "1 % switch (not followable)", [(float(actual), float(SWITCH * old_cost))]))
            P = Point(t["x"], uvs, obj, o, mode, old.D2cam, old.D2pose, lam=t["lam"])
            # what the solver reported for this iteration
            for name, got, want, tol in (("record cost", rec[2], P.cost, 1e-12 * old_cost),
                                         ("record actual", rec[3], actual, 1e-12 * old_cost),
                                         ("record step norm", rec[4], sn, sn_tol),
                                         ("record gnorm", rec[5], P.gnorm, 1e-10 * g0)):
                err(name, abs(got - want) / max(tol, np.finfo(float).tiny))
                if not abs(got - want) <= tol:
                    fail(k, f"{name}: solver {got!r}, reference {want!r} (tolerance {tol:.3g})")
            last_sn = rec[4]
            # damping
            lam_ref = damping_update(lam, ratio, o["lambda_min"])
            tt = 2 * ratio - 1
            rtol = 6 * tt * tt * d_ratio / max(0.1, 1 - tt ** 3) + 1e-15     # from the uncertainty of the ratio
            free = lam * max(0.1, 1 - tt ** 3)
            ok_lam = abs(t["lam"] - lam_ref) <= rtol * lam_ref
            if abs(free - o["lambda_min"]) <= rtol * free:                  # the lambda_min clamp is a tie
                ok_lam |= t["lam"] == o["lambda_min"] or abs(t["lam"] - free) <= rtol * free
            err("lambda / its tolerance", abs(t["lam"] - lam_ref) / lam_ref / rtol)
            if t["lam"] == o["lambda_min"] and lam_ref == o["lambda_min"]:
                events.add("lambda_min clamp")
            if not ok_lam:
                fail(k, f"lambda after an accepted step: solver {t['lam']!r}, reference {lam_ref!r} (ratio {ratio:.6g})")
            nu = 2.0
            pattern.append("A")
            if term is not None:
                expect_status = term
            elif decide(k, "gtol", [(P.gnorm, o["gtol"], gtol_margin)], last and t["status"] == 1):
                expect_status = 1
            if expect_status is not None and not last:
                fail(k, f"the reference ends the solve here with status {expect_status}, the solver goes on")
        else:
            d_ref = P.step(lam)
            cost_new = robust_cost(P.x + d_ref, uvs, obj, o["loss"], o["f_scale"])[0]
            actual = P.cost - cost_new
            pred = P.pred(d_ref, lam)
            margin = COST_ULP * P.cost + STEP_RTOL * abs(pred)
            decide(k, "accept", [(-actual, 0.0, margin)], False)
            sn = np.linalg.norm(d_ref)
            if decide(k, "xtol (rejected)", [(sn, o["xtol"] * (o["xtol"] + xn), STEP_RTOL * sn)],
                      last and t["status"] == 3):
                expect_status = 3
                if t["lam"] != lam:
                    fail(k, "lambda changed on the rejected step that met xtol")
            else:
                lam_ref = lam * nu
                if t["lam"] != lam_ref:
                    fail(k, f"lambda after a rejection: solver {t['lam']!r}, expected {lam_ref!r} = lambda * nu")
                nu *= 2.0
                if lam_ref > o["lambda_max"]:
                    expect_status = -1
            pattern.append("r")
            if expect_status is not None and not last:
                fail(k, f"the reference ends the solve here with status {expect_status}, the solver goes on")
        if not np.array_equal(t["x"], P.x):
            fail(k, "internal: the reference did not move with the solver")
        check_point_values(k + 1, t)
    if expect_status is None:
        expect_status = 0
        if o["max_nfev"] is not None and full["nfev"] < o["max_nfev"]:
            fail(len(states) - 1, f"the solve stopped with status {full['status']} before its budget "
                                  f"where the reference goes on")
    # totals: the full run and the run cut at its own nfev must both agree with the replay
    K = len(states)
    cost, sumsq, n = robust_cost(P.x, uvs, obj, o["loss"], o["f_scale"])
    for tag, r in (("full run", full), (f"run cut at max_nfev={K}", states[-1])):
        checks = (("status", r["status"] == expect_status, r["status"], expect_status),
                  ("nfev", r["nfev"] == K, r["nfev"], K),
                  ("njev", r["njev"] == 1 + n_acc, r["njev"], 1 + n_acc),
                  ("iterations", r["iterations"] == n_acc, r["iterations"], n_acc),
                  ("x", np.array_equal(r["x"], P.x), "", ""),
                  ("damping", r["lam"] == states[-1]["lam"], r["lam"], states[-1]["lam"]),
                  ("step_norm", r.get("step_norm") is None or abs(r["step_norm"] - last_sn) <= 1e-15 * last_sn,
                   r.get("step_norm"), last_sn),
                  ("cost", abs(r["cost"] - P.cost) <= 1e-12 * P.cost, r["cost"], P.cost),
                  ("optimality", abs(r["optimality"] - P.gnorm) <= 1e-10 * g0, r["optimality"], P.gnorm),
                  ("rms", r.get("rms") is None or abs(r["rms"] - np.sqrt(sumsq / n)) <= 1e-12 * np.sqrt(sumsq / n),
                   r.get("rms"), np.sqrt(sumsq / n)))
        for name, ok, got, want in checks:
            if not ok:
                raise ReplayError(f"{tag} after {K} evaluations: {name} {got!r}, the replay gives {want!r}")
    report = dict(pattern="".join(pattern), status=expect_status, errors=errs, ties=ties, transitions=K - 1,
                  events=sorted(events))
    if log:
        log(f"  {K - 1} transitions, status {expect_status}: {report['pattern'] or '(none)'}")
        log("  largest errors: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(errs.items())))
        log(f"  ties: {len(ties)} {ties if ties else ''}")
        log(f"  events: {report['events']}")
    return report
