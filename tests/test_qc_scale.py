"""Reprojection-error QC (viz.reprojection_residuals: homography_transfer_kernel in k7_qc.cu and the
radix-selection median of viz._device_median) at production sizes, up to 32 cameras, boards of 4 to
128 corners, with all five distortion coefficients and a skewed K.

Checks, per scene:
1. against the same algorithm (the oracle's restatement of cv2, ``tests/qc_reference.py``) frame by
   frame: identical NaN pattern, transferred corners within FRAME_TOL on >= FRAME_FRAC of the frames,
   and every other frame a valid end point of the same LM (its objective no worse than the DLT's and,
   where the oracle's LM converged, within S_TOL of the converged float64 minimiser's);
2. against exact truth on a noise-free distortion-free rig, with a per-frame bound from the float32
   rounding of the detections inside findHomography, the board size and the pixel scale;
3. the per-camera median exactly (4 ulp) against np.nanmedian of the kernel's own transferred corners;
4. against the real OpenCV calls on a sample of frames, where cv2 is importable.
The CPU tests at the end show that checks 1-3 reject plausible wrong kernels.
"""
import functools
import re
import time

import numpy as np
import pytest

from conftest import split_cams
from oracle import np_oracle as orc
import qc_reference as qr
import multicam_calibration_b200 as mcc
from multicam_calibration_b200.synthetic import forward_model, make_scene

gpu = pytest.mark.gpu

# Tolerances, measured on a B200 (the per-scene values print with pytest -s).
# FRAME_TOL / FRAME_FRAC: where the kernel and the oracle take the same LM path the transferred corners
# differ by the eigen-solver's and FMA's rounding only (exact rig: 2.1e-7 at most).  The frames outside
# are boards seen at a grazing angle, where ten LM iterations do not reach the minimiser and rounding
# sends the two down different paths: 96.5 % (32 cameras) to 100 % (4 corners) of the frames were
# within FRAME_TOL.
FRAME_TOL = 1e-6          # board units (mm)
FRAME_FRAC = 0.95
# S checks on the frames outside FRAME_TOL, relative to S* + 2 N FRAME_TOL^2 (residuals below FRAME_TOL
# do not matter; S* is ~0 on a 4-corner board): the kernel never ends above the DLT (measured: always
# below it), and where the oracle converged (within CONVERGED of S*) the kernel ends within S_TOL of S*.
# The oracle's own LM ends within 5e-6 S* on 99 % of the frames and up to 2.6 S* above it on grazing
# frames; there the kernel, like cv2 (up to 2 S* where the oracle converged), may stop a few iterations
# short: measured 0.034 at worst.  A kernel without the refinement ends 2.9 S* above, one with the skew
# in the normalisation 1.05 (test_same_algorithm_check_rejects_wrong_kernels).
CONVERGED = 1e-5
S_TOL = 0.1
U32 = 2.0 ** -24          # unit roundoff of float32
MEDIAN_ULP = 4            # measured: 1 ulp at most, on every scene
# cv2 against the kernel, sampled frames within 1e-5 board units: 94.2 % (full distortion and skew)
# to 100 % (4 corners); test_io_qc_cpu's 95 % holds on qc.npz's 48 frames, not on 20,000.
CV2_FRAC = 0.93


# ------------------------------------------------------------------ scenes
def _full_distortion(scene_cams, strength, skew):
    """(ext, intr) of a make_scene rig with all five coefficients at ``strength`` times those of
    tests/golden/qc.npz (k1, k2 from the rig, p1 = 1e-4 (c + 1), p2 = -2e-4, k3 = 1e-3) and K[0, 1] = skew."""
    ext, intr = split_cams(scene_cams)
    out = []
    for c, (K, d) in enumerate(intr):
        K = K.copy()
        K[0, 1] = skew
        out.append((K, strength * np.array([d[0], d[1], 1e-4 * (c + 1), -2e-4, 1e-3])))
    return ext, out


def _detections(ext, intr, obj, poses, sigma, rng):
    """Detections of the board corners through the full (k1, k2, p1, p2, k3) model and a skewed K."""
    pts = orc.embed_calib_objpoints(obj, poses)
    uvs = np.empty((len(ext), len(poses), len(obj), 2))
    for c, (K, d) in enumerate(intr):
        Xc = orc.apply_rigid_transform(ext[c], pts)
        x, y = Xc[..., 0] / Xc[..., 2], Xc[..., 1] / Xc[..., 2]
        k1, k2, p1, p2, k3 = d
        r2 = x * x + y * y
        rad = 1 + r2 * (k1 + r2 * (k2 + r2 * k3))
        xd = x * rad + 2 * p1 * x * y + p2 * (r2 + 2 * x * x)
        yd = y * rad + p1 * (r2 + 2 * y * y) + 2 * p2 * x * y
        uvs[c, ..., 0] = K[0, 0] * xd + K[0, 1] * yd + K[0, 2]
        uvs[c, ..., 1] = K[1, 1] * yd + K[1, 2]
    return uvs + rng.normal(0, sigma, uvs.shape) if sigma else uvs


def _distorted(C, F, board=(5, 7), strength=1.0, skew=0.0, sigma=0.5, p_view=0.2, p_corner=0.0, seed=0):
    sc = make_scene(C, F, board=board, sigma=0.0, seed=seed)
    ext, intr = _full_distortion(sc.true_cams, strength, skew)
    rng = np.random.default_rng([seed, 17])
    uvs = _detections(ext, intr, sc.objpoints, sc.true_poses, sigma, rng)
    uvs[rng.random((C, F)) < p_view] = np.nan
    if p_corner:
        uvs[rng.random((C, F, len(sc.objpoints))) < p_corner] = np.nan
    return qr.Scene(uvs, ext, intr, sc.objpoints, sc.true_poses)


def _production():
    """configs[2] as bench.py builds it: 6 x 50,000 x 35, sigma 0.5 px, 20 % missing views; the QC runs
    with the true calibration (k1, k2 only) and board poses."""
    sc = make_scene(6, 50_000, sigma=0.5, p_missing_view=0.2, seed=0)
    ext, intr = split_cams(sc.true_cams)
    return qr.Scene(sc.uvs, ext, intr, sc.objpoints, sc.true_poses)


def _dropouts():
    """Per-corner dropouts, camera 3 with no complete frame, camera 0 with an even and camera 1 with an
    odd number of complete frames (35 corners: the parity of the median's count), 6 x 3,001 pairs so
    the last CTA of 64 is partial."""
    s = _distorted(6, 3001, strength=1.0, skew=0.4, p_corner=0.002, seed=31)
    rng = np.random.default_rng(32)
    s.uvs[3, np.arange(3001), rng.integers(0, 35, 3001)] = np.nan
    for c, parity in ((0, 0), (1, 1)):
        complete = np.nonzero(s.complete()[c])[0]
        if len(complete) % 2 != parity:
            s.uvs[c, complete[0], 0] = np.nan
    return s


def _exact(C=16, F=5000, board=(9, 11), seed=2):
    """Noise-free detections of a distortion-free rig (make_scene's k1, k2 set to 0)."""
    sc = make_scene(C, F, board=board, sigma=0.0, seed=seed)
    cams = sc.true_cams.copy()
    cams[:, 4:6] = 0.0
    ext, intr = split_cams(cams)
    return qr.Scene(forward_model(cams, sc.true_poses, sc.objpoints), ext, intr, sc.objpoints, sc.true_poses)


SCENES = {
    "production_6x50000": _production,
    "cams32_32x2000": lambda: _distorted(32, 2000, seed=5),
    "board2x2_6x3000": lambda: _distorted(6, 3000, board=(2, 2), seed=6),
    "board6x6_6x3000": lambda: _distorted(6, 3000, board=(6, 6), seed=7),
    "board9x11_6x3000": lambda: _distorted(6, 3000, board=(9, 11), seed=8),
    "board8x16_6x3000": lambda: _distorted(6, 3000, board=(8, 16), seed=9),
    "distortion1x_skew_6x3000": lambda: _distorted(6, 3000, strength=1.0, skew=0.8, seed=10),
    "distortion3x_skew_6x3000": lambda: _distorted(6, 3000, strength=3.0, skew=-1.5, seed=11),
    "dropouts_6x3001": _dropouts,
    "exact_16x5000x99": _exact,
}


@functools.lru_cache(maxsize=None)
def scene(name):
    return SCENES[name]()


def sample_pairs(s, n, seed, extra=()):
    """A fixed random sample of ``n`` complete (camera, frame) pairs (all of them when fewer), sorted,
    with the incomplete pairs ``extra`` appended."""
    complete = np.argwhere(s.complete())
    rng = np.random.default_rng(seed)
    if len(complete) > n:
        complete = complete[np.sort(rng.choice(len(complete), n, replace=False))]
    return np.concatenate([complete, np.asarray(extra, dtype=complete.dtype).reshape(-1, 2)])


# ------------------------------------------------------------------ checks shared by the GPU and CPU tests
def frame_diff(a, b):
    """Per frame, the largest |a - b| over its corners (0 where both are NaN rows)."""
    ok = ~np.isnan(b).any((-1, -2))
    return np.abs(np.where(ok[:, None, None], a - b, 0.0)).max((-1, -2)), ok


def same_algorithm_check(tr, ref):
    """Check 1 on one set of pairs: ``tr`` (P, N, 2) the kernel's transfer, ``ref`` qr.transfer's.
    Returns a dict; ``ok`` is the verdict."""
    nan_same = bool(np.array_equal(np.isnan(tr), np.isnan(ref["tr"])))
    diff, ok = frame_diff(tr, ref["tr"])
    good = ok & (diff <= FRAME_TOL)
    frac = float(good.sum() / max(ok.sum(), 1))
    worst_gap, worst_dlt, unconverged = 0.0, -np.inf, 0
    for i in np.nonzero(ok & ~good)[0]:
        M, m = ref["M"][i], ref["m"][i]
        if not np.isfinite(tr[i]).all():
            worst_gap = np.inf
            break
        S_k = qr.sum_squares(qr.recover_homography(ref["rep"][i], tr[i]), M, m)
        S_star = qr.sum_squares(qr.converged_minimiser(ref["H"][i], M, m), M, m)
        S_o = qr.sum_squares(ref["H"][i], M, m)
        S_dlt = qr.sum_squares(ref["H_dlt"][i], M, m)
        scale = S_star + 2 * len(M) * FRAME_TOL ** 2
        worst_dlt = max(worst_dlt, (S_k - S_dlt) / scale)
        if S_o - S_star <= CONVERGED * scale:
            worst_gap = max(worst_gap, (S_k - S_star) / scale)
        else:
            unconverged += 1
    return dict(ok=bool(nan_same and frac >= FRAME_FRAC and worst_gap <= S_TOL and worst_dlt <= S_TOL),
                nan_same=nan_same, frac_within=frac, frames=int(ok.sum()), outside=int((ok & ~good).sum()),
                unconverged=unconverged, max_diff=float(diff[ok].max(initial=0.0)), worst_gap=float(worst_gap),
                worst_vs_dlt=float(worst_dlt))


def exact_bound(s, pairs):
    """Per pair, the bound of check 2.  float32 rounding moves detection n by up to u32 |uv_n| per
    coordinate; the board plane sees that as s_n u32 |uv_n|, with s_n the local scale in board units
    per pixel (the largest ratio of a grid edge at corner n to its image).  A least-squares fit carries
    input errors into its output through a projection, so to first order no transferred corner moves
    by more than the 2-norm of those errors.  Boards seen at a grazing angle are far from first order:
    there :func:`exact_check` falls back to the error of the float64 minimiser of the rounded points."""
    rows, cols = np.unique(s.obj[:, 0]).size, np.unique(s.obj[:, 1]).size
    uv = s.uvs[pairs[:, 0], pairs[:, 1]].reshape(len(pairs), cols, rows, 2)
    grid = s.obj[:, :2].reshape(cols, rows, 2)
    scale = np.zeros(uv.shape[:3])
    for axis in (1, 2):
        ratio = np.linalg.norm(np.diff(grid, axis=axis - 1), axis=-1)[None] / np.linalg.norm(np.diff(uv, axis=axis), axis=-1)
        lo = [slice(None)] * 3
        hi = [slice(None)] * 3
        lo[axis], hi[axis] = slice(None, -1), slice(1, None)
        scale[tuple(lo)] = np.maximum(scale[tuple(lo)], ratio)
        scale[tuple(hi)] = np.maximum(scale[tuple(hi)], ratio)
    moved = scale * U32 * np.abs(uv).max(-1)
    return np.sqrt(2.0 * (moved ** 2).reshape(len(pairs), -1).sum(1))


def exact_check(tr, s, pairs):
    """Check 2: every transferred corner of ``tr`` (P, N, 2) within its frame's :func:`exact_bound`, or
    where that first-order bound is exceeded, within twice the error of H* (the float64 minimiser of
    the same objective on the same float32-rounded points: the error the rounding itself causes)."""
    err = np.linalg.norm(tr - s.obj[:, :2], axis=-1).max(-1)
    bound = exact_bound(s, pairs)
    over = np.nonzero(~(err <= bound))[0]
    if len(over):
        ref = qr.transfer(s, pairs[over])
        for j, i in enumerate(over):
            if np.isnan(ref["H"][j]).any():
                continue
            Hs = qr.converged_minimiser(ref["H"][j], ref["M"][j], ref["m"][j])
            e_star = np.linalg.norm(orc.perspective_transform(ref["rep"][j], Hs) - s.obj[:, :2], axis=-1).max()
            bound[i] = max(bound[i], 2.0 * e_star)
    ratio = err / bound
    return dict(ok=bool(np.isfinite(ratio).all() and ratio.max() <= 1.0), max_err=float(err.max()),
                worst_ratio=float(ratio.max()), fallback=int(len(over)), bound_median=float(np.median(bound)))


def median_check(med, tr, obj):
    """Check 3: ``med`` within MEDIAN_ULP ulp of np.nanmedian of the distances of ``tr`` (C, F, N, 2)."""
    host = qr.camera_medians(tr, obj)
    nan_same = bool(np.array_equal(np.isnan(med), np.isnan(host)))
    fin = ~np.isnan(host)
    ulps = np.abs(med[fin] - host[fin]) / np.spacing(host[fin]) if fin.any() else np.zeros(0)
    counts = (~np.isnan(tr).any(-1)).reshape(len(tr), -1).sum(1)
    return dict(ok=bool(nan_same and ulps.max(initial=0.0) <= MEDIAN_ULP), nan_same=nan_same,
                max_ulp=float(ulps.max(initial=0.0)), counts=counts.tolist())


def opencv_check(tr, cv, obj):
    """Check 4 on one set of pairs, compare_transfer's rule (test_io_qc_cpu.py) against cv2's output
    ``cv``: NaN pattern equal, >= CV2_FRAC of the frames within 1e-5 board units, per camera the
    medians over those frames within 1e-6 relative and over all sampled frames within 1e-2."""
    nan_same = bool(np.array_equal(np.isnan(tr), np.isnan(cv)))
    diff, ok = frame_diff(tr, cv)
    good = ok & (diff <= 1e-5)
    frac = float(good.sum() / max(ok.sum(), 1))
    worst_good, worst_all = 0.0, 0.0
    e_k, e_c = np.linalg.norm(tr - obj[:, :2], axis=-1), np.linalg.norm(cv - obj[:, :2], axis=-1)
    for sel in (good, ok):
        a, b = np.median(e_k[sel]), np.median(e_c[sel])
        if sel is good:
            worst_good = abs(a - b) / b
        else:
            worst_all = abs(a - b) / b
    return dict(ok=bool(nan_same and frac >= CV2_FRAC and worst_good <= 1e-6 and worst_all <= 1e-2),
                nan_same=nan_same, frac_within=frac, median_rel_good=float(worst_good), median_rel_all=float(worst_all))


# ------------------------------------------------------------------ GPU: every scene
@functools.lru_cache(maxsize=None)
def kernel_run(name):
    s = scene(name)
    t = time.perf_counter()
    out = mcc.reprojection_residuals(*s.args())
    return out, time.perf_counter() - t


@gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_qc_scene_against_oracle_and_exact_median(name):
    s = scene(name)
    (med, rep, tr), seconds = kernel_run(name)
    C, F, N = s.uvs.shape[:3]
    assert med.shape == (C,) and rep.shape == tr.shape == (C, F, N, 2)
    # NaN rows exactly where a corner is missing (no scene here has a degenerate board)
    complete = s.complete()
    assert np.array_equal(~np.isnan(tr).any((-1, -2)), complete)
    assert np.array_equal(np.isnan(tr).all((-1, -2)), ~complete)
    # check 3 on every value of the launch
    m3 = median_check(med, tr, s.obj)
    print(f"\n{name}: {C} x {F} x {N} in {seconds:.2f} s; median max {m3['max_ulp']:.3g} ulp, "
          f"counts {m3['counts'][:4]}{'...' if C > 4 else ''}")
    assert m3["ok"], m3
    # check 1 on a fixed sample (the oracle fits about 2,500 frames a second)
    incomplete = np.argwhere(~complete)[:256]
    pairs = sample_pairs(s, 4000 if N > 64 else 15000, seed=len(name), extra=incomplete)
    ref = qr.transfer(s, pairs)
    np.testing.assert_allclose(rep[pairs[:, 0], pairs[:, 1]], ref["rep"], rtol=0, atol=1e-9)   # pixels
    m1 = same_algorithm_check(tr[pairs[:, 0], pairs[:, 1]], ref)
    print(f"{name}: oracle on {m1['frames']} frames: {m1['frac_within']:.4%} within {FRAME_TOL:g}, "
          f"max |diff| {m1['max_diff']:.3g}, {m1['outside']} outside ({m1['unconverged']} where the oracle did not "
          f"converge): worst S - S* {m1['worst_gap']:.3g}, worst S - S(DLT) {m1['worst_vs_dlt']:.3g} (of S* + floor)")
    assert m1["ok"], m1
    if name.startswith("exact"):
        # check 2 on every frame
        idx = np.argwhere(complete)
        m2 = exact_check(tr[idx[:, 0], idx[:, 1]], s, idx)
        print(f"{name}: exact truth on {len(idx)} frames: max error {m2['max_err']:.3g}, largest error/bound "
              f"{m2['worst_ratio']:.3g}, bound median {m2['bound_median']:.3g}, {m2['fallback']} frames on H*")
        assert m2["ok"], m2
        assert np.all(med < 1e-4)


@gpu
@pytest.mark.parametrize("name", [n for n in SCENES if not n.startswith("exact")])
def test_qc_scene_against_opencv(name):
    pytest.importorskip("cv2")
    s = scene(name)
    (med, rep, tr), _ = kernel_run(name)
    pairs = sample_pairs(s, 20000, seed=len(name) + 1, extra=np.argwhere(~s.complete())[:256])
    t = time.perf_counter()
    cv = qr.cv2_transfer(s, pairs)
    m4 = opencv_check(tr[pairs[:, 0], pairs[:, 1]], cv, s.obj)
    print(f"\n{name}: cv2 on {len(pairs)} pairs ({time.perf_counter() - t:.1f} s): {m4['frac_within']:.4%} within 1e-5, "
          f"medians over those {m4['median_rel_good']:.3g}, over all {m4['median_rel_all']:.3g} relative")
    assert m4["ok"], m4


# ------------------------------------------------------------------ GPU: edges and limits
@gpu
def test_collinear_board_gives_nan_rows_and_median():
    """A board of one row: findHomography's DLT sees zero spread along the board's x axis.  cv2 returns
    None there and the reference's plot_residuals would raise on it; the kernel gives NaN rows, so the
    camera's median is NaN, and frames of a proper board in the same call are unaffected."""
    s = _distorted(3, 130, board=(1, 9), seed=12)
    med, _, tr = mcc.reprojection_residuals(*s.args())
    assert np.isnan(tr).all() and np.isnan(med).all()


@gpu
def test_limits_raise_with_the_kernel_message():
    msg = re.escape("mcba_homography_transfer: at most 32 cameras and 128 points per frame")
    s = _distorted(2, 8, board=(3, 43), seed=13)                       # 129 corners
    with pytest.raises(mcc._native.McbaError, match=msg):
        mcc.reprojection_residuals(*s.args())
    s = _distorted(33, 8, seed=14)
    with pytest.raises(mcc._native.McbaError, match=msg):
        mcc.reprojection_residuals(*s.args())
    s = _distorted(2, 8, board=(1, 3), seed=15)                        # 3 corners
    with pytest.raises(mcc._native.McbaError, match=re.escape("at least 4 points per frame")):
        mcc.reprojection_residuals(*s.args())


@gpu
def test_no_frames():
    s = _distorted(3, 5, seed=16)
    med, rep, tr = mcc.reprojection_residuals(s.uvs[:, :0], list(s.ext), s.intr, s.obj, s.poses[:0])
    assert rep.shape == tr.shape == (3, 0, 35, 2) and med.shape == (3,) and np.isnan(med).all()


# ------------------------------------------------------------------ 4 corners: refined or not (CPU)
def test_four_corner_refinement_stays_at_rounding_level():
    """cv2.findHomography refines only when N > 4; the kernel and the oracle also refine at N = 4.  With 4
    points the DLT fits exactly, so the refinement only moves the result by rounding: on 6 x 400 frames
    of a 2 x 2 board it moved the transferred corners by at most 1.4e-10 board units (median 4e-14),
    and the refined and unrefined transfers agree with cv2 to the same quantiles (99 %: 9e-11, both)."""
    s = _distorted(6, 400, board=(2, 2), seed=6)
    pairs = sample_pairs(s, 10 ** 9, 0)
    ref = qr.transfer(s, pairs)
    dlt = np.stack([orc.perspective_transform(r, H) for r, H in zip(ref["rep"], ref["H_dlt"])])
    moved = np.abs(dlt - ref["tr"]).max((-1, -2))
    print(f"\n4 corners: refinement moves the transfer by at most {moved.max():.3g} (median {np.median(moved):.3g})")
    assert moved.max() <= 1e-8 and np.median(moved) <= 1e-12
    cv2 = pytest.importorskip("cv2")  # noqa: F841
    cv = qr.cv2_transfer(s, pairs)
    q_ref = np.quantile(np.abs(ref["tr"] - cv).max((-1, -2)), 0.99)
    q_dlt = np.quantile(np.abs(dlt - cv).max((-1, -2)), 0.99)
    print(f"4 corners vs cv2, 99th percentile: refined {q_ref:.3g}, DLT only {q_dlt:.3g}")
    assert q_ref <= 1e-8 and q_dlt <= 1e-8


# ------------------------------------------------------------------ the checks reject wrong kernels (CPU)
def _cpu_scene():
    return _distorted(6, 240, strength=3.0, skew=-1.5, seed=21)


WRONG = {"no float32 rounding": dict(round32=False), "no LM refinement": dict(refine=False),
         "4 undistortion iterations": dict(n_iter=4), "skew in the normalisation": dict(skew_in_norm=True)}


def test_checks_accept_the_oracle():
    s = _cpu_scene()
    pairs = sample_pairs(s, 10 ** 9, 0)
    ref = qr.transfer(s, pairs)
    assert same_algorithm_check(ref["tr"], ref)["ok"]
    tr = np.full(s.uvs.shape, np.nan)
    tr[pairs[:, 0], pairs[:, 1]] = ref["tr"]
    assert median_check(qr.camera_medians(tr, s.obj), tr, s.obj)["ok"]
    e = _exact(2, 150)
    idx = sample_pairs(e, 10 ** 9, 0)
    m2 = exact_check(qr.transfer(e, idx)["tr"], e, idx)
    print(f"\noracle: exact truth error/bound {m2['worst_ratio']:.3g}")
    assert m2["ok"], m2


@pytest.mark.parametrize("wrong", sorted(WRONG))
def test_same_algorithm_check_rejects_wrong_kernels(wrong):
    s = _cpu_scene()
    pairs = sample_pairs(s, 10 ** 9, 0)
    ref = qr.transfer(s, pairs)
    bad = qr.transfer(s, pairs, **WRONG[wrong])
    m1 = same_algorithm_check(bad["tr"], ref)
    print(f"\n{wrong}: {m1['frac_within']:.4%} within {FRAME_TOL:g}, worst S - S* {m1['worst_gap']:.3g}")
    assert not m1["ok"]


def test_median_check_rejects_the_lower_middle_value():
    s = _cpu_scene()
    pairs = sample_pairs(s, 10 ** 9, 0)
    tr = np.full(s.uvs.shape, np.nan)
    tr[pairs[:, 0], pairs[:, 1]] = qr.transfer(s, pairs)["tr"]
    counts = (~np.isnan(tr).any(-1)).reshape(len(tr), -1).sum(1)
    assert (counts % 2 == 0).any()
    m3 = median_check(qr.camera_medians(tr, s.obj, how="lower"), tr, s.obj)
    print(f"\nlower middle value: {m3['max_ulp']:.3g} ulp")
    assert not m3["ok"]
