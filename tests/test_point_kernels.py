"""Point kernels at production sizes, beyond eight cameras and on the triangulation fallback.

Triangulation (k5_points.cu) is checked against bounds derived from the numpy SVD of every pair's
DLT matrix (``tests/point_reference.py``): a pair's solution must satisfy the residual and
forward-error bounds of a backward-stable solve, and an all-pairs median must be within the largest
bound among the point's pairs of ``orc.triangulate``.  The DLT matrices are built from
``mcc.undistort_points``, which runs the kernel's own ``undistort5``.  Projection, undistortion,
board embedding, the consensus board poses (k6_init.cu) and the frame selection (k0_frontend.cu) are
compared with the oracle past one grid-stride round and at every template instantiation.  The CPU
tests at the end show that the triangulation checks reject plausible wrong kernels.
"""
import re

import numpy as np
import pytest

from conftest import split_cams
from oracle import np_oracle as orc
import point_reference as pr
import multicam_calibration_b200 as mcc
from multicam_calibration_b200.synthetic import make_camera_poses, make_keypoints, make_scene

gpu = pytest.mark.gpu
CEILING_MM = 1e-9      # absolute ceiling of a median against the oracle (configs[4]: 2.2e-11 on 5,000 points)


# ------------------------------------------------------------------ checks shared by the GPU and CPU tests
def pair_check(all_uvs, ext, intr, out, und):
    """Residual and forward-error ratios (each must be <= 1) of a 2-camera triangulation ``out``."""
    Ps = pr.projection_matrices(ext, intr)
    A = pr.dlt(und[0], und[1], Ps[0], Ps[1])
    return pr.pair_ratios(A, out)


def median_check(out, ref, und, ext, intr):
    """An all-pairs triangulation ``out`` against the oracle's ``ref``: identical NaN pattern, and
    every point within its pair bound and within ``CEILING_MM``.  Returns a dict; ``ok`` is the verdict."""
    tol, npairs = pr.point_tolerance(und, pr.projection_matrices(ext, intr))
    nan_same = np.array_equal(np.isnan(out), np.isnan(ref))
    fin = ~np.isnan(ref).any(1)
    with np.errstate(invalid="ignore"):
        diff = np.nan_to_num(np.abs(out[fin] - ref[fin]), nan=np.inf).max(1) if fin.any() else np.zeros(0)
    ratio = diff / tol[fin] if fin.any() else np.zeros(0)
    worst = float(ratio.max()) if ratio.size else 0.0
    maxdiff = float(diff.max()) if diff.size else 0.0
    return dict(ok=bool(nan_same and worst <= 1.0 and maxdiff <= CEILING_MM), nan_same=nan_same,
                worst_ratio=worst, max_diff=maxdiff, pair_counts=set(np.unique(npairs[fin]).tolist()))


def device_undistorted(all_uvs, intr):
    return np.stack([mcc.undistort_points(u, K, dc) for u, (K, dc) in zip(all_uvs, intr)])


def oracle_undistorted(all_uvs, intr):
    return np.stack([orc.undistort_points(u, K, dc) for u, (K, dc) in zip(all_uvs, intr)])


# ------------------------------------------------------------------ 1. the pair solver on its own
@gpu
@pytest.mark.parametrize("kind", ["ring", "baseline", "parallel", "exact"])
def test_pair_solver_within_svd_bounds(kind):
    all_uvs, ext, intr = pr.pair_rig(kind)
    out = mcc.triangulate(all_uvs, list(ext), intr)
    und = device_undistorted(all_uvs, intr)
    Ps = pr.projection_matrices(ext, intr)
    A = pr.dlt(und[0], und[1], Ps[0], Ps[1])
    if kind == "baseline":
        print(f"rig {kind}: Jacobi fallback on {1 - pr.qr_settles(A).mean():.1%} of the pairs")
    if kind == "parallel":
        # the exact point is at infinity along the common ray: the result is huge or infinite and
        # parallel to the ray, like the oracle's
        _, v, theta = pr.svd_bound(A)
        d = pr.ray_directions(und[0], ext[0], intr[0][0])
        ref = orc.triangulate(all_uvs, list(ext), intr)
        for name, p in (("device", out), ("oracle", ref)):
            assert not np.isnan(p).any(), name
            fin = np.isfinite(p).all(1)
            assert np.isinf(p[~fin]).all(), name                       # all three coordinates infinite
            s = np.sign(p[~fin])
            sd = np.sign(d[~fin])
            assert np.all((s == sd).all(1) | (s == -sd).all(1)), name
            x = pr.unit_homogeneous(p[fin])
            assert np.all(np.abs(x[:, 3]) <= theta[fin]), name            # |p| >~ 1 / theta
            res, fwd = pr.pair_ratios(A[fin], p[fin])
            assert np.nanmax(res, initial=0) <= 1 and np.nanmax(fwd, initial=0) <= 1, name
            print(f"rig {kind} ({name}): {int((~fin).sum())} infinite, smallest finite |p| "
                  f"{np.linalg.norm(p[fin], axis=1).min(initial=np.inf):.3g} mm, "
                  f"residual {np.nanmax(res, initial=0):.3g}, forward {np.nanmax(fwd, initial=0):.3g}")
        return
    assert np.isfinite(out).all()
    res, fwd = pr.pair_ratios(A, out)
    print(f"rig {kind}: largest measured/bound ratio residual {res.max():.3g}, forward {fwd.max():.3g}")
    assert res.max() <= 1.0 and fwd.max() <= 1.0


# ------------------------------------------------------------------ 2. configs[4] in full
@gpu
def test_configs4_full_workload_against_oracle():
    """1 M points x 6 cameras, sigma 0.3 px, 20 % missing views (the bench workload): every grid-stride
    round of the triangulation kernel, both parities of the median."""
    all_uvs, ext, intr, _ = make_keypoints(1_000_000, 6, sigma=0.3, p_missing=0.2, seed=0)
    out = mcc.triangulate(all_uvs, list(ext), intr)
    views = sum((~np.isnan(u).any(1)).astype(int) for u in all_uvs)
    assert np.array_equal(np.isnan(out).any(1), views < 2)
    assert np.array_equal(np.isnan(out).all(1), views < 2)
    sub = [u[::5] for u in all_uvs]
    ref = orc.triangulate(sub, list(ext), intr)
    rep = median_check(out[::5], ref, device_undistorted(sub, intr), ext, intr)
    print(f"configs[4], {len(ref)} points compared: max |diff| {rep['max_diff']:.3g} mm, "
          f"largest diff/bound {rep['worst_ratio']:.3g}, pair counts {sorted(rep['pair_counts'])}")
    assert {1, 3, 6, 10, 15} <= rep["pair_counts"]
    assert rep["ok"], rep


# ------------------------------------------------------------------ 3. camera counts
@gpu
@pytest.mark.parametrize("C", [1, 2, 8, 9, 16, 32])
def test_triangulate_camera_counts(C):
    """C <= 8 runs triangulate_kernel<8>, 9..32 triangulate_kernel<32>; C = 1 has no pair."""
    n = 5000 if C >= 16 else 20000
    all_uvs, ext, intr, _ = make_keypoints(n, C, sigma=0.3, p_missing=0.3, seed=100 + C)
    out = mcc.triangulate(all_uvs, list(ext), intr)
    assert out.shape == (n, 3)
    if C == 1:
        assert np.isnan(out).all()
        return
    ref = orc.triangulate(all_uvs, list(ext), intr)
    rep = median_check(out, ref, device_undistorted(all_uvs, intr), ext, intr)
    print(f"{C} cameras: max |diff| {rep['max_diff']:.3g} mm, largest diff/bound {rep['worst_ratio']:.3g}, "
          f"up to {max(rep['pair_counts'])} pairs per point")
    assert rep["ok"], rep


@gpu
def test_triangulate_rejects_33_cameras():
    all_uvs, ext, intr, _ = make_keypoints(10, 33, sigma=0.3, p_missing=0.0, seed=1)
    with pytest.raises(mcc._native.McbaError, match=re.escape("1 <= n_cameras <= 32")):
        mcc.triangulate(all_uvs, list(ext), intr)


# ------------------------------------------------------------------ 4. non-finite observations
@gpu
def test_triangulate_non_finite_observations_follow_the_oracle():
    """A view whose pixel undistorts to NaN (+-inf, 1e300, one NaN coordinate) is not seen: its pairs
    are dropped, as in the oracle, instead of entering the median as x = +inf."""
    n = 6000
    all_uvs, ext, intr, _ = make_keypoints(n, 6, sigma=0.3, p_missing=0.2, seed=4)
    uvs = [u.copy() for u in all_uvs]
    rng = np.random.default_rng(9)
    groups = np.array_split(rng.permutation(n)[:3000], 6)
    values = [(0, np.inf), (1, -np.inf), (0, 1e300), (1, -1e300), (0, np.nan), (1, np.nan)]
    for g, (coord, val) in zip(groups, values):
        cams = rng.integers(0, 6, len(g))
        for c in range(6):
            uvs[c][g[cams == c], coord] = val
    rest = np.setdiff1d(np.arange(n), np.concatenate(groups))
    two = rng.permutation(rest[~np.isnan(all_uvs[0][rest]).any(1) & ~np.isnan(all_uvs[1][rest]).any(1)])[:300]
    for c in range(2, 6):                               # exactly two views, one of them not finite
        uvs[c][two] = np.nan
    uvs[0][two, 0] = np.inf
    und = device_undistorted(uvs, intr)
    assert np.array_equal(np.isnan(und), np.isnan(oracle_undistorted(uvs, intr)))
    out = mcc.triangulate(uvs, list(ext), intr)
    ref = orc.triangulate(uvs, list(ext), intr)
    assert not np.isinf(out).any()
    assert np.isnan(ref[two]).all() and np.isnan(out[two]).all()
    rep = median_check(out, ref, und, ext, intr)
    print(f"non-finite views: max |diff| {rep['max_diff']:.3g} mm, largest diff/bound {rep['worst_ratio']:.3g}")
    assert rep["ok"], rep


# ------------------------------------------------------------------ 5. projection and undistortion past one grid
def _projection_close(uv, ref, K):
    """NaN and signed-infinity patterns equal; finite values to 1e-12 relative to the sum the
    principal point enters (a pixel near 0 is a cancellation of ``f x`` against ``c``)."""
    assert np.array_equal(np.isnan(uv), np.isnan(ref))
    inf = np.isinf(ref)
    assert np.array_equal(np.isinf(uv), inf) and np.array_equal(uv[inf], ref[inf])
    fin = np.isfinite(ref)
    scale = np.abs(ref) + np.abs(np.array([K[0, 2], K[1, 2]]))
    err = np.abs(uv - ref)[fin] / scale[fin]
    assert err.max() <= 1e-12, err.max()
    return err.max()


def _points_with_plane_and_behind(n, seed):
    """N(0, 80) points; the first 1 % on the plane z = 0, the next 1 % at z < 0.  A camera with
    rotation 0 and t_z = 0 (``_PLANE_EXT``) has exactly them on its Z = 0 plane and behind it."""
    rng = np.random.default_rng(seed)
    pts = rng.normal(0, 80, (n, 3))
    k = n // 100
    pts[:k, 2] = 0.0
    pts[k:2 * k, 2] = -np.abs(pts[k:2 * k, 2]) - 1.0
    return pts


_PLANE_EXT = np.array([0.0, 0.0, 0.0, 5.0, -3.0, 0.0])


@gpu
def test_undistort_points_past_one_grid():
    rng = np.random.default_rng(21)
    n = 1_000_000
    K = np.array([[1210.0, 0.7, 633.0], [0, 1190.0, 518.0], [0, 0, 1]])
    dist = np.array([-0.21, 0.09, 1.2e-3, -8e-4, -0.02])
    uv = np.stack([rng.uniform(-50, 1330, n), rng.uniform(-50, 1074, n)], axis=1)
    uv[rng.random(n) < 0.01, 0] = np.nan
    uv[rng.random(n) < 0.01, 1] = np.nan
    uv[rng.random(n) < 0.001, 0] = np.inf
    uv[rng.random(n) < 0.001, 1] = -np.inf
    out = mcc.undistort_points(uv, K, dist)
    ref = orc.undistort_points(uv, K, dist)
    assert np.array_equal(np.isnan(out), np.isnan(ref)) and not np.isinf(ref).any() and not np.isinf(out).any()
    fin = ~np.isnan(ref)
    print(f"undistort_points, 1 M pixels: max |diff| {np.abs(out[fin] - ref[fin]).max():.3g} px")
    np.testing.assert_allclose(out[fin], ref[fin], rtol=0, atol=1e-9)


@gpu
def test_project_points_past_one_grid():
    pts = _points_with_plane_and_behind(1_000_000, 22)
    all_uvs, ext, intr, _ = make_keypoints(1, 6, seed=3)
    for e in (ext[1], _PLANE_EXT):
        for K, dist in ((intr[1][0], intr[1][1][:2]), (intr[1][0], None)):
            uv = mcc.project_points(pts, e, K, dist)
            ref = orc.project_points(pts, e, K, dist)
            worst = _projection_close(uv, ref, K)
            print(f"project_points ext={np.round(e, 2).tolist()} dist={dist is not None}: {worst:.3g}, "
                  f"{int(np.isnan(ref).any(1).sum())} NaN / {int(np.isinf(ref).any(1).sum())} inf rows")


@gpu
@pytest.mark.parametrize("C", [16, 17, 64])
def test_project_points_multi_camera_counts(C):
    """16 cameras travel by value; 17 and 64 through the device-pointer path."""
    pts = _points_with_plane_and_behind(400_000, 23)
    ext, intr = split_cams(make_scene(C, 1, sigma=0.0, seed=C).true_cams)
    ext[0] = _PLANE_EXT
    variants = [intr] + ([[(K, None) for K, _ in intr]] if C == 17 else [])
    for it in variants:
        uv = mcc.project_points_multi(pts, list(ext), it)
        assert uv.shape == (C, len(pts), 2)
        worst = max(_projection_close(uv[c], orc.project_points(pts, ext[c], K, None if d is None else d[:2]), K)
                    for c, (K, d) in enumerate(it))
        print(f"project_points_multi, {C} cameras (dist={it[0][1] is not None}): largest relative error {worst:.3g}")


@gpu
def test_project_points_multi_rejects_65_cameras():
    ext, intr = split_cams(make_scene(65, 1, sigma=0.0, seed=1).true_cams)
    with pytest.raises(mcc._native.McbaError, match=re.escape("1 <= n_cameras <= 64")):
        mcc.project_points_multi(np.zeros((4, 3)), list(ext), intr)


@gpu
def test_embed_calib_objpoints_past_one_grid():
    """50,000 frames x 35 corners = 1.75 M points, more than one grid-stride round."""
    rng = np.random.default_rng(24)
    F = 50_000
    obj = make_scene(1, 1).objpoints
    poses = np.concatenate([rng.normal(0, 0.6, (F, 3)), rng.normal(0, 60, (F, 3))], axis=1)
    out = mcc.embed_calib_objpoints(obj, poses)
    ref = orc.embed_calib_objpoints(obj, poses)
    # |R q + t|'s rounding is relative to |q| + |t| (each row of R has unit norm)
    scale = np.linalg.norm(obj, axis=1)[None, :, None] + np.abs(poses[:, None, 3:])
    err = (np.abs(out - ref) / scale).max()
    print(f"embed_calib_objpoints, {F} x {len(obj)}: largest relative error {err:.3g}")
    assert err <= 1e-12


# ------------------------------------------------------------------ 6. initialisation and frame selection
@gpu
@pytest.mark.parametrize("C", [8, 9, 16, 17, 32])
def test_consensus_poses_camera_counts(C):
    """consensus_poses_kernel<8> / <16> / <32>, frames seen by no camera, by one and by an even number."""
    F = 20_000
    poses, ext, _ = make_camera_poses(C, F, p_missing=0.3, seed=C)
    rng = np.random.default_rng(C)
    poses[:, :10] = np.nan                                             # no camera
    for f in range(10, 40):                                            # one camera
        poses[np.arange(C) != f % C, f] = np.nan
    for f in range(40, 100):                                           # exactly two, four or six cameras
        keep = rng.choice(C, 2 * (1 + f % 3), replace=False)
        poses[np.setdiff1d(np.arange(C), keep), f] = np.nan
    seen = (~np.isnan(poses).any(2)).sum(0)
    assert {0, 1, 2, 4, 6} <= set(seen.tolist())
    cons = mcc.consensus_calib_poses(poses, ext)
    ref = orc.consensus_calib_poses(poses, ext)
    assert np.array_equal(np.isnan(cons), np.isnan(ref)) and np.isnan(cons[:10]).all()
    fin = ~np.isnan(ref)
    print(f"consensus_calib_poses, {C} cameras: max |diff| {np.abs(cons[fin] - ref[fin]).max():.3g}")
    np.testing.assert_allclose(cons[fin], ref[fin], rtol=0, atol=1e-9)


@gpu
def test_consensus_poses_rejects_33_cameras():
    poses, ext, _ = make_camera_poses(33, 10, seed=1)
    with pytest.raises(mcc._native.McbaError, match="at most 32 cameras"):
        mcc.consensus_calib_poses(poses, ext)


@gpu
def test_estimate_all_extrinsics_32_cameras():
    poses, ext_true, _ = make_camera_poses(32, 20_000, p_missing=0.3, seed=32)
    ext, tree = mcc.estimate_all_extrinsics(poses, root=0)
    ext_o, tree_o = orc.estimate_all_extrinsics(poses, root=0)
    assert tree == [tuple(int(v) for v in e) for e in tree_o]
    print(f"estimate_all_extrinsics, 32 cameras: max |diff| {np.abs(ext - ext_o).max():.3g}")
    np.testing.assert_allclose(ext, ext_o, rtol=0, atol=1e-9)


def _frame_worst(uvs, ext, intr, obj, poses):
    """Per-frame worst mean error of ``orc.select_frames`` (its lines restated), NaN where not eligible."""
    use = np.nonzero((~np.isnan(uvs).any((-1, -2))).sum(0) > 1)[0]
    err = np.linalg.norm(uvs[:, use] - orc.predict_calib_uvs(ext, intr, obj, poses[use]), axis=-1)
    worst = np.full(uvs.shape[1], np.nan)
    with np.errstate(invalid="ignore"), np.testing.suppress_warnings() as sup:
        sup.filter(RuntimeWarning)
        worst[use] = np.nanmax(np.nanmean(err, axis=-1), axis=0)
    return worst


def _select_frames_scene(C, F, seed):
    sc = make_scene(C, F, sigma=0.3, p_missing_view=0.2, seed=seed)
    uvs = sc.uvs.copy()
    rng = np.random.default_rng(seed + 1)
    bad = rng.choice(F, F // 100, replace=False)
    uvs[:, bad] += rng.normal(0, 40.0, uvs[:, bad].shape)              # gross outlier frames
    _, ext, intr, obj, poses = sc.init_args()
    return uvs, ext, intr, obj, poses


@gpu
@pytest.mark.parametrize("shape,path", [((6, 50_000), "device"), ((6, 50_000), "sharded"), ((32, 2_000), "device")])
def test_select_frames_at_scale(shape, path, capsys):
    """The exact nanmedian threshold (radix sort; both parities of the finite count) and the frame
    mask at configs[2] (6 x 50,000 x 35, seed 0 like the benchmark) and at 32 cameras."""
    from multicam_calibration_b200 import bundle_adjustment as ba
    C, F = shape
    uvs, ext, intr, obj, poses = _select_frames_scene(C, F, 0 if C == 6 else 5)
    parities = set()
    for flip in (False, True):
        if flip:                                   # one corner fewer in a frame that stays eligible
            complete = ~np.isnan(uvs).any((-1, -2))
            f = int(np.nonzero(complete[0] & (complete.sum(0) >= 3))[0][0])
            uvs = uvs.copy()
            uvs[0, f, 0] = np.nan
        eligible = (~np.isnan(uvs).any((-1, -2))).sum(0) > 1
        parities.add(int((~np.isnan(uvs[:, eligible]).any(-1)).sum()) % 2)
        worst = _frame_worst(uvs, ext, intr, obj, poses)
        given_thr = float(np.nanmedian(worst)) * 1.37 if not flip else given_thr
        for given in (None, given_thr):
            use_o, thr_o = orc.select_frames(uvs, ext, intr, obj, poses, n_frames=None, outlier_threshold=given,
                                             verbose=False)
            if path == "device":
                use = mcc.select_frames(uvs, ext, intr, obj, poses, n_frames=None, outlier_threshold=given)
            else:
                use, _, _ = ba._select_frames_sharded(uvs, ext, intr, obj, poses, None, given)
            printed = float(capsys.readouterr().out.strip().splitlines()[-1].split()[-1])
            assert printed == pytest.approx(float(thr_o), rel=1e-12)
            edge = np.nonzero(np.abs(worst - thr_o) <= 1e-12 * thr_o)[0]
            differ = np.setxor1d(use, use_o)
            with capsys.disabled():
                print(f"select_frames {C} x {F} ({path}, threshold {'given' if given else 'auto'}, "
                      f"parity flipped {flip}): threshold {printed!r}, {len(use)} kept, {len(differ)} differ, "
                      f"{len(edge)} frames within 1e-12 of the threshold")
            assert np.all(np.isin(differ, edge)), differ
    assert parities == {0, 1}


# ------------------------------------------------------------------ 7. sharpness of the triangulation checks (CPU)
def test_baseline_rig_takes_the_jacobi_fallback():
    """The 0.5 mm baseline rig exercises smallest_right_singular_vector: a changed exit test of
    null_vector_qr shows up here as lost coverage."""
    all_uvs, ext, intr = pr.pair_rig("baseline")
    und = oracle_undistorted(all_uvs, intr)
    Ps = pr.projection_matrices(ext, intr)
    frac = 1.0 - pr.qr_settles(pr.dlt(und[0], und[1], Ps[0], Ps[1])).mean()
    print(f"rig baseline: Jacobi fallback on {frac:.1%} of the pairs")
    assert frac >= 0.30
    all_uvs, ext, intr = pr.pair_rig("ring")
    und = oracle_undistorted(all_uvs, intr)
    Ps = pr.projection_matrices(ext, intr)
    assert pr.qr_settles(pr.dlt(und[0], und[1], Ps[0], Ps[1])).mean() == 1.0


@pytest.mark.parametrize("kind", ["ring", "baseline", "exact"])
def test_pair_bounds_accept_the_oracle(kind):
    all_uvs, ext, intr = pr.pair_rig(kind)
    res, fwd = pair_check(all_uvs, ext, intr, orc.triangulate(all_uvs, list(ext), intr),
                          oracle_undistorted(all_uvs, intr))
    assert res.max() <= 1.0 and fwd.max() <= 1.0


WRONG = {"4 undistortion iterations": dict(n_iter=4), "lower middle value": dict(median="lower"),
         "second-smallest singular vector": dict(vector=-2)}


@pytest.mark.parametrize("wrong", sorted(WRONG))
def test_triangulation_checks_reject_wrong_kernels(wrong):
    """Each wrong kernel fails the configs[4] median check, and (where it changes a 2-camera
    result) the pair bounds of every rig it changes."""
    all_uvs, ext, intr, _ = make_keypoints(20_000, 6, sigma=0.3, p_missing=0.2, seed=0)
    ref = orc.triangulate(all_uvs, list(ext), intr)
    out = pr.triangulate_variant(all_uvs, ext, intr, **WRONG[wrong])
    rep = median_check(out, ref, oracle_undistorted(all_uvs, intr), ext, intr)
    print(f"{wrong}: configs[4] check {rep['ok']}, max |diff| {rep['max_diff']:.3g}, "
          f"diff/bound {rep['worst_ratio']:.3g}")
    assert not rep["ok"]
    assert median_check(ref, ref, oracle_undistorted(all_uvs, intr), ext, intr)["ok"]
    if wrong == "lower middle value":
        return                                                        # one pair: nothing to take the median of
    for kind in ("ring", "baseline", "exact"):
        uvs2, ext2, intr2 = pr.pair_rig(kind)
        with np.errstate(all="ignore"):
            res, fwd = pair_check(uvs2, ext2, intr2, pr.triangulate_variant(uvs2, ext2, intr2, **WRONG[wrong]),
                                  oracle_undistorted(uvs2, intr2))
        print(f"{wrong}, rig {kind}: residual {np.nanmax(res):.3g}, forward {np.nanmax(fwd):.3g}")
        assert max(np.nanmax(res), np.nanmax(fwd)) > 1.0
