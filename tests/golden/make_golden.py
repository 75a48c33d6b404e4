"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Run in the build container only (needs ``/root/reference``):

    python tests/golden/make_golden.py                 # regenerate every fixture
    python tests/golden/make_golden.py --only ba_cfg1  # one fixture
    python tests/golden/make_golden.py --check         # regenerate in memory and assert that every
                                                       # array equals the committed file (wall-clock
                                                       # fields excepted)

The reference package ``__init__`` star-imports modules whose dependencies
(vidio, h5py, matplotlib) are not installed, so its two hot-path modules are
imported through a stub package (SURVEY.md 8c).  Besides writing the ``.npz``
fixtures the script asserts that ``oracle/np_oracle.py`` reproduces the
reference on every fixture, which is what pins the oracle.
"""
import importlib
import io
import os
import sys
import types
import warnings
from contextlib import redirect_stdout

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

REF = "/root/reference/multicam_calibration"


def load_reference():
    pkg = types.ModuleType("multicam_calibration")
    pkg.__path__ = [REF]
    sys.modules["multicam_calibration"] = pkg
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        geo = importlib.import_module("multicam_calibration.geometry")
        ba = importlib.import_module("multicam_calibration.bundle_adjustment")
    return geo, ba


def close(a, b, tol, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    nan = np.isnan(a)
    assert (nan == np.isnan(b)).all(), what + ": NaN pattern"
    scale = max(1.0, float(np.nanmax(np.abs(a))) if (~nan).any() else 1.0)
    err = float(np.max(np.abs(a[~nan] - b[~nan]))) / scale if (~nan).any() else 0.0
    print(f"  oracle vs reference  {what:42s} max rel-to-scale err = {err:.3e}")
    assert err <= tol, (what, err)


def _versions():
    import cv2
    import scipy
    return np.array([np.__version__, scipy.__version__, cv2.__version__])


def gen_geometry(geo, ba):
    import cv2
    from oracle import np_oracle as orc
    versions = _versions()
    rng = np.random.default_rng(1234)
    r = rng.normal(0, 1.0, (40, 3))
    r[0] = 0.0                      # theta == 0 branch (geometry.py:30)
    r[1] = [1e-9, 0, 0]
    t6 = np.concatenate([r, rng.normal(0, 50, (40, 3))], axis=1)
    pts = rng.normal(0, 80, (40, 7, 3)) + [0, 0, 600]
    K = np.array([[1210.0, 0.7, 633.0], [0, 1190.0, 518.0], [0, 0, 1]])   # skew kept by project_points
    dist = np.array([-0.11, 0.06, 0.001, -0.002, 0.01])
    ext = np.array([0.3, -0.2, 0.1, 5.0, -3.0, 20.0])
    g = dict(
        versions=versions,
        r=r, R=geo.rodrigues(r), r_back=geo.rodrigues_inv(geo.rodrigues(r)),
        t6=t6, T=geo.get_transformation_matrix(t6),
        t6_back=geo.get_transformation_vector(geo.get_transformation_matrix(t6)),
        pts=pts, ext=ext, K=K, dist=dist,
        pts_rigid_vec=geo.apply_rigid_transform(ext, pts),
        pts_rigid_mat=geo.apply_rigid_transform(geo.get_transformation_matrix(ext), pts),
        uv_dist=geo.project_points(pts, ext, K, dist),
        uv_nodist=geo.project_points(pts, ext, K, None),
        P=geo.get_projection_matrix(ext, (K, dist)),
    )
    uv_in = g["uv_dist"].copy()
    uv_in[3, 2, 0] = np.nan
    uv_in[5] = np.nan
    g["uv_in"] = uv_in
    g["uv_undist"] = geo.undistort_points(uv_in, K, dist)
    close(g["R"], orc.rodrigues(r), 1e-15, "rodrigues")
    close(g["r_back"], orc.rodrigues_inv(orc.rodrigues(r)), 1e-12, "rodrigues_inv")
    close(g["T"], orc.transformation_matrix(t6), 1e-15, "get_transformation_matrix")
    close(g["pts_rigid_vec"], orc.apply_rigid_transform(ext, pts), 1e-15, "apply_rigid_transform")
    close(g["uv_dist"], orc.project_points(pts, ext, K, dist), 1e-14, "project_points(dist)")
    close(g["uv_nodist"], orc.project_points(pts, ext, K, None), 1e-14, "project_points(None)")
    close(g["P"], orc.projection_matrix(ext, (K, dist)), 1e-15, "get_projection_matrix")
    close(g["uv_undist"], orc.undistort_points(uv_in, K, dist), 1e-11, "undistort_points (cv2, 5 it)")
    # independent pins: OpenCV's own Rodrigues / projectPoints
    for i in range(5):
        assert np.abs(cv2.Rodrigues(r[i + 2])[0] - g["R"][i + 2]).max() < 1e-14
    K0 = K.copy(); K0[0, 1] = 0
    uv_cv = cv2.projectPoints(pts.reshape(-1, 3), ext[:3], ext[3:], K0,
                              np.r_[dist[:2], 0, 0, 0])[0].reshape(40, 7, 2)
    close(uv_cv, orc.project_points(pts, ext, K0, dist), 1e-12, "cv2.projectPoints(k1,k2)")
    return g


def gen_triangulate(geo, ba):
    from oracle import np_oracle as orc
    from multicam_calibration_b200.synthetic import make_keypoints
    versions = _versions()
    all_uvs, exts, intr, pts3 = make_keypoints(300, 4, sigma=0.3, p_missing=0.3, seed=3)
    intr = [(Kc, np.r_[dc[:2], 0.0005, -0.0003, 0.002]) for Kc, dc in intr]   # full 5-coef model
    all_uvs[0][:4] = np.nan; all_uvs[1][:4] = np.nan; all_uvs[2][:4] = np.nan   # <2 views -> NaN rows
    all_uvs[1][7, 0] = np.nan                                                    # half-NaN observation
    with redirect_stdout(io.StringIO()):
        tri = geo.triangulate(all_uvs, list(exts), intr)
    close(tri, orc.triangulate(all_uvs, list(exts), intr), 1e-9, "triangulate")
    return dict(versions=versions, all_uvs=np.stack(all_uvs), extrinsics=exts,
                Ks=np.stack([k for k, _ in intr]), dists=np.stack([d for _, d in intr]),
                points=tri, truth=pts3)


def gen_ba_small(geo, ba):
    """Residuals, predictions and the reference's finite-difference Jacobians on a small scene."""
    from scipy.optimize._numdiff import approx_derivative
    from oracle import np_oracle as orc
    from multicam_calibration_b200.synthetic import make_scene
    versions = _versions()
    sc = make_scene(4, 12, sigma=0.3, p_missing_view=0.2, p_missing_corner=0.1, seed=7)
    uvs = sc.uvs.copy()
    uvs[0, 0, 0, 0] = np.nan          # u missing, v present: element-wise mask (bundle_adjustment.py:97)
    uvs[2, 5, 3, 1] = np.nan
    x0 = sc.x0()
    res = ba.residuals(x0, uvs, sc.objpoints)
    A = ba.bundle_adjustment_sparsity(uvs)
    J2 = approx_derivative(ba.residuals, x0, method="2-point", sparsity=A,
                           args=(uvs, sc.objpoints)).tocsr()
    J3 = approx_derivative(ba.residuals, x0, method="3-point", sparsity=A,
                           args=(uvs, sc.objpoints)).tocsr()
    ext0, intr0, poses0 = ba.deserialize_params(x0, 4)
    pred = ba.predict_calib_uvs(ext0, intr0, sc.objpoints, poses0)
    world = ba.embed_calib_objpoints(sc.objpoints, poses0)
    close(res, orc.residuals(x0, uvs, sc.objpoints), 1e-13, "residuals")
    close(pred, orc.predict_calib_uvs(ext0, intr0, sc.objpoints, poses0), 1e-14, "predict_calib_uvs")
    close(world, orc.embed_calib_objpoints(sc.objpoints, poses0), 1e-15, "embed_calib_objpoints")
    close(x0, orc.serialize_params(ext0, intr0, poses0), 0, "serialize(deserialize(x))")
    assert (A.toarray() == orc.sparsity_pattern(uvs).toarray()).all()
    Ja = orc.dense_residual_jacobian(x0, uvs, sc.objpoints)
    e3 = np.linalg.norm(Ja - J3.toarray()) / np.linalg.norm(Ja)
    e2 = np.linalg.norm(Ja - J2.toarray()) / np.linalg.norm(Ja)
    print(f"  analytic J vs reference FD: 3-point {e3:.2e}, 2-point {e2:.2e} (Frobenius-relative)")
    assert e3 < 1e-8 and e2 < 1e-5
    return dict(versions=versions, uvs=uvs, objpoints=sc.objpoints, x0=x0, residuals=res, predicted=pred,
                world=world, J2_data=J2.data, J2_indices=J2.indices, J2_indptr=J2.indptr,
                J3_data=J3.data, J3_indices=J3.indices, J3_indptr=J3.indptr,
                A_indices=A.tocsr().indices, A_indptr=A.tocsr().indptr)


def gen_frontend(geo, ba):
    """Frame selection of bundle_adjust (bundle_adjustment.py:265-296) incl. the RNG sub-sampling."""
    from oracle import np_oracle as orc
    from multicam_calibration_b200.synthetic import make_scene
    versions = _versions()
    sc = make_scene(5, 60, sigma=0.3, p_missing_view=0.45, p_missing_corner=0.02, seed=11)
    uvs = sc.uvs.copy()
    uvs[:, 17] += 40.0                 # gross outlier frame -> excluded by the 5x median rule
    poses_nan = sc.init_poses.copy()
    args = (uvs, *sc.init_args()[1:4], poses_nan)
    out = {}
    for tag, nf in (("all", None), ("sub", 20)):
        np.random.seed(0)
        buf = io.StringIO()
        with redirect_stdout(buf):
            e, i, p, use, result = ba.bundle_adjust(*args, n_frames=nf, max_nfev=2, verbose=0)
        out[f"use_{tag}"] = use
        out[f"msg_{tag}"] = np.array(buf.getvalue())
        out[f"x_{tag}"] = result.x
        np.random.seed(0)
        with redirect_stdout(io.StringIO()):
            use_o, thr = orc.select_frames(*args, n_frames=nf)
        assert (use_o == use).all(), tag
    return dict(versions=versions, uvs=uvs, objpoints=sc.objpoints, init_cams=sc.init_cams,
                init_poses=poses_nan, **out)


def gen_convergence(geo, ba):
    """6 cameras x 40 frames to convergence: the reference's default run and a tight scipy solution."""
    from oracle import np_oracle as orc
    from multicam_calibration_b200.synthetic import make_scene
    versions = _versions()
    sc = make_scene(6, 40, sigma=0.3, p_missing_view=0.15, seed=5)
    args = sc.init_args()
    np.random.seed(0)
    with redirect_stdout(io.StringIO()):
        e_d, i_d, p_d, use_d, r_d = ba.bundle_adjust(*args, n_frames=None, verbose=0)
    # tight oracle: the reference residual function, scipy trf with an exact dense
    # solve and the analytic Jacobian so stationarity is not FD-limited (SURVEY H2)
    from scipy.optimize import least_squares
    uv_used = sc.uvs[:, use_d]
    x0 = ba.serialize_params(args[1], args[2], args[4][use_d])
    r_t = least_squares(ba.residuals, x0, jac=lambda x, u, o: orc.analytic_jac_for_scipy(x, u, o).toarray(),
                        args=(uv_used, sc.objpoints), method="trf", loss="soft_l1", x_scale="jac",
                        tr_solver="exact", ftol=1e-15, xtol=1e-15, gtol=1e-15, max_nfev=400, verbose=0)
    rms = lambda x: float(np.sqrt(np.mean(ba.residuals(x, uv_used, sc.objpoints) ** 2)))
    print(f"  convergence: default stop cost {r_d.cost:.9f} rms {rms(r_d.x):.9f} nfev {r_d.nfev} | "
          f"tight cost {r_t.cost:.12f} rms {rms(r_t.x):.12f} nfev {r_t.nfev} opt {r_t.optimality:.2e}")
    # scipy's exact-solve trf stops at optimality ~1e-3 (its xtol test fires on the gauge drift); a few
    # Gauss-Newton steps on the same (reference) residual function take the gradient to rounding level
    # so that k1, k2 of x_tight are good to 1e-8 relative, and the two points are checked against each other
    x_p, cost_p, g_p = orc.sparse_gauss_newton_polish(r_t.x, uv_used, sc.objpoints, fun=ba.residuals)
    ia, ib = r_t.x[:72].reshape(6, 12), x_p[:72].reshape(6, 12)
    Ta, Tb = orc.relative_camera_transforms(ia[:, 6:]), orc.relative_camera_transforms(ib[:, 6:])
    d_intr = float(np.abs(ia[:, :6] / ib[:, :6] - 1).max())
    d_T = float(np.abs(Ta - Tb).max() / np.abs(Tb).max())
    print(f"  convergence: polished cost {cost_p:.12f} rms {rms(x_p):.12f} |g|inf {g_p:.2e}; scipy tight vs polished: "
          f"intrinsics {d_intr:.1e} rel, transforms {d_T:.1e} rel")
    assert g_p < 1e-6 and d_intr < 1e-5 and d_T < 1e-6 and abs(rms(x_p) - rms(r_t.x)) < 1e-7
    return dict(versions=versions, uvs=sc.uvs, objpoints=sc.objpoints, init_cams=sc.init_cams,
                init_poses=sc.init_poses, use_frames=use_d,
                x_default=r_d.x, cost_default=r_d.cost, rms_default=rms(r_d.x),
                nfev_default=r_d.nfev, status_default=r_d.status,
                x_scipy_tight=r_t.x, cost_scipy_tight=r_t.cost, optimality_scipy_tight=r_t.optimality,
                x_tight=x_p, cost_tight=cost_p, rms_tight=rms(x_p), optimality_tight=g_p)


def gen_ba_cfg1(geo, ba):
    """BASELINE configs[0] (6 cameras x 500 frames x 35 corners, sigma = 0.3 px, every detection
    present: 105 000 observations): the UNMODIFIED reference ``bundle_adjust`` with its defaults
    (bundle_adjustment.py:195-327: trf + LSMR + 2-point finite differences, ftol = 1e-4, soft_l1),
    timed here, and the tight minimum of the same objective.  A dense Jacobian (210 000 x 3 072)
    does not fit scipy's ``tr_solver='exact'`` at this size, so the tight point is reached from the
    reference's own result by Gauss-Newton on the reference residual function with the analytic
    sparse Jacobian and a sparse direct solve (``oracle.sparse_gauss_newton_polish``); the stored
    ``optimality_tight`` (||J^T rho' f||_inf at x_tight, evaluated with the reference residuals) is
    its certificate."""
    import hashlib
    import json
    import time
    from oracle import np_oracle as orc
    from multicam_calibration_b200.synthetic import make_scene
    scene = dict(n_cameras=6, n_frames=500, sigma=0.3, seed=0)
    sc = make_scene(**scene)
    args = sc.init_args()
    np.random.seed(0)
    buf = io.StringIO()
    t0 = time.perf_counter()
    with redirect_stdout(buf):
        e_d, i_d, p_d, use_d, r_d = ba.bundle_adjust(*args, n_frames=None, verbose=0)
    wall = time.perf_counter() - t0
    uv_used = sc.uvs[:, use_d]
    rms = lambda x: float(np.sqrt(np.mean(ba.residuals(x, uv_used, sc.objpoints) ** 2)))
    trace = []
    x_t, cost_t, g_t = orc.sparse_gauss_newton_polish(r_d.x, uv_used, sc.objpoints, fun=ba.residuals, trace=trace)
    print(f"  cfg1: reference default {wall:.1f} s, cost {r_d.cost:.9f} rms {rms(r_d.x):.9f} nfev {r_d.nfev} "
          f"njev {r_d.njev} status {r_d.status} | tight cost {cost_t:.12f} rms {rms(x_t):.12f} |g|inf {g_t:.2e} "
          f"after {len(trace)} Gauss-Newton steps")
    assert g_t < 1e-6
    x0 = ba.serialize_params(args[1], args[2], args[4][use_d])
    # the 1.7 MB observation array is not stored: tests/conftest.py regenerates it from `scene` and
    # checks it against `uvs_sha256`
    return dict(versions=_versions(), scene=np.array(json.dumps(scene)),
                uvs_sha256=np.array(hashlib.sha256(np.ascontiguousarray(sc.uvs).tobytes()).hexdigest()),
                objpoints=sc.objpoints, init_cams=sc.init_cams,
                init_poses=sc.init_poses, use_frames=use_d, x0=x0, msg_default=np.array(buf.getvalue()),
                x_default=r_d.x, cost_default=r_d.cost, rms_default=rms(r_d.x), nfev_default=r_d.nfev,
                njev_default=r_d.njev, status_default=r_d.status, optimality_default=r_d.optimality,
                wall_s_default=wall, wall_host=np.array(f"{os.cpu_count()} cores; scipy trf is single-threaded"),
                x_tight=x_t, cost_tight=cost_t, rms_tight=rms(x_t), optimality_tight=g_t)


FIXTURES = {"geometry": gen_geometry, "triangulate": gen_triangulate, "ba_small": gen_ba_small,
            "frontend": gen_frontend, "convergence": gen_convergence, "ba_cfg1": gen_ba_cfg1}
# wall-clock and host descriptions differ between runs: excluded from --check
VOLATILE = ("wall_",)


def check_fixture(name, fresh):
    """Regenerated arrays against the committed file: inputs (everything the scene generator makes)
    must be bit-identical; outputs of the reference agree to rounding (BLAS summation order)."""
    path = os.path.join(HERE, name + ".npz")
    old = np.load(path, allow_pickle=False)
    keys = sorted(k for k in fresh if not k.startswith(VOLATILE))
    assert keys == sorted(k for k in old.files if not k.startswith(VOLATILE)), (name, keys, old.files)
    worst = 0.0
    for k in keys:
        a, b = np.asarray(fresh[k]), old[k]
        assert a.shape == b.shape and a.dtype.kind == b.dtype.kind, (name, k, a.shape, b.shape)
        if a.dtype.kind in "US" or a.dtype.kind in "iub":
            assert np.array_equal(a, b), (name, k)
            continue
        assert np.array_equal(np.isnan(a), np.isnan(b)), (name, k)
        if np.array_equal(a, b, equal_nan=True):
            continue
        ok = ~np.isnan(a)
        err = float(np.abs(a[ok] - b[ok]).max() / max(1.0, np.abs(b[ok]).max()))
        worst = max(worst, err)
        assert err < 1e-9, (name, k, err)
    print(f"  check {name}: {len(keys)} arrays equal to the committed fixture (worst rounding difference {worst:.1e})")


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--only", action="append", choices=sorted(FIXTURES))
    a = ap.parse_args()
    geo, ba = load_reference()
    for name in (a.only or list(FIXTURES)):
        print(name)
        fresh = FIXTURES[name](geo, ba)
        if a.check:
            check_fixture(name, fresh)
        else:
            np.savez_compressed(os.path.join(HERE, name + ".npz"), **fresh)
    print("golden fixtures", "checked against" if a.check else "written to", HERE)


if __name__ == "__main__":
    main()
