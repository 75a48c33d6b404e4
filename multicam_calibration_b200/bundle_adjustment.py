"""Drop-in for ``multicam_calibration.bundle_adjustment`` (reference
bundle_adjustment.py:10-327) on the B200 engine.

Same function names, argument order, parameter-vector layout, observation
arrays and return values.  ``bundle_adjust`` replaces the reference's
``scipy.optimize.least_squares(method='trf', jac_sparsity=...)`` call with a
device Levenberg-Marquardt loop over fused residual + analytic-Jacobian +
Schur kernels (see DESIGN.md); the finite-difference sparsity pattern is never
built on that path.
"""
import ctypes

import numpy as np

from . import _native
from ._native import check
from .engine import BAProblem
from .geometry import project_points_multi

na = np.newaxis


def embed_calib_objpoints(calib_objpoints, calib_poses, _keep_on_device=False):
    """(N,3), (F,6) -> (F,N,3) world points (bundle_adjustment.py:10-30)."""
    torch = _native.require_cuda()
    lib = _native.load()
    dev = torch.cuda.current_device()
    obj = np.ascontiguousarray(calib_objpoints, dtype=np.float64)
    poses = np.ascontiguousarray(calib_poses, dtype=np.float64)
    d_obj = _native.to_device(obj, dev)
    d_pose = _native.to_device(poses.reshape(-1, 6), dev)
    F, N = d_pose.shape[0], obj.shape[0]
    d_out = torch.empty((F, N, 3), dtype=torch.float64, device=d_obj.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.mcba_embed_points(dev, stream, ctypes.c_void_p(d_pose.data_ptr()), F,
                                ctypes.c_void_p(d_obj.data_ptr()), N, ctypes.c_void_p(d_out.data_ptr())))
    if _keep_on_device:
        return d_out
    return _native.to_host(d_out).reshape(*poses.shape[:-1], N, 3)


def predict_calib_uvs(all_extrinsics, all_intrinsics, calib_objpoints, calib_poses):
    """(C,F,N,2) predicted corner positions (bundle_adjustment.py:33-63): the world points stay
    on the device and are projected into every camera in one pass."""
    d_world = embed_calib_objpoints(calib_objpoints, calib_poses, _keep_on_device=True)
    F, N = d_world.shape[0], d_world.shape[1]
    return project_points_multi(None, all_extrinsics, all_intrinsics, _device_points=(d_world.reshape(-1, 3), (F, N)))


def serialize_params(all_extrinsics, all_intrinsics, calib_poses):
    """Flat parameter vector, 12 per camera then 6 per frame (bundle_adjustment.py:128-157)."""
    blocks = []
    for ext, (K, dist) in zip(all_extrinsics, all_intrinsics):
        K = np.asarray(K)
        blocks.append(np.concatenate([[K[0, 0], K[1, 1], K[0, 2], K[1, 2]],
                                      np.asarray(dist)[:2], np.asarray(ext)]))
    blocks.append(np.asarray(calib_poses).ravel())
    return np.concatenate(blocks)


def deserialize_params(x, n_cameras):
    """Inverse of :func:`serialize_params` (bundle_adjustment.py:160-192)."""
    x = np.asarray(x)
    cams = x[:12 * n_cameras].reshape(n_cameras, 12)
    all_intrinsics = []
    for p in cams:
        K = np.eye(3)
        K[[0, 1, 0, 1], [0, 1, 2, 2]] = p[:4]
        all_intrinsics.append((K, np.pad(p[4:6], (0, 3))))
    return np.array(cams[:, 6:]), all_intrinsics, x[12 * n_cameras:].reshape((-1, 6))


_problems = {}


def _problem_for(all_calib_uvs, calib_objpoints):
    """One cached device allocation (the workspaces of the last problem shape, ~0.7 GB at
    BASELINE configs[2]); observations are re-uploaded on every call (the caller's array may
    have changed).  ``all_calib_uvs``: numpy array or float64 CUDA tensor."""
    torch = _native.require_cuda()
    uvs = all_calib_uvs if hasattr(all_calib_uvs, "is_cuda") else np.asarray(all_calib_uvs)
    key = (tuple(uvs.shape), torch.cuda.current_device())
    prob = _problems.get(key)
    if prob is None:
        for old in _problems.values():
            old.close()
        _problems.clear()
        prob = BAProblem(uvs, calib_objpoints)
        _problems[key] = prob
    else:
        prob.set_observations(uvs, calib_objpoints)
    return prob


def release_device_memory():
    """Free the cached device problem (workspaces kept between calls of the same shape) and, in a
    multi-GPU run, the cached sharded problem with its communicator (call on every rank)."""
    for old in _problems.values():
        old.close()
    _problems.clear()
    from . import distributed
    distributed.release_sharded_problem()


def residuals(params, all_calib_uvs, calib_objpoints):
    """observed - predicted for every finite observation scalar, C order
    (bundle_adjustment.py:66-98)."""
    return _problem_for(all_calib_uvs, calib_objpoints).residuals(params)


def bundle_adjustment_sparsity(all_calib_uvs):
    """Jacobian sparsity pattern (bundle_adjustment.py:101-125).  Kept for API
    parity only -- the engine uses analytic blocks and never builds it."""
    from scipy.sparse import csr_matrix
    C, F, N, _ = all_calib_uvs.shape
    mask = ~np.isnan(all_calib_uvs)
    cam = np.broadcast_to(np.arange(C)[:, na, na, na], mask.shape)[mask]
    frm = np.broadcast_to(np.arange(F)[na, :, na, na], mask.shape)[mask]
    cols = np.concatenate([cam[:, na] * 12 + np.arange(12), C * 12 + frm[:, na] * 6 + np.arange(6)], axis=1)
    m = cam.size
    A = csr_matrix((np.ones(m * 18, dtype=int), cols.ravel(), np.arange(m + 1) * 18),
                   shape=(m, C * 12 + F * 6))
    return A.tolil()


def _select_frames_device(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints, calib_poses,
                          n_frames, outlier_threshold):
    """Device front end: returns ``(use_frames, d_uvs)`` with the full observation array left on
    the GPU so that the kept frames can be gathered there."""
    torch = _native.require_cuda()
    lib = _native.load()
    dev = torch.cuda.current_device()
    uvs = np.ascontiguousarray(all_calib_uvs, dtype=np.float64)
    C, F, N, _ = uvs.shape
    x_all = serialize_params(all_extrinsics, all_intrinsics, calib_poses)
    d_uvs = _native.to_device(uvs, dev)
    d_x = _native.to_device(x_all, dev)
    d_obj = _native.to_device(calib_objpoints, dev)
    d_use = torch.empty(F, dtype=torch.uint8, device=f"cuda:{dev}")
    stats = (ctypes.c_double * 4)()
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    thr = float("nan") if outlier_threshold is None else float(outlier_threshold)
    check(lib.mcba_select_frames(dev, stream, ctypes.c_void_p(d_uvs.data_ptr()), C, F, N,
                                 ctypes.c_void_p(d_obj.data_ptr()), ctypes.c_void_p(d_x.data_ptr()), thr,
                                 ctypes.c_void_p(d_use.data_ptr()), stats))
    use_frames = torch.nonzero(d_use).ravel().cpu().numpy()
    threshold = outlier_threshold if outlier_threshold is not None else stats[0]
    print(f"Excluding {int(stats[2])} out of {len(use_frames)} frames "
          f"based on an outlier threshold of {threshold}")
    if not (n_frames is None or n_frames > len(use_frames)):
        use_frames = np.random.choice(use_frames, n_frames, replace=False)
    return use_frames, d_uvs


def _select_frames_sharded(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints, calib_poses,
                           n_frames, outlier_threshold):
    """The same front end with the frames sharded over the ranks of ``torch.distributed``'s default
    group (every rank is called with the same, full host arrays, like the reference's call under
    torchrun).  Rank r uploads and scans only its contiguous range of ALL frames; the nanmedian of
    :281-282 is found exactly over all ranks by radix selection (256-bin histograms are the only
    thing summed across ranks); rank 0 draws the random sub-sample of :293-296 and broadcasts it, so
    every rank sees the same ``use_frames`` whatever its RNG state.

    Returns ``(use_frames, d_uvs_local, frames_per_rank)``: the kept frames (global indices, identical
    on all ranks), THIS rank's share of their observations on its device -- the kept frames of its own
    range when all are used (nothing is re-uploaded), a balanced slice of the drawn sample otherwise --
    and how many frames every rank holds."""
    from . import distributed
    torch = _native.require_cuda()
    lib = _native.load()
    W, r = distributed.world_size(), distributed.rank()
    dev = distributed.local_device()
    torch.cuda.set_device(dev)
    uvs = np.asarray(all_calib_uvs, dtype=np.float64)
    C, F, N, _ = uvs.shape
    if F < W:
        raise ValueError(f"{F} frames cannot be sharded over {W} ranks")
    a, b = distributed.shard_bounds(F, W, r)
    Fl = b - a
    device = f"cuda:{dev}"
    d_uvs = torch.empty((C, Fl, N, 2), dtype=torch.float64, device=device)
    for c in range(C):                                   # uvs[c, a:b] is contiguous: no host-side copy of the shard
        _native.upload_into(d_uvs[c], uvs[c, a:b])
    x_loc = serialize_params(all_extrinsics, all_intrinsics, np.asarray(calib_poses, dtype=np.float64)[a:b])
    d_x, d_obj = _native.to_device(x_loc, dev), _native.to_device(calib_objpoints, dev)
    d_err = torch.empty((C, Fl, N), dtype=torch.float64, device=device)
    d_mean = torch.empty((C, Fl), dtype=torch.float64, device=device)
    d_elig = torch.empty(Fl, dtype=torch.uint8, device=device)
    d_use = torch.empty(Fl, dtype=torch.uint8, device=device)
    d_hist = torch.empty(256, dtype=torch.int64, device=device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    ptr = lambda t: ctypes.c_void_p(t.data_ptr())
    counts = (ctypes.c_int64 * 2)()
    check(lib.mcba_frame_errors(dev, stream, ptr(d_uvs), C, Fl, N, ptr(d_obj), ptr(d_x), ptr(d_err), ptr(d_mean),
                                ptr(d_elig), counts))
    n_eligible, n_finite = (int(v) for v in distributed.allreduce_sum(np.array([counts[0], counts[1]], dtype=np.int64)))
    if outlier_threshold is None:
        import torch.distributed as dist
        on_device = W > 1 and dist.get_backend() == "nccl"

        def summed_histogram(prefix, prefix_bits):    # 256 counts of THIS pass, already summed over the ranks
            check(lib.mcba_key_histogram(dev, stream, ptr(d_err), d_err.numel(), ctypes.c_uint64(prefix), prefix_bits,
                                         ptr(d_hist)))
            if on_device:
                dist.all_reduce(d_hist)               # on the device: one host round trip per pass
                return d_hist.cpu().numpy()
            return distributed.allreduce_sum(d_hist.cpu().numpy())
        threshold = 5.0 * distributed.global_nanmedian(summed_histogram, n_finite, reduce=lambda a: np.asarray(a))
    else:
        threshold = outlier_threshold
    excluded = ctypes.c_int64()
    check(lib.mcba_apply_threshold(dev, stream, ptr(d_mean), ptr(d_elig), C, Fl, float(threshold), ptr(d_use),
                                   ctypes.byref(excluded)))
    use_local = torch.nonzero(d_use).ravel()
    # one exchange: every rank's kept frames (global indices; exact in float64) and its excluded count
    kept, excl = distributed.gather_concat([(use_local + a).to(torch.float64), np.array([float(excluded.value)])])
    n_excluded = int(sum(float(e.cpu()[0]) for e in excl))
    use_frames = np.concatenate([k.cpu().numpy() for k in kept]).astype(np.int64)
    if r == 0:
        print(f"Excluding {n_excluded} out of {len(use_frames)} frames "
              f"based on an outlier threshold of {threshold}")
    if n_frames is None or n_frames > len(use_frames):
        out = torch.empty((C, int(use_local.numel()), N, 2), dtype=torch.float64, device=device)
        if use_local.numel():
            check(lib.mcba_gather_frames(dev, stream, ptr(d_uvs), C, Fl, N, ptr(use_local), int(use_local.numel()), ptr(out)))
        return use_frames, out, np.array([int(k.numel()) for k in kept], dtype=np.int64)
    # random sub-sample (bundle_adjustment.py:293-296): drawn once, on rank 0, from ITS global numpy RNG
    chosen = np.random.choice(use_frames, n_frames, replace=False) if r == 0 else None
    chosen = distributed.broadcast_object(chosen)
    lo, hi = distributed.shard_bounds(len(chosen), W, r)
    mine = chosen[lo:hi]
    out = torch.empty((C, len(mine), N, 2), dtype=torch.float64, device=device)
    if len(mine):
        _native.upload_into(out, uvs[:, mine])          # a shard of the (small) sample from the caller's array
    counts = np.array([distributed.shard_bounds(len(chosen), W, q)[1] - distributed.shard_bounds(len(chosen), W, q)[0]
                       for q in range(W)], dtype=np.int64)
    return chosen, out, counts


def select_frames(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints, calib_poses,
                  n_frames=10000, outlier_threshold=None):
    """Frame eligibility, outlier rejection and sub-sampling of
    bundle_adjustment.py:265-296 (same rule, same print, same use of the global numpy RNG);
    the statistics run on the device (``mcba_select_frames``)."""
    return _select_frames_device(np.asarray(all_calib_uvs, dtype=np.float64), all_extrinsics, all_intrinsics,
                                 np.asarray(calib_objpoints, dtype=np.float64),
                                 np.asarray(calib_poses, dtype=np.float64), n_frames, outlier_threshold)[0]


def _gather_frames_device(d_uvs, use_frames):
    """``all_calib_uvs[:, use_frames]`` on the device."""
    torch = _native.require_cuda()
    lib = _native.load()
    dev = d_uvs.device.index
    C, F, N, _ = d_uvs.shape
    d_idx = torch.as_tensor(np.ascontiguousarray(use_frames, dtype=np.int64)).to(d_uvs.device)
    out = torch.empty((C, len(use_frames), N, 2), dtype=torch.float64, device=d_uvs.device)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.mcba_gather_frames(dev, stream, ctypes.c_void_p(d_uvs.data_ptr()), C, F, N,
                                 ctypes.c_void_p(d_idx.data_ptr()), len(use_frames), ctypes.c_void_p(out.data_ptr())))
    return out


def bundle_adjust(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints, calib_poses,
                  n_frames=10000, outlier_threshold=None, **opt_kwargs):
    """Bundle adjustment of all cameras and board poses (bundle_adjustment.py:195-327).

    Returns ``(adjusted_extrinsics, adjusted_intrinsics, adjusted_calib_poses,
    use_frames, result)`` exactly like the reference; ``result`` has the fields of
    ``scipy.optimize.OptimizeResult`` (``jac`` is None: the Jacobian is never
    materialised).  ``opt_kwargs`` accepts ``ftol, xtol, gtol, max_nfev, loss
    ('soft_l1' | 'linear'), f_scale, verbose``, and the engine-only ``hessian`` and
    ``fixed``: a (C, 12) bool mask in ``serialize_params`` order of camera parameters
    held at their initial values (e.g. ``fixed[:, :6] = True`` keeps the intrinsics,
    ``fixed[0, 6:] = True`` keeps camera 0 where it is and so pins the gauge, all True
    refines the board poses only); when ``torch.distributed`` is initialised with more
    than one rank the frames are sharded across ranks.
    """
    from . import distributed
    from .engine import check_fixed
    all_calib_uvs = np.asarray(all_calib_uvs, dtype=np.float64)
    calib_poses = np.asarray(calib_poses, dtype=np.float64)
    calib_objpoints = np.asarray(calib_objpoints, dtype=np.float64)
    n_cameras = all_calib_uvs.shape[0]
    check_fixed(opt_kwargs.get("fixed"), n_cameras)
    if distributed.world_size() > 1:
        # every rank uploads, scans and solves only its own frames; use_frames is rank-contiguous
        use_frames, d_local, counts = _select_frames_sharded(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints,
                                                             calib_poses, n_frames, outlier_threshold)
        lo = int(counts[:distributed.rank()].sum())
        x0_local = serialize_params(all_extrinsics, all_intrinsics, calib_poses[use_frames[lo:lo + int(d_local.shape[1])]])
        x, result = distributed.solve_sharded(d_local, calib_objpoints, x0_local, frames_per_rank=counts, **opt_kwargs)
        del d_local
    else:
        use_frames, d_uvs = _select_frames_device(all_calib_uvs, all_extrinsics, all_intrinsics, calib_objpoints,
                                                  calib_poses, n_frames, outlier_threshold)
        x0 = serialize_params(all_extrinsics, all_intrinsics, calib_poses[use_frames])
        prob = _problem_for(_gather_frames_device(d_uvs, use_frames), calib_objpoints)
        del d_uvs
        x, result = prob.solve(x0, **opt_kwargs)
        on_device = result.pop_lazy("fun")

        def fun():   # result.fun on first access (bundle_adjustment.py:66-98 at the solution)
            try:
                return on_device()
            except RuntimeError:   # the cached problem has moved on: rebuild from the caller's arrays
                return residuals(x, all_calib_uvs[:, use_frames], calib_objpoints)
        result.set_lazy("fun", fun)
    ext, intr, poses = deserialize_params(result.x, n_cameras)
    return ext, intr, poses, use_frames, result
