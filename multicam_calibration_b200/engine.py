"""Device-resident bundle-adjustment problem on top of the ``libmcba`` C ABI.

PyTorch is used for device memory, streams and (multi-GPU) rendezvous only; all
arithmetic runs in the hand-written sm_100a kernels behind ``include/mcba.h``.
"""
import ctypes

import numpy as np

from . import _native
from ._native import Options, Result, check

TERMINATION_MESSAGES = {   # scipy optimize/_lsq/common.py / least_squares.py
    -1: "The damping grew without bound: no descent step was found.",
    0: "The maximum number of function evaluations is exceeded.",
    1: "`gtol` termination condition is satisfied.",
    2: "`ftol` termination condition is satisfied.",
    3: "`xtol` termination condition is satisfied.",
    4: "Both `ftol` and `xtol` termination conditions are satisfied.",
}

_UNSUPPORTED = ("jac", "jac_sparsity", "bounds", "tr_solver", "tr_options", "diff_step",
                "args", "kwargs", "callback", "workers")


class OptimizeResult(dict):
    """Attribute-access dict with the fields of ``scipy.optimize.OptimizeResult``.

    Fields registered with :meth:`set_lazy` (``fun``: the 2·O-entry residual vector at the
    solution, 134 MB at BASELINE configs[2]) are computed on the device and brought to the
    host on first access only; the solve itself never waits for them."""
    __setattr__ = dict.__setitem__

    def _lazy_fields(self):
        try:
            return object.__getattribute__(self, "_lazy_store")
        except AttributeError:
            object.__setattr__(self, "_lazy_store", {})
            return object.__getattribute__(self, "_lazy_store")

    def set_lazy(self, name, thunk):
        self._lazy_fields()[name] = thunk
        dict.pop(self, name, None)

    def pop_lazy(self, name):
        """Remove and return the thunk of a lazy field (to wrap it)."""
        return self._lazy_fields().pop(name)

    def __missing__(self, name):
        lazy = self._lazy_fields()
        if name in lazy:
            value = lazy.pop(name)()
            dict.__setitem__(self, name, value)
            return value
        raise KeyError(name)

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError as e:      # like scipy's OptimizeResult: a typo is an error, hasattr() works
            raise AttributeError(name) from e

    def get(self, name, default=None):
        try:
            return self[name]
        except KeyError:
            return default

    def __contains__(self, name):
        return dict.__contains__(self, name) or name in self._lazy_fields()

    def keys(self):
        return list(dict.keys(self)) + list(self._lazy_fields())

    def __dir__(self):
        return list(self.keys())


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _on_stream(fn):
    """Run a method with the problem's CUDA stream current, so torch copies and
    the library's kernels are ordered on one stream."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        cuda = self.torch.cuda
        with cuda.device(self.device):
            # Work the caller queued on ITS current stream (e.g. the device gather that produced a
            # tensor argument) must precede ours: the problem's stream is non-blocking and has no
            # implicit ordering against it.  Captured before the stream switch below.
            caller = cuda.current_stream(self.device)
            if caller != self.stream:
                self.stream.wait_stream(caller)
            with cuda.stream(self.stream):
                return fn(self, *a, **k)
    return wrapper


def check_fixed(fixed, n_cameras):
    """``fixed`` (camera parameters held at their initial values, ``serialize_params`` order) as the 12C
    bytes of ``mcba_set_fixed``, or None when nothing is held (None or an all-False mask)."""
    if fixed is None:
        return None
    mask = np.asarray(fixed)
    if mask.dtype != np.bool_:
        raise ValueError(f"fixed must be a boolean array, got dtype {mask.dtype}")
    if mask.shape != (n_cameras, 12):
        raise ValueError(f"fixed must have shape ({n_cameras}, 12) (fx fy cx cy k1 k2 rvec tvec per camera), "
                         f"got {mask.shape}")
    if not mask.any():
        return None
    return np.ascontiguousarray(mask, dtype=np.uint8).ravel()


def parse_options(opt_kwargs, n_params):
    """Map ``least_squares`` keyword arguments (bundle_adjustment.py:301-304) to
    :class:`Options`; scipy-only knobs the engine replaces are rejected loudly."""
    kw = dict(verbose=2, x_scale="jac", ftol=1e-4, method="trf", loss="soft_l1")
    kw.update(opt_kwargs)
    for k in _UNSUPPORTED:
        if k in kw:
            raise TypeError(f"bundle_adjust: least_squares option {k!r} is not supported by the "
                            "B200 engine (analytic Jacobian + Schur + Levenberg-Marquardt).")
    if kw.pop("method") not in ("trf", "lm"):
        raise ValueError("bundle_adjust: only method='trf' (replaced by device LM) is accepted")
    if kw.pop("x_scale") != "jac":
        raise ValueError("bundle_adjust: only x_scale='jac' is supported")
    loss = kw.pop("loss")
    if loss not in ("linear", "soft_l1"):
        raise ValueError("bundle_adjust: loss must be 'soft_l1' or 'linear'")
    o = Options()
    _native.load().mcba_default_options(ctypes.byref(o))
    tol = lambda v: 0.0 if v is None else float(v)
    o.ftol, o.xtol, o.gtol = tol(kw.pop("ftol")), tol(kw.pop("xtol", 1e-8)), tol(kw.pop("gtol", 1e-8))
    max_nfev = kw.pop("max_nfev", None)
    o.max_nfev = 0 if max_nfev is None else int(max_nfev)
    o.loss = _native.LOSSES[loss]
    o.f_scale = float(kw.pop("f_scale", 1.0))
    o.verbose = int(kw.pop("verbose"))
    hessian = kw.pop("hessian", "auto")
    if hessian not in _native.HESSIANS:
        raise ValueError(f"bundle_adjust: hessian must be one of {sorted(_native.HESSIANS)}")
    o.hessian = _native.HESSIANS[hessian]
    for name in ("lambda0", "lambda_min", "lambda_max"):
        if name in kw:
            setattr(o, name, float(kw.pop(name)))
    if kw:
        raise TypeError(f"bundle_adjust: unexpected keyword arguments {sorted(kw)}")
    return o


class BAProblem:
    """Observations + device state for one (rank-local) set of frames.

    Parameters
    ----------
    all_calib_uvs : (C, F, N, 2) float64, NaN = missing (this rank's frames)
    calib_objpoints : (N, 3)
    comm : optional ``(unique_id_bytes, rank, world_size)`` for multi-GPU solves
    """

    def __init__(self, all_calib_uvs, calib_objpoints, device=None, comm=None):
        torch = _native.require_cuda()
        self.torch = torch
        self.lib = _native.load()
        on_device = hasattr(all_calib_uvs, "is_cuda")     # a float64 CUDA tensor: no host round trip
        uvs = all_calib_uvs if on_device else np.ascontiguousarray(all_calib_uvs, dtype=np.float64)
        obj = np.ascontiguousarray(calib_objpoints, dtype=np.float64)
        if uvs.ndim != 4 or uvs.shape[-1] != 2 or obj.shape != (uvs.shape[2], 3):
            raise ValueError("all_calib_uvs must be (C,F,N,2) and calib_objpoints (N,3)")
        self.C, self.F, self.N, _ = (int(v) for v in uvs.shape)
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.n_params = 12 * self.C + 6 * self.F
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            self.stream = torch.cuda.Stream(device=self.device)
            check(self.lib.mcba_create(ctypes.byref(self._h), self.C, self.F, self.N, self.device))
            check(self.lib.mcba_set_stream(self._h, ctypes.c_void_p(self.stream.cuda_stream)))
        self.rank, self.world = 0, 1
        if comm is not None:
            uid, rank, world = comm
            buf = ctypes.create_string_buffer(bytes(uid), 128)
            check(self.lib.mcba_comm_init(self._h, buf, int(rank), int(world)))
            self.rank, self.world = int(rank), int(world)
            self._open_peer_memory()
        self.set_observations(uvs, obj)

    def _open_peer_memory(self):
        """Exchange buffers of all ranks mapped through CUDA IPC (handles gathered with
        torch.distributed): the per-evaluation sums then run as one kernel over NVLink peer memory
        (csrc/mcba_peer.cu).  ``MCBA_NO_PEER=1`` keeps the NCCL all-reduce (A/B measurements)."""
        import os
        import torch.distributed as dist
        self.peer_memory = False
        if self.world <= 1 or os.environ.get("MCBA_NO_PEER") or not (dist.is_available() and dist.is_initialized()):
            return
        # every step is collective: a rank that cannot export / map still takes part in the gathers,
        # and the peer path is used only if EVERY rank mapped every buffer (else all ranks keep NCCL)
        import sys
        mine = ctypes.create_string_buffer(64)
        ok = self.lib.mcba_comm_ipc_export(self._h, self.rank, self.world, mine) == _native.MCBA_OK
        if os.environ.get("MCBA_TEST_PEER_FAIL") == str(self.rank):   # tests: this rank pretends it cannot export
            ok = False
        handles = [None] * self.world
        dist.all_gather_object(handles, (ok, bytes(mine.raw)))
        ok = all(h[0] for h in handles)
        if ok:
            blob = ctypes.create_string_buffer(b"".join(h[1] for h in handles), 64 * self.world)
            ok = self.lib.mcba_comm_ipc_open(self._h, blob) == _native.MCBA_OK
        votes = [None] * self.world
        dist.all_gather_object(votes, bool(ok))          # also: every rank has mapped before the first push
        self.peer_memory = all(votes)
        if not self.peer_memory:
            self.lib.mcba_comm_ipc_enable(self._h, 0)
            if self.rank == 0:
                print("multicam_calibration_b200: CUDA IPC peer buffers unavailable "
                      f"({self.lib.mcba_last_error().decode(errors='replace')}); using the NCCL all-reduce", file=sys.stderr)

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.mcba_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _dev(self, a):
        return _native.to_device(a, self.device)

    def _empty(self, *shape):
        return self.torch.empty(shape, dtype=self.torch.float64, device=f"cuda:{self.device}")

    def _x(self, params):
        params = np.asarray(params, dtype=np.float64).ravel()
        if params.size != self.n_params:
            raise ValueError(f"params has {params.size} entries, expected {self.n_params}")
        return self._dev(params)

    @_on_stream
    def set_observations(self, uvs, obj=None):
        """``uvs``: (C,F,N,2) numpy array, or a float64 CUDA tensor of that shape (device copy)."""
        on_device = hasattr(uvs, "is_cuda")
        if not on_device:
            uvs = np.ascontiguousarray(uvs, dtype=np.float64)
        if tuple(uvs.shape) != (self.C, self.F, self.N, 2):
            raise ValueError("observation shape changed")
        if obj is not None:
            self._obj = np.ascontiguousarray(obj, dtype=np.float64)
        if on_device:
            if not uvs.is_cuda or uvs.dtype != self.torch.float64:
                raise ValueError("device observations must be a float64 CUDA tensor")
            d_uvs = uvs.contiguous()     # ordered after its producer by _on_stream
            d_obj = self._dev(self._obj)
        else:   # pageable numpy -> device at PCIe rate (mcba_upload), then the device path
            d_uvs, d_obj = self._dev(uvs), self._dev(self._obj)
        check(self.lib.mcba_set_observations(self._h, _ptr(d_uvs), _ptr(d_obj), 1))
        if self.world > 1:   # finite scalars per camera: where this rank's residuals go in the gathered vector
            self._per_camera = self.torch.isfinite(d_uvs).sum(dim=(1, 2, 3)).cpu().numpy().astype(np.int64)
        check(self.lib.mcba_synchronize(self._h))   # uvs may be a temporary
        self._obs_token = object()

    @property
    def n_residuals(self):
        m, o = ctypes.c_int64(), ctypes.c_int64()
        check(self.lib.mcba_num_residuals(self._h, ctypes.byref(m), ctypes.byref(o)))
        return m.value

    @property
    def n_observations(self):
        m, o = ctypes.c_int64(), ctypes.c_int64()
        check(self.lib.mcba_num_residuals(self._h, ctypes.byref(m), ctypes.byref(o)))
        return o.value

    @property
    def kernel_launches(self):
        return int(self.lib.mcba_kernel_launches(self._h))

    @_on_stream
    def plan_info(self):
        """Kernel variants this problem's evaluation and solve take (``mcba_plan_info``): a dict of
        ``_native.PLAN_FIELDS`` with ``k2c_mode`` and ``solve`` named, plus ``units``, the live
        (tile, camera) units of every camera."""
        n = len(_native.PLAN_FIELDS) + self.C
        out = (ctypes.c_int64 * n)()
        check(self.lib.mcba_plan_info(self._h, out, n))
        info = dict(zip(_native.PLAN_FIELDS, (int(v) for v in out)))
        info["k2c_mode"] = _native.K2C_MODES[info["k2c_mode"]]
        info["solve"] = _native.SOLVE_TIERS[info["solve"]]
        info["units"] = [int(v) for v in out[len(_native.PLAN_FIELDS):]]
        return info

    # ------------------------------------------------------------------ per-call operators
    @_on_stream
    def residuals(self, params):
        """bundle_adjustment.py:66-98."""
        x = self._x(params)
        r = self._empty(self.n_residuals)
        check(self.lib.mcba_residuals(self._h, _ptr(x), _ptr(r)))
        return _native.to_host(r)

    @_on_stream
    def residuals_device(self, params):
        """Residual vector left on the device + the number of entries per camera (the vector is
        camera-major, bundle_adjustment.py:97) -- what a frame-sharded solve gathers."""
        x = self._x(params)
        r = self._empty(self.n_residuals)
        check(self.lib.mcba_residuals(self._h, _ptr(x), _ptr(r)))
        check(self.lib.mcba_synchronize(self._h))
        per_cam = getattr(self, "_per_camera", None)
        return r, per_cam

    @_on_stream
    def predict(self, params):
        x = self._x(params)
        uv = self._empty(self.C, self.F, self.N, 2)
        check(self.lib.mcba_predict(self._h, _ptr(x), _ptr(uv)))
        return _native.to_host(uv)

    @_on_stream
    def jacobian_blocks(self, params):
        """Residual-Jacobian blocks ``Jc (C,F,N,2,12)``, ``Jp (C,F,N,2,6)``."""
        x = self._x(params)
        Jc = self._empty(self.C, self.F, self.N, 2, 12)
        Jp = self._empty(self.C, self.F, self.N, 2, 6)
        check(self.lib.mcba_jacobian_blocks(self._h, _ptr(x), _ptr(Jc), _ptr(Jp)))
        return _native.to_host(Jc), _native.to_host(Jp)

    @_on_stream
    def cost(self, params, loss="soft_l1", f_scale=1.0):
        x = self._x(params)
        c, s, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_int64()
        check(self.lib.mcba_cost(self._h, _ptr(x), _native.LOSSES[loss], float(f_scale),
                                 ctypes.byref(c), ctypes.byref(s), ctypes.byref(n)))
        return c.value, s.value, n.value

    @_on_stream
    def build_reduced(self, params, lam=0.0, loss="soft_l1", f_scale=1.0):
        """Reduced camera system ``(S, b, g_cam, cost)`` at ``params``."""
        x = self._x(params)
        nc = 12 * self.C
        S, b, g = np.empty((nc, nc)), np.empty(nc), np.empty(nc)
        cost = ctypes.c_double()
        check(self.lib.mcba_build_reduced(
            self._h, _ptr(x), float(lam), _native.LOSSES[loss], float(f_scale),
            S.ctypes.data_as(ctypes.c_void_p), b.ctypes.data_as(ctypes.c_void_p),
            g.ctypes.data_as(ctypes.c_void_p), ctypes.cast(ctypes.byref(cost), ctypes.c_void_p)))
        self._x_last = x
        return S, b, g, cost.value

    @_on_stream
    def set_fixed(self, fixed):
        """Hold camera parameters at their initial values in the following :meth:`solve_step` calls
        (``mcba_set_fixed``): ``fixed`` (C, 12) bool in ``serialize_params`` order, or None.  :meth:`solve` and
        :meth:`covariance` set their own mask on every call."""
        mask = check_fixed(fixed, self.C)
        check(self.lib.mcba_set_fixed(self._h, None if mask is None else mask.ctypes.data_as(ctypes.c_void_p)))

    @_on_stream
    def covariance(self, params, reference_camera=0, loss="soft_l1", f_scale=1.0, sigma=None, poses=True, fixed=None):
        """Covariance of the calibration at ``params`` (``mcba_covariance``): ``(Sigma_cam (12C,12C),
        Sigma_pose (F,6,6) or None, stats)``.

        ``s^2 inv(J~^T J~)`` with J~ the residual Jacobian scaled as scipy's ``least_squares`` scales it
        for the robust loss (``result.jac``), the extrinsics of ``reference_camera`` held fixed (exact
        zeros), NaN for cameras and frames without observations.  ``s^2 = sigma^2``, or
        ``2 cost / (m - p)`` with ``p`` the free parameters.  For ``loss='linear'`` this is the asymptotic
        covariance of the least-squares estimate; for ``soft_l1`` it is scipy's usual recipe with the
        robust-scaled Jacobian, not an M-estimator sandwich.  Singular systems raise
        ``numpy.linalg.LinAlgError``.

        ``fixed`` (C, 12) bool: parameters held fixed, conditioned on (their rows and columns are exactly 0).
        When it holds all six extrinsics of a camera that fixes the gauge, and ``reference_camera`` must be None
        or such a camera; otherwise the mask may hold no extrinsic entry."""
        if loss not in ("linear", "soft_l1"):
            raise ValueError("covariance: loss must be 'linear' or 'soft_l1'")
        x = self._x(params)
        self.set_fixed(fixed)
        nc = 12 * self.C
        cam = np.empty((nc, nc))
        pose = self._empty(self.F, 6, 6) if poses else None
        stats = np.zeros(9)
        sigma2 = -1.0 if sigma is None else float(sigma) ** 2
        code = self.lib.mcba_covariance(
            self._h, _ptr(x), _native.LOSSES[loss], float(f_scale), -1 if reference_camera is None else int(reference_camera), sigma2,
            cam.ctypes.data_as(ctypes.c_void_p), _ptr(pose) if poses else None, stats.ctypes.data_as(ctypes.c_void_p))
        if code == _native.ERR_SOLVER:
            raise np.linalg.LinAlgError(self.lib.mcba_last_error().decode(errors="replace"))
        if code == _native.ERR_ARG:
            raise ValueError(self.lib.mcba_last_error().decode(errors="replace"))
        check(code)
        self._x_last = x
        keys = ("sigma2", "dof", "n_residuals", "cost", "empty_frames", "min_pose_pivot",
                "eval_ms", "camera_ms", "pose_ms")
        info = dict(zip(keys, (float(v) for v in stats)))
        info["n_residuals"] = int(info["n_residuals"])
        info["empty_frames"] = int(info["empty_frames"])
        return cam, (_native.to_host(pose) if poses else None), info

    @_on_stream
    def gradient(self):
        g = self._empty(self.n_params)
        check(self.lib.mcba_gradient(self._h, _ptr(g)))
        return _native.to_host(g)

    @_on_stream
    def solve_step(self, lam):
        """Damped step from the system of the last :meth:`build_reduced`."""
        xn = self._empty(self.n_params)
        check(self.lib.mcba_solve_step(self._h, _ptr(self._x_last), float(lam), _ptr(xn)))
        return _native.to_host(xn)

    def _fun_thunk(self, xs):
        """Residual vector at ``xs`` on first access of ``result.fun``: from this problem when it
        still holds the same observations, else from a device copy of them kept with the result."""
        token = self._obs_token

        def thunk():
            if getattr(self, "_h", None) is not None and self._h.value and self._obs_token is token:
                return self.residuals(xs)
            raise RuntimeError("result.fun: the problem was closed or its observations replaced before the "
                               "residual vector was requested; call residuals(result.x, uvs, objpoints)")
        return thunk

    # ------------------------------------------------------------------ the solve
    @_on_stream
    def solve(self, x0, fixed=None, **opt_kwargs):
        """Levenberg-Marquardt on the device; returns ``(x, OptimizeResult)``.

        ``fixed`` (C, 12) bool, ``serialize_params`` order: camera parameters held at their values in ``x0``
        (Levenberg-Marquardt on the free sub-problem; ``optimality`` and the default ``max_nfev`` count free
        parameters only, ``grad`` stays complete)."""
        opts = parse_options(opt_kwargs, self.n_params)
        self.set_fixed(fixed)
        verbose = opts.verbose if self.rank == 0 else 0
        keep = []
        if verbose >= 2:
            print("{0:^15}{1:^15}{2:^15}{3:^15}{4:^15}{5:^15}".format(
                "Iteration", "Total nfev", "Cost", "Cost reduction", "Step norm", "Optimality"))

            def _cb(user, it, nfev, cost, red, step, opt):
                red_s = " " * 15 if red != red else f"{red:^15.2e}"
                step_s = " " * 15 if step != step else f"{step:^15.2e}"
                print(f"{it:^15}{nfev:^15}{cost:^15.4e}{red_s}{step_s}{opt:^15.2e}")
            cb = _native.ITER_CALLBACK(_cb)
            keep.append(cb)
            opts.iter_callback = cb
        x = self._x(x0)
        grad = self._empty(self.n_params)
        res = Result()
        check(self.lib.mcba_lm_run(self._h, _ptr(x), ctypes.byref(opts), ctypes.byref(res), _ptr(grad)))
        xs = _native.to_host(x)
        out = OptimizeResult(
            x=xs, cost=res.cost, grad=_native.to_host(grad), optimality=res.optimality,
            active_mask=np.zeros_like(xs), nfev=res.nfev, njev=res.njev, status=res.status,
            message=TERMINATION_MESSAGES.get(res.status, "unknown"), success=res.status > 0,
            jac=None, initial_cost=res.cost0, rms=res.rms, iterations=res.iterations,
            solve_ms=res.solve_ms, step_norm=res.step_norm, damping=res.lambda_,
            kernel_launches=res.kernel_launches, n_residuals=res.n_residuals)
        if self.world == 1:
            out.set_lazy("fun", self._fun_thunk(xs))
        if verbose >= 1:
            print(out.message)
            print(f"Function evaluations {res.nfev}, initial cost {res.cost0:.4e}, final cost "
                  f"{res.cost:.4e}, first-order optimality {res.optimality:.2e}.")
        return xs, out
