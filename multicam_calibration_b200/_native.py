"""ctypes binding of ``libmcba.so`` (the C ABI declared in ``include/mcba.h``).

There is no CPU fallback: if the library has not been built, or no CUDA device
is present, every compute entry point raises.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmcba.so")
CSRC = os.path.join(_HERE, "csrc")

MCBA_OK = 0
ERR_ARG = -1
ERR_SOLVER = -3
ERR_NONFINITE = -4
LOSSES = {"linear": 0, "soft_l1": 1, "soft_l1_irls": 0x101}
HESSIANS = {"auto": 0, "triggs": 1, "irls": 2}

# mcba_plan_info: indices of the launch choices (include/mcba.h MCBA_PLAN_*); the live units per camera follow
PLAN_FIELDS = ("k2p_warps", "k2p_grid", "k2c_mode", "k2c_warps", "k2c_parts", "syrk_warps", "syrk_gy",
               "syrk_static_nb", "solve", "tiles", "backsub_grid", "cameras")
K2C_MODES = {1: "ring", 2: "stream"}
SOLVE_TIERS = {0: "cusolver", 3: "regs3", 8: "regs8", 119: "smem19"}

ITER_CALLBACK = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                 ctypes.c_double, ctypes.c_double, ctypes.c_double)


class Options(ctypes.Structure):
    _fields_ = [("ftol", ctypes.c_double), ("xtol", ctypes.c_double), ("gtol", ctypes.c_double),
                ("max_nfev", ctypes.c_int32), ("loss", ctypes.c_int32), ("f_scale", ctypes.c_double),
                ("verbose", ctypes.c_int32), ("hessian", ctypes.c_int32),
                ("lambda0", ctypes.c_double), ("lambda_min", ctypes.c_double),
                ("lambda_max", ctypes.c_double), ("iter_callback", ITER_CALLBACK),
                ("callback_user", ctypes.c_void_p)]


class Result(ctypes.Structure):
    _fields_ = [("cost", ctypes.c_double), ("cost0", ctypes.c_double), ("optimality", ctypes.c_double),
                ("rms", ctypes.c_double), ("step_norm", ctypes.c_double), ("lambda_", ctypes.c_double),
                ("solve_ms", ctypes.c_double), ("n_residuals", ctypes.c_int64),
                ("nfev", ctypes.c_int32), ("njev", ctypes.c_int32), ("iterations", ctypes.c_int32),
                ("status", ctypes.c_int32), ("kernel_launches", ctypes.c_int64)]


# include/mcba.h MCBA_REFINE_LOSS_*: refine_points' own codes (scipy's five losses)
REFINE_LOSSES = {"linear": 0, "soft_l1": 1, "huber": 2, "cauchy": 3, "arctan": 4}


class RefineOptions(ctypes.Structure):
    _fields_ = [("loss", ctypes.c_int32), ("f_scale", ctypes.c_double), ("sigma", ctypes.c_double),
                ("ftol", ctypes.c_double), ("xtol", ctypes.c_double), ("gtol", ctypes.c_double),
                ("max_iter", ctypes.c_int32), ("flags", ctypes.c_int32)]


class McbaError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libmcba error {code}: {message}")
        self.code = code


_P = ctypes.c_void_p
_D = ctypes.c_double
_I = ctypes.c_int
_L = ctypes.c_int64
_SIGNATURES = {
    "mcba_last_error": (ctypes.c_char_p, []),
    "mcba_version": (_I, []),
    "mcba_default_options": (None, [ctypes.POINTER(Options)]),
    "mcba_create": (_I, [ctypes.POINTER(_P), _I, _L, _I, _I]),
    "mcba_destroy": (_I, [_P]),
    "mcba_set_stream": (_I, [_P, _P]),
    "mcba_synchronize": (_I, [_P]),
    "mcba_set_observations": (_I, [_P, _P, _P, _I]),
    "mcba_num_residuals": (_I, [_P, ctypes.POINTER(_L), ctypes.POINTER(_L)]),
    "mcba_residuals": (_I, [_P, _P, _P]),
    "mcba_predict": (_I, [_P, _P, _P]),
    "mcba_jacobian_blocks": (_I, [_P, _P, _P, _P]),
    "mcba_cost": (_I, [_P, _P, _I, _D, ctypes.POINTER(_D), ctypes.POINTER(_D), ctypes.POINTER(_L)]),
    "mcba_build_reduced": (_I, [_P, _P, _D, _I, _D, _P, _P, _P, _P]),
    "mcba_build_reduced_host": (_I, [_P, _P, _P, _P, _D, _I, _D, _P, _P, _P]),
    "mcba_solve_step": (_I, [_P, _P, _D, _P]),
    "mcba_set_fixed": (_I, [_P, _P]),
    "mcba_gradient": (_I, [_P, _P]),
    "mcba_covariance": (_I, [_P, _P, _I, _D, _I, _D, _P, _P, _P]),
    "mcba_lm_run": (_I, [_P, _P, ctypes.POINTER(Options), ctypes.POINTER(Result), _P]),
    "mcba_comm_unique_id": (_I, [_P]),
    "mcba_comm_init": (_I, [_P, _P, _I, _I]),
    "mcba_comm_ipc_export": (_I, [_P, _I, _I, _P]),
    "mcba_comm_ipc_open": (_I, [_P, _P]),
    "mcba_comm_ipc_enable": (_I, [_P, _I]),
    "mcba_project_points": (_I, [_I, _P, _P, _L, _P, _P, _P, _P]),
    "mcba_project_points_multi": (_I, [_I, _P, _P, _L, _I, _P, _P, _P, _P]),
    "mcba_embed_points": (_I, [_I, _P, _P, _L, _P, _I, _P]),
    "mcba_undistort_points": (_I, [_I, _P, _P, _L, _P, _P, _P]),
    "mcba_triangulate": (_I, [_I, _P, _P, _I, _L, _P, _P, _P, _P]),
    "mcba_refine_points": (_I, [_I, _P, _P, _I, _L, _P, _P, _P, _P, ctypes.POINTER(RefineOptions),
                                _P, _P, _P, _P, _P, _P, _P, _P]),
    "mcba_point_covariance": (_I, [_I, _P, _P, _I, _L, _P, _P, _P, _P, _P, _I, _D, _D, _P, _P, _P]),
    "mcba_kernel_launches": (_L, [_P]),
    "mcba_plan_info": (_I, [_P, ctypes.POINTER(_L), _I]),
    "mcba_profile": (_I, [_P, _I, ctypes.POINTER(_D), ctypes.POINTER(_I)]),
    "mcba_measure_fp64_peak": (_I, [_I, ctypes.POINTER(_D)]),
    "mcba_select_frames": (_I, [_I, _P, _P, _I, _L, _I, _P, _P, _D, _P, ctypes.POINTER(_D)]),
    "mcba_frame_errors": (_I, [_I, _P, _P, _I, _L, _I, _P, _P, _P, _P, _P, ctypes.POINTER(_L)]),
    "mcba_key_histogram": (_I, [_I, _P, _P, _L, ctypes.c_uint64, _I, _P]),
    "mcba_apply_threshold": (_I, [_I, _P, _P, _P, _I, _L, _D, _P, ctypes.POINTER(_L)]),
    "mcba_gather_frames": (_I, [_I, _P, _P, _I, _L, _I, _P, _L, _P]),
    "mcba_pairwise_transform": (_I, [_I, _P, _P, _P, _L, ctypes.POINTER(_D), ctypes.POINTER(_L)]),
    "mcba_consensus_poses": (_I, [_I, _P, _P, _P, _I, _L, _P]),
    "mcba_transformation_vectors": (_I, [_I, _P, _P, _L, _I, _P]),
    "mcba_homography_transfer": (_I, [_I, _P, _P, _P, _P, _I, _L, _I, _P, _P, _P, _P]),
    "mcba_upload": (_I, [_I, _P, _P, _P, ctypes.c_size_t]),
    "mcba_download": (_I, [_I, _P, _P, _P, ctypes.c_size_t]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def build(verbose=False):
    """Compile ``libmcba.so`` for sm_100a with nvcc (cross-compiles without a GPU)."""
    proc = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if verbose or proc.returncode:
        print(proc.stdout[-4000:])
        print(proc.stderr[-4000:])
    if proc.returncode:
        raise RuntimeError("building libmcba.so failed")
    return LIB_PATH


def load():
    """Load the library and bind the signatures; raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA library has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C "
            f"{CSRC}`). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != MCBA_OK:
        msg = load().mcba_last_error().decode(errors="replace")
        if code == ERR_NONFINITE:
            raise ValueError(msg or "Residuals are not finite in the initial point.")
        raise McbaError(code, msg)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("multicam_calibration_b200 needs a CUDA device (B200, sm_100a); "
                           "there is no CPU fallback.")
    return torch


def to_device(array, device=None):
    """float64 numpy array -> CUDA tensor through ``mcba_upload`` (staged, PCIe rate for pageable
    memory), ordered on torch's current stream of ``device``."""
    import numpy as np
    torch = require_cuda()
    dev = torch.cuda.current_device() if device is None else int(device)
    a = np.ascontiguousarray(array, dtype=np.float64)
    out = torch.empty(a.shape, dtype=torch.float64, device=f"cuda:{dev}")
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(load().mcba_upload(dev, stream, ctypes.c_void_p(out.data_ptr()), a.ctypes.data_as(ctypes.c_void_p),
                             a.nbytes))
    return out


def upload_into(dst, array):
    """float64 numpy array -> an existing contiguous CUDA tensor (view) of the same size, through
    ``mcba_upload``; ordered on torch's current stream of the tensor's device."""
    import numpy as np
    torch = require_cuda()
    a = np.ascontiguousarray(array, dtype=np.float64)
    if not dst.is_contiguous() or dst.dtype != torch.float64 or dst.numel() != a.size:
        raise ValueError("upload_into: destination must be a contiguous float64 CUDA tensor of the source's size")
    dev = dst.device.index
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(load().mcba_upload(dev, stream, ctypes.c_void_p(dst.data_ptr()), a.ctypes.data_as(ctypes.c_void_p), a.nbytes))
    return dst


def to_host(tensor):
    """CUDA tensor -> fresh numpy array through ``mcba_download`` (current stream of its device)."""
    import numpy as np
    torch = require_cuda()
    t = tensor.contiguous()
    dev = t.device.index
    out = np.empty(tuple(t.shape), dtype=np.dtype(str(t.dtype).replace("torch.", "")))
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(load().mcba_download(dev, stream, out.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(t.data_ptr()),
                               out.nbytes))
    return out
