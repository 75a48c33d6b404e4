#!/usr/bin/env python
"""Benchmark of the bundle-adjustment hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this engine (B200)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's S, b, g_cam,
                                                             # cost and gradient as DIR/*.npy

The metric is BASELINE.json's: observations/s through residual + analytic Jacobian + Schur
accumulation (`value`, `e2e`), with the BA time-to-converge on the same data in `ba_converge`.
A "step" is one pass of residual + analytic Jacobian + Schur accumulation (the reduced camera
system S, b) over every observation of the workload.

Workloads (BASELINE.json configs):
  --config 2 (default)  6 cameras x 50,000 frames x 35 corners, 20 % missing detections, 0.5 px noise
  --config 3            16 cameras x 200,000 frames over 8 GPUs (25,000 frames per GPU)
  --scaling weak (default): the frame count above is PER GPU;  --scaling strong: it is the TOTAL,
  split over the ranks (config 3 is quoted at 8 GPUs: 200,000 frames total / N in strong mode).
Frames are sharded over ranks and only the packed reduced system is summed across them.

What one default run reports besides the headline (all driver-visible in the ONE JSON line):
  multi_gpu_parity  (N > 1) the sharded S, b, cost against a single-GPU rebuild of the gathered
                    shards, for the peer-memory kernel and for NCCL, and bit-identity across ranks
  strong            (N > 1, weak runs) the 50,000-frame problem split N ways, with the limiter named
  ba_converge       LM time-to-converge on the device and through the public bundle_adjust call
  extra             configs[3] shard per GPU; (N = 1) configs[4] triangulate / project_points of
                    1M keypoints x 6 cameras and the K1 residual kernel, each with its own roofline,
                    cpu_baseline and e2e through the public numpy API
Prints ONE JSON line on rank 0.
"""
import argparse
import contextlib
import ctypes
import io
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

_BASELINE = os.path.join(ROOT, "BASELINE.json")
METRIC = json.load(open(_BASELINE))["metric"] if os.path.exists(_BASELINE) \
    else "obs/s residual+Jacobian+Schur; BA time-to-converge, 6 cams×50k frames"
UNIT = "obs/s"
SIGMA, P_MISSING, CORNERS = 0.5, 0.2, 35
CONFIGS = {   # BASELINE.json configs[k]: cameras, frames (per GPU in weak mode), GPUs the config is quoted on
    2: dict(cams=6, frames=50_000, quoted_gpus=1, name="BASELINE.json configs[2]"),
    3: dict(cams=16, frames=200_000, quoted_gpus=8, name="BASELINE.json configs[3]"),
}
CPU_SAMPLE_FRAMES = int(os.environ.get("MCBA_BENCH_SAMPLE_FRAMES", 1000))      # frames of the workload timed on the host per step
CPU_CONVERGE_FRAMES = int(os.environ.get("MCBA_BENCH_CONVERGE_FRAMES", 500))   # scipy trf to convergence: BASELINE configs[0] (6 x 500), ~1 min of one core
ALG_FMA_PER_OBS = 250.0   # projection + Jacobian rows ~65, robust weights ~30, A_cf / q_cf accumulation ~150, bookkeeping ~5
LAMBDA, LOSS = 1e-3, "soft_l1"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return json.load(open(path)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def workload_name(cams, frames, scaling, world, tag):
    per = "frames/GPU" if scaling == "weak" else f"frames split over {world} GPU(s)"
    return (f"{cams} cams x {frames} {per} x {CORNERS} corners, {int(P_MISSING * 100)}% missing detections, "
            f"sigma={SIGMA} px ({tag})")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __new__(cls, index):
        # NVML in-process (1 ms period) when available: the timed region lasts milliseconds,
        # shorter than nvidia-smi's start-up; the nvidia-smi loop is the fallback.
        try:
            import pynvml  # noqa: F401
            return object.__new__(NvmlClockSampler)
        except Exception:
            return object.__new__(cls)

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        out = self.proc.communicate(timeout=10)[0]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class NvmlClockSampler(ClockSampler):
    """Polled from the launching thread while the timed kernels are in flight (no helper
    thread: a Python thread competing for the GIL would slow the enqueue loop itself)."""

    def __init__(self, index):
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")
        phys = int(vis[index]) if index < len(vis) and vis[index].strip().isdigit() else index
        self.dev = pynvml.nvmlDeviceGetHandleByIndex(phys)
        self.sm, self.reasons = [], set()
        self.mx = pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM)
        nv = pynvml
        self.names = {getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                      getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                      getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                      getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap"}
        self.get_reasons = (getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None)
                            or nv.nvmlDeviceGetCurrentClocksThrottleReasons)

    def sample(self):
        try:
            self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.dev, self.nv.NVML_CLOCK_SM))
            mask = self.get_reasons(self.dev)
            for bit, name in self.names.items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def poll_until(self, event):
        """Sample until the CUDA event has completed (i.e. during the timed region)."""
        self.sample()
        while not event.query():
            self.sample()

    def stop(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": float(self.mx),
                "samples": len(self.sm), "reasons": sorted(self.reasons), "source": "nvml polled during the timed region"}


# ---------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the path (numpy/scipy port in oracle/)
# ---------------------------------------------------------------------------------------------
def cpu_reference_step(sc_uvs, obj, x0, A):
    """One residual evaluation + one finite-difference Jacobian through the sparsity pattern:
    what scipy's trf does per outer iteration for bundle_adjustment.py:307-313."""
    from scipy.optimize._numdiff import approx_derivative
    from oracle import np_oracle as orc
    f0 = orc.residuals(x0, sc_uvs, obj)
    J = approx_derivative(orc.residuals, x0, method="2-point", f0=f0, sparsity=A, args=(sc_uvs, obj))
    return f0, J


def reference_recorded():
    """What the UNMODIFIED reference measured on BASELINE configs[0] (6 cameras x 500 frames) when
    tests/golden/make_golden.py ran it in the build container (the reference is not on the GPU box)."""
    path = os.path.join(ROOT, "tests", "golden", "ba_cfg1.npz")
    if not os.path.exists(path):
        return None
    d = np.load(path, allow_pickle=True)
    return {"config": "BASELINE.json configs[0]: 6 cams x 500 frames x 35 corners, sigma=0.3 px",
            "wall_s": float(d["wall_s_default"]), "nfev": int(d["nfev_default"]), "njev": int(d["njev_default"]),
            "status": int(d["status_default"]), "cost": float(d["cost_default"]), "rms_px": float(d["rms_default"]),
            "host": str(d["wall_host"]), "versions (numpy, scipy, cv2)": [str(v) for v in d["versions"]],
            "what": "multicam_calibration.bundle_adjust(..., n_frames=None) of /root/reference, recorded in tests/golden/ba_cfg1.npz"}


def cpu_converge(frames, cams=6):
    """The reference path to convergence on a bounded sample of the workload: scipy least_squares
    (trf + LSMR + 2-point FD through jac_sparsity, reference defaults ftol=1e-4, soft_l1) on the
    oracle's restatement of bundle_adjust (bundle_adjustment.py:195-327)."""
    from multicam_calibration_b200.synthetic import make_scene
    from oracle import np_oracle as orc
    sc = make_scene(cams, frames, sigma=SIGMA, p_missing_view=P_MISSING, seed=0)
    np.random.seed(0)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        *_, use, res = orc.bundle_adjust(*sc.init_args(), n_frames=None, verbose=0)
    wall = time.perf_counter() - t0
    rms = float(np.sqrt(np.mean(res.fun ** 2)))
    return {"frames": frames, "frames_used": int(len(use)), "wall_s": wall, "nfev": int(res.nfev), "njev": int(res.njev),
            "status": int(res.status), "rms_px": rms, "cost": float(res.cost),
            "what": f"scipy least_squares trf+LSMR, 2-point FD Jacobian through jac_sparsity, ftol=1e-4, single thread, "
                    f"{cams} cams x {frames} frames of the workload (the shape of BASELINE configs[0])"}


def cpu_baseline(steps=1, warmup=0, frames=CPU_SAMPLE_FRAMES, converge_frames=0, cams=6):
    from multicam_calibration_b200.synthetic import make_scene
    from oracle import np_oracle as orc
    sc = make_scene(cams, frames, sigma=SIGMA, p_missing_view=P_MISSING, seed=0)
    x0 = sc.x0()
    A = orc.sparsity_pattern(sc.uvs)
    for _ in range(warmup):
        cpu_reference_step(sc.uvs, sc.objpoints, x0, A)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_reference_step(sc.uvs, sc.objpoints, x0, A)
    dt = (time.perf_counter() - t0) / steps
    conv = cpu_converge(converge_frames, cams) if converge_frames else None
    return {"converge": conv, "value": sc.n_obs / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": (f"{cams} cams x {frames} frames of the workload ({sc.n_obs} obs): numpy residuals + scipy "
                       f"2-point finite-difference Jacobian through jac_sparsity (18 colour groups), "
                       f"{dt:.2f} s/step, single thread (scipy path is serial); host has {os.cpu_count()} cores"),
            "s_per_step": dt, "n_obs": sc.n_obs, "reference_recorded": reference_recorded()}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return None
    cfg = CONFIGS[args.config]
    cams = args.cams or cfg["cams"]
    base = cpu_baseline(steps=args.steps, warmup=min(args.warmup, 1), converge_frames=CPU_CONVERGE_FRAMES, cams=cams)
    frames = args.frames or cfg["frames"]
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["s_per_step"] * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(cams, frames, args.scaling, args.gpus, cfg["name"]),
                       "sample_frames": CPU_SAMPLE_FRAMES},
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "converge", "reference_recorded")},
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    return line


# ---------------------------------------------------------------------------------------------
# this engine
# ---------------------------------------------------------------------------------------------
class Ctx:
    """Process-wide state of the engine arm."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from multicam_calibration_b200 import _native, distributed
        self.torch, self.dist, self.native, self.distributed = torch, dist, _native, distributed
        _native.require_cuda()   # no CPU fallback: the engine arm needs a B200
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.rank = int(os.environ.get("RANK", 0))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        if self.world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torchrun --nproc-per-node {args.gpus}")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{self.local}"))
        self.lib = _native.load()

    def comm(self):
        return (self.distributed.broadcast_unique_id(), self.rank, self.world) if self.world > 1 else None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        if self.world == 1:
            return list(values)
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def sum_over_ranks(self, values):
        if self.world == 1:
            return list(values)
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t)
        return t.tolist()


def local_scene(ctx, cams, frames, scaling):
    """This rank's frames: its own shard of the scene (weak), or its contiguous range of the one
    `frames`-frame scene every rank generates identically (strong)."""
    from multicam_calibration_b200.synthetic import make_scene
    if scaling == "weak":
        sc = make_scene(cams, frames, sigma=SIGMA, p_missing_view=P_MISSING, seed=0, shard=ctx.rank)
        return sc, sc.uvs, sc.x0()
    sc = make_scene(cams, frames, sigma=SIGMA, p_missing_view=P_MISSING, seed=0, shard=0)
    a, b = ctx.distributed.shard_bounds(frames, ctx.world, ctx.rank)
    uvs = np.ascontiguousarray(sc.uvs[:, a:b])
    x0 = np.concatenate([sc.init_cams.ravel(), sc.init_poses[a:b].ravel()])
    return sc, uvs, x0


def timed_steps(ctx, prob, d_x, steps, warmup, sampler_index=None, keep_outputs=False):
    """`warmup` untimed + `steps` timed passes of residual + Jacobian + Schur with everything resident
    in HBM; CUDA events on the problem's stream, barrier + synchronize on both sides, max over ranks.
    Returns (ms total, per-kernel ms per step [K2p, K2c, SYRK, finalize + all-reduce], launches, clocks,
    outputs).  keep_outputs: the last timed pass also copies S, b, g_cam and the cost to the host (what a
    caller of mcba_build_reduced receives) and `outputs` holds them; otherwise it is None."""
    torch, lib, h = ctx.torch, ctx.lib, prob._h
    check, null = ctx.native.check, ctypes.c_void_p()
    loss = ctx.native.LOSSES[LOSS]
    nc = 12 * prob.C
    outputs = {"S": np.empty((nc, nc)), "b": np.empty(nc), "g_cam": np.empty(nc), "cost": np.empty(1)} if keep_outputs else None
    no_out = [null] * 4
    last_out = [a.ctypes.data_as(ctypes.c_void_p) for a in outputs.values()] if keep_outputs else no_out

    def step(out=no_out):
        check(lib.mcba_build_reduced(h, ctypes.c_void_p(d_x.data_ptr()), LAMBDA, loss, 1.0, *out))

    for _ in range(warmup):
        step()
    sampler = ClockSampler(sampler_index) if sampler_index is not None else None   # NVML start-up must not skew rank 0 against the others
    check(lib.mcba_profile(h, 1, None, None))
    launches0 = prob.kernel_launches
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(prob.stream)
    for i in range(steps):
        step(last_out if i == steps - 1 else no_out)
    e1.record(prob.stream)
    if sampler is not None and hasattr(sampler, "poll_until"):
        sampler.poll_until(e1)
    ctx.barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    kms = (ctypes.c_double * 4)()
    kn = ctypes.c_int()
    check(lib.mcba_profile(h, 0, kms, ctypes.byref(kn)))
    per = [kms[i] / max(kn.value, 1) for i in range(4)]
    return ms, per, prob.kernel_launches - launches0, clocks, outputs


def multi_gpu_parity(ctx, prob, uvs_local, obj, x_local):
    """Driver-visible proof that the sharded reduced camera system is the single-GPU one: every
    rank builds S, b, cost on its shard with the sums over ranks done (a) by the peer-memory kernel
    and (b) by NCCL; rank 0 then gathers ALL shards over NVLink, rebuilds the system on one GPU
    without any communicator and compares.  Also: are the summed systems bit-identical on all ranks
    (they must be, every rank factors its own copy)."""
    torch, dist, lib, check = ctx.torch, ctx.dist, ctx.lib, ctx.native.check
    nc = 12 * prob.C
    modes = (["peer"] if getattr(prob, "peer_memory", False) else []) + ["nccl"]
    sharded = {}
    for mode in modes:
        check(lib.mcba_comm_ipc_enable(prob._h, 1 if mode == "peer" else 0))
        S, b, _, cost = prob.build_reduced(x_local, lam=LAMBDA, loss=LOSS)
        packed = torch.from_numpy(np.concatenate([S.ravel(), b, [cost]])).cuda()
        lo, hi = packed.clone(), packed.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        sharded[mode] = (S, b, cost, bool(torch.equal(lo, hi)))
    check(lib.mcba_comm_ipc_enable(prob._h, 1 if getattr(prob, "peer_memory", False) else 0))
    # gather every rank's observations (device, NVLink) and poses (host, small)
    d_local = torch.from_numpy(np.ascontiguousarray(uvs_local)).cuda()
    parts = ctx.distributed.gather_device_vectors(d_local.reshape(-1))
    poses = ctx.distributed.gather_arrays(x_local[nc:])
    out = None
    if ctx.rank == 0:
        from multicam_calibration_b200.engine import BAProblem
        C, _, N, _ = uvs_local.shape
        d_all = torch.cat([p.reshape(C, -1, N, 2) for p in parts], dim=1).contiguous()
        del parts
        single = BAProblem(d_all, obj, device=ctx.local)
        x_all = np.concatenate([x_local[:nc]] + [np.asarray(p).ravel() for p in poses])
        S1, b1, _, cost1 = single.build_reduced(x_all, lam=LAMBDA, loss=LOSS)
        single.close()
        del d_all
        out = []
        for mode in modes:
            S, b, cost, same = sharded[mode]
            out.append({"collective": mode,
                        "S_rel": float(np.abs(S - S1).max() / np.abs(S1).max()),
                        "b_rel": float(np.abs(b - b1).max() / np.abs(b1).max()),
                        "cost_rel": float(abs(cost - cost1) / abs(cost1)),
                        "bit_identical_across_ranks": same,
                        "frames_single_gpu": int(x_all.size - nc) // 6})
    del d_local
    torch.cuda.empty_cache()
    ctx.barrier()
    return out


def e2e_steps(ctx, prob, uvs, obj, x0, steps, pinned):
    """The same pass through the host-buffer C-ABI call: uvs, objpoints and x cross PCIe inside the
    timed region, S, b and the cost come back.  pinned=True: page-locked host tensors (the contract's
    e2e); pinned=False: the pageable numpy arrays a user of the reference holds."""
    torch, lib, check = ctx.torch, ctx.lib, ctx.native.check
    C = prob.C
    loss = ctx.native.LOSSES[LOSS]
    if pinned:
        keep = [torch.from_numpy(uvs).pin_memory(), torch.from_numpy(np.ascontiguousarray(obj)).pin_memory(),
                torch.from_numpy(x0).pin_memory(), torch.empty(144 * C * C, dtype=torch.float64).pin_memory(),
                torch.empty(12 * C, dtype=torch.float64).pin_memory(), torch.empty(1, dtype=torch.float64).pin_memory()]
        ptrs = [ctypes.c_void_p(t.data_ptr()) for t in keep]
        sizes = [t.numel() * 8 for t in keep]
    else:
        keep = [np.ascontiguousarray(uvs), np.ascontiguousarray(obj), np.ascontiguousarray(x0),
                np.empty(144 * C * C), np.empty(12 * C), np.empty(1)]
        ptrs = [a.ctypes.data_as(ctypes.c_void_p) for a in keep]
        sizes = [a.nbytes for a in keep]

    def step():
        check(lib.mcba_build_reduced_host(prob._h, ptrs[0], ptrs[1], ptrs[2], LAMBDA, loss, 1.0, ptrs[3], ptrs[4], ptrs[5]))

    for _ in range(2):
        step()
    ctx.barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    f0.record(prob.stream)
    for _ in range(steps):
        step()
    f1.record(prob.stream)
    ctx.barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    # every call ends with a host synchronisation (the outputs are host buffers), so the event time and
    # the host clock bracket the same work; the larger of the two is reported
    ms = max(f0.elapsed_time(f1), wall_ms if ctx.world == 1 else 0.0)
    return ms, sum(sizes[:3]), sum(sizes[3:])


def api_converge(ctx, scene, repeats=3):
    """The public call a user of the reference makes: pageable numpy arrays in, calibration out.
    Under torchrun every rank makes the same call and the frames are sharded inside it."""
    import multicam_calibration_b200 as mcc
    out = []
    for _ in range(repeats):    # the first call allocates the cached device problem (and, N > 1, its communicator)
        np.random.seed(0)
        ctx.barrier()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            *_, use, r = mcc.bundle_adjust(*scene.init_args(), n_frames=None, verbose=0)
        dt = time.perf_counter() - t0
        out.append((ctx.max_over_ranks([dt])[0], r, len(use)))
    dt, r, n_use = min(out, key=lambda t: t[0])
    return {"wall_ms": dt * 1e3, "first_call_ms": out[0][0] * 1e3, "device_ms": r.solve_ms, "iterations": r.iterations,
            "nfev": r.nfev, "status": r.status, "rms_px": r.rms, "cost": r.cost, "frames_used": n_use,
            "frames_total": int(scene.uvs.shape[1]), "n_gpus": ctx.world,
            "collective": r.get("collective") if ctx.world > 1 else None,
            "call": "multicam_calibration_b200.bundle_adjust(uvs, extrinsics, intrinsics, objpoints, poses, n_frames=None): "
                    "pageable numpy in, frame selection + upload + LM solve, calibration out"
                    + ("; every rank uploads and solves only its frames" if ctx.world > 1 else "")}


def measure_problem(ctx, cams, frames, scaling, steps, warmup, sampler=False, parity=False, converge=True, e2e=True,
                    keep_outputs=False):
    """One workload end to end on every rank: sharded problem, optional multi-GPU parity, timed
    device-resident steps, e2e through host buffers, LM time-to-converge.  keep_outputs: out["outputs"]
    holds what the last timed step computed (S, b, g_cam, cost, and the full gradient [g_cam | g_pose]
    of this rank's frames)."""
    from multicam_calibration_b200.engine import BAProblem
    torch = ctx.torch
    sc, uvs, x0 = local_scene(ctx, cams, frames, scaling)
    n_obs_local = int((~np.isnan(uvs).any(-1)).sum())
    prob = BAProblem(uvs, sc.objpoints, device=ctx.local, comm=ctx.comm())
    out = {"scene": sc, "frames_local": int(uvs.shape[1]), "n_obs_local": n_obs_local}
    out["collective"] = None if ctx.world == 1 else ("peer" if getattr(prob, "peer_memory", False) else "nccl")
    if parity and ctx.world > 1:
        out["parity"] = multi_gpu_parity(ctx, prob, uvs, sc.objpoints, x0)
    with torch.cuda.device(ctx.local), torch.cuda.stream(prob.stream):
        d_x = torch.as_tensor(x0).cuda()
        ms, per, launches, clocks, outputs = timed_steps(ctx, prob, d_x, steps, warmup,
                                                         ctx.local if (sampler and ctx.rank == 0) else None, keep_outputs)
        if keep_outputs:   # the gradient of the last evaluation, before e2e / converge evaluate again
            outputs["gradient"] = prob.gradient()
            out["outputs"] = outputs
        out["ms"] = ctx.max_over_ranks([ms])[0]
        out["kernels_ms"] = per                      # rank 0's launches
        out["kernels_ms_max"] = ctx.max_over_ranks(per)
        out["clocks"] = clocks
        n_obs_total, launches_total = ctx.sum_over_ranks([n_obs_local, launches])
        out["n_obs_total"], out["launches"] = int(n_obs_total), int(launches_total)
        if e2e:
            n_e2e = max(3, min(steps, 10))
            ms_p, h2d, d2h = e2e_steps(ctx, prob, uvs, sc.objpoints, x0, n_e2e, pinned=True)
            ms_q, _, _ = e2e_steps(ctx, prob, uvs, sc.objpoints, x0, n_e2e, pinned=False)
            ms_p, ms_q = ctx.max_over_ranks([ms_p, ms_q])
            out["e2e"] = {"steps": n_e2e, "ms_pinned": ms_p / n_e2e, "ms_pageable": ms_q / n_e2e, "h2d": h2d, "d2h": d2h}
        if converge:
            prob.set_observations(uvs, sc.objpoints)
            prob.solve(x0, verbose=0, max_nfev=3)          # warm-up: loads every kernel variant the LM loop uses
            ctx.barrier()
            t0 = time.perf_counter()
            _, res = prob.solve(x0, verbose=0)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            _, res_t = prob.solve(x0, ftol=1e-10, xtol=1e-10, verbose=0)
            dev_ms, tight_ms = ctx.max_over_ranks([res.solve_ms, res_t.solve_ms])
            out["converge"] = {"device_ms": dev_ms, "wall_s": wall, "iterations": res.iterations, "nfev": res.nfev,
                               "status": res.status, "rms_px": res.rms, "cost": res.cost, "tol": "ftol=1e-4 (reference default)",
                               "tight": {"device_ms": tight_ms, "iterations": res_t.iterations, "rms_px": res_t.rms,
                                         "cost": res_t.cost, "optimality": res_t.optimality, "tol": "ftol=xtol=1e-10"}}
    prob.close()
    torch.cuda.empty_cache()
    return out


def roofline_block(m, frames_local, peaks, peak_kind, fp64_peak):
    k2_ms = m["kernels_ms"][0]
    alg_bytes = 16.0 * m["n_obs_local"] + 48.0 * frames_local          # SURVEY.md 8(d): 16 B/obs + 48 B/frame (rank 0's launch)
    achieved = alg_bytes / (k2_ms * 1e-3) / 1e9
    fma_rate = ALG_FMA_PER_OBS * m["n_obs_local"] / (k2_ms * 1e-3)     # DESIGN.md section 4
    traffic = None
    prof_json = os.path.join(ROOT, "profiles", "k2_frames_traffic.json")
    if os.path.exists(prof_json):
        traffic = json.load(open(prof_json)).get("dram_bytes_per_launch")
    return {"bound": "hbm", "kernel": "k2p_kernel (residual + analytic Jacobian + robust weights + A_cf accumulation)",
            "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peak_kind,
            "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": k2_ms,
            "fp64_pipe": {"achieved": fma_rate * 2e-12, "peak": fp64_peak * 2e-12, "unit": "TFLOP/s",
                          "frac": fma_rate / fp64_peak if fp64_peak else None, "fma_per_obs": ALG_FMA_PER_OBS,
                          "peak_source": "DFMA loop timed in this run (mcba_measure_fp64_peak)"},
            "note": "the kernel does ~250 FP64 FMAs per 16-byte observation: it is bound by the FP64 "
                    "pipe (fp64_pipe.frac), not by HBM; frac is the HBM figure the contract asks for"}


DUMP_LIMIT_BYTES = 63_000_000     # under 64 MB with room for the .npy headers


def dump_outputs(path, outputs):
    """Write each output as `path/<name>.npy` (float64), smallest first.  An output that does not fit in
    what is left of DUMP_LIMIT_BYTES is replaced by a fixed, seeded sample of its entries, with their
    flat indices in `<name>_index.npy`, so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    left = DUMP_LIMIT_BYTES
    for name, a in sorted(outputs.items(), key=lambda kv: kv[1].size):
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > left:
            idx = np.sort(np.random.default_rng(0).choice(a.size, left // 16, replace=False))
            a = a.ravel()[idx]
            np.save(os.path.join(path, name + "_index.npy"), idx.astype(np.float64))
            left -= a.nbytes
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes


def kernels_block(per):
    return {"k2p_corner_walk": per[0], "k2c_frame_schur": per[1], "k2_syrk": per[2], "finalize_allreduce": per[3]}


# ---------------------------------------------------------------------------------------------
# extras (N = 1): BASELINE configs[4] and the K1 residual kernel
# ---------------------------------------------------------------------------------------------
def _timed(torch, fn, reps=10, warm=3, stream=None):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def _wall(fn, reps=3):
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best


def extra_geometry(ctx, peaks, peak_kind, points, cpu):
    """BASELINE configs[4]: geometry.triangulate (geometry.py:361-433) and project_points (:277-325) of
    `points` keypoints across 6 cameras.  Device-resident kernel time with its roofline, e2e through the
    public numpy functions (pageable arrays in and out), and the oracle port on a bounded sample."""
    import multicam_calibration_b200 as mcc
    from multicam_calibration_b200.synthetic import make_keypoints
    torch, lib, check, dev = ctx.torch, ctx.lib, ctx.native.check, ctx.local
    all_uvs, ext, intr, pts = make_keypoints(points, 6, sigma=0.3, p_missing=0.2, seed=0)
    P, C = points, 6
    Ks = np.ascontiguousarray(np.stack([K for K, _ in intr]))
    dist5 = np.ascontiguousarray(np.stack([np.asarray(d, dtype=np.float64) for _, d in intr]))
    dist2 = np.ascontiguousarray(dist5[:, :2])
    ext = np.ascontiguousarray(ext)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    uv = np.ascontiguousarray(np.stack(all_uvs))
    d_obs = torch.as_tensor(uv).cuda()
    d_pts = torch.as_tensor(pts).cuda()
    d_out = torch.empty((P, 3), dtype=torch.float64, device="cuda")
    d_uv = torch.empty((C, P, 2), dtype=torch.float64, device="cuda")
    hbm = peaks["hbm_gbs"]

    def tri():
        check(lib.mcba_triangulate(dev, stream, ctypes.c_void_p(d_obs.data_ptr()), C, P, vp(ext), vp(Ks), vp(dist5),
                                   ctypes.c_void_p(d_out.data_ptr())))

    def proj():
        check(lib.mcba_project_points_multi(dev, stream, ctypes.c_void_p(d_pts.data_ptr()), P, C, vp(ext), vp(Ks), vp(dist2),
                                            ctypes.c_void_p(d_uv.data_ptr())))

    out = {"workload": f"{P} keypoints x {C} cameras, sigma=0.3 px, 20% missing views (BASELINE.json configs[4])"}
    ms = _timed(torch, tri)
    tri_bytes = P * (C * 16 + 24)              # 16 B per view read + 24 B per point written
    res = d_out.cpu().numpy()
    ok = np.isfinite(res).all(1)
    wall = _wall(lambda: mcc.triangulate(all_uvs, list(ext), intr))
    blk = {"metric": "points/s geometry.triangulate", "value": P / (ms * 1e-3), "unit": "points/s", "ms": ms,
           "roofline": {"bound": "hbm", "kernel": "triangulate_kernel", "achieved": tri_bytes / (ms * 1e-3) / 1e9, "peak": hbm,
                        "unit": "GB/s", "frac": tri_bytes / (ms * 1e-3) / 1e9 / hbm, "traffic": None, "peak_source": peak_kind,
                        "algorithmic_bytes_per_launch": tri_bytes,
                        "note": "15 view pairs x (4x4 DLT null vector by Householder QR + inverse iteration) per point: FP64 bound"},
           "e2e": {"value": P / wall, "unit": "points/s", "ms": wall * 1e3, "h2d_bytes_per_step": int(uv.nbytes),
                   "d2h_bytes_per_step": int(res.nbytes), "call": "multicam_calibration_b200.triangulate(list of (P,2) numpy, extrinsics, intrinsics)"},
           "median_error_vs_truth": float(np.median(np.linalg.norm(res[ok] - pts[ok], axis=1))),
           "fraction_triangulated": float(ok.mean())}
    if cpu:
        from oracle import np_oracle as orc
        ns = 5000
        t0 = time.perf_counter()
        ref = orc.triangulate([u[:ns] for u in all_uvs], list(ext), intr)
        dt = time.perf_counter() - t0
        good = np.isfinite(ref).all(1) & ok[:ns]
        blk["cpu_baseline"] = {"value": ns / dt, "unit": "points/s", "cores": 1, "kind": "port",
                               "sample": f"first {ns} keypoints x {C} views through the oracle's restatement of geometry.triangulate "
                                         f"(undistort, all-pairs DLT, per-point nanmedian loop), {dt:.2f} s"}
        blk["max_abs_diff_vs_oracle_sample"] = float(np.abs(res[:ns][good] - ref[good]).max())
    out["triangulate"] = blk

    ms = _timed(torch, proj)
    pr_bytes = P * 24 + C * P * 16
    wall = _wall(lambda: mcc.project_points_multi(pts, list(ext), intr))
    blk = {"metric": "views/s geometry.project_points (all cameras of the rig in one pass)", "value": C * P / (ms * 1e-3),
           "unit": "views/s", "ms": ms,
           "roofline": {"bound": "hbm", "kernel": "project_points_multi_kernel", "achieved": pr_bytes / (ms * 1e-3) / 1e9, "peak": hbm,
                        "unit": "GB/s", "frac": pr_bytes / (ms * 1e-3) / 1e9 / hbm, "traffic": None, "peak_source": peak_kind,
                        "algorithmic_bytes_per_launch": pr_bytes},
           "e2e": {"value": C * P / wall, "unit": "views/s", "ms": wall * 1e3, "h2d_bytes_per_step": int(pts.nbytes),
                   "d2h_bytes_per_step": int(C * P * 16), "call": "multicam_calibration_b200.project_points_multi(points, extrinsics, intrinsics)"}}
    if cpu:
        from oracle import np_oracle as orc
        ns = 200_000
        t0 = time.perf_counter()
        for c in range(C):
            orc.project_points(pts[:ns], ext[c], Ks[c], dist2[c])
        dt = time.perf_counter() - t0
        blk["cpu_baseline"] = {"value": C * ns / dt, "unit": "views/s", "cores": 1, "kind": "port",
                               "sample": f"first {ns} keypoints x {C} cameras through the oracle's project_points, {dt:.2f} s"}
    out["project_points"] = blk
    return out


def extra_k1(ctx, scene, peaks, peak_kind, cpu):
    """K1: residuals(params, uvs, objpoints) (bundle_adjustment.py:66-98) on the main workload."""
    import multicam_calibration_b200 as mcc
    from multicam_calibration_b200.engine import BAProblem
    torch, lib, check = ctx.torch, ctx.lib, ctx.native.check
    prob = BAProblem(scene.uvs, scene.objpoints, device=ctx.local)
    x0 = scene.x0()
    hbm = peaks["hbm_gbs"]
    with torch.cuda.device(ctx.local), torch.cuda.stream(prob.stream):
        d_x = torch.as_tensor(x0).cuda()
        m = prob.n_residuals
        d_r = torch.empty(m, dtype=torch.float64, device="cuda")
        ms = _timed(torch, lambda: check(lib.mcba_residuals(prob._h, ctypes.c_void_p(d_x.data_ptr()), ctypes.c_void_p(d_r.data_ptr()))),
                    stream=prob.stream)
    prob.close()
    n_obs = scene.n_obs
    slots = int((~np.isnan(scene.uvs).all((-1, -2))).sum()) * scene.uvs.shape[2]   # slots of the (camera, frame) rows with a detection
    alg = 32.0 * n_obs + 48.0 * scene.uvs.shape[1]          # SURVEY 8(d): 16 B read + 16 B written per finite observation, + pose
    mcc.residuals(x0, scene.uvs, scene.objpoints)           # allocates the cached problem
    wall = _wall(lambda: mcc.residuals(x0, scene.uvs, scene.objpoints))
    blk = {"metric": "obs/s residuals (K1, materialised)", "value": n_obs / (ms * 1e-3), "unit": UNIT, "ms": ms,
           "roofline": {"bound": "hbm", "kernel": "residual_chunks_kernel", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm,
                        "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / hbm, "traffic": None, "peak_source": peak_kind,
                        "algorithmic_bytes_per_launch": alg,
                        "touched_bytes_per_launch": 16.0 * slots + 8.0 * m,
                        "touched_frac": (16.0 * slots + 8.0 * m) / (ms * 1e-3) / 1e9 / hbm,
                        "note": "algorithmic = 32 B per finite observation; touched = the slots of every (camera, frame) row with at "
                                "least one detection (rows of a camera that did not see the board are skipped) + the residuals"},
           "e2e": {"value": n_obs / wall, "unit": UNIT, "ms": wall * 1e3, "h2d_bytes_per_step": int(scene.uvs.nbytes + x0.nbytes),
                   "d2h_bytes_per_step": int(8 * m), "call": "multicam_calibration_b200.residuals(params, uvs, objpoints), pageable numpy"}}
    mcc.release_device_memory()
    if cpu:
        from multicam_calibration_b200.synthetic import make_scene
        from oracle import np_oracle as orc
        s = make_scene(scene.uvs.shape[0], 5000, sigma=SIGMA, p_missing_view=P_MISSING, seed=0)
        xs = s.x0()
        t0 = time.perf_counter()
        for _ in range(3):
            orc.residuals(xs, s.uvs, s.objpoints)
        dt = (time.perf_counter() - t0) / 3
        blk["cpu_baseline"] = {"value": s.n_obs / dt, "unit": UNIT, "cores": 1, "kind": "port",
                               "sample": f"{s.uvs.shape[0]} cams x 5000 frames ({s.n_obs} obs) through the oracle's residuals, {dt:.3f} s per call"}
    return blk


def run_engine(args):
    ctx = Ctx(args)
    torch, world, rank = ctx.torch, ctx.world, ctx.rank
    cfg = CONFIGS[args.config]
    cams = args.cams or cfg["cams"]
    if args.frames:
        frames = args.frames
    elif args.scaling == "weak":
        frames = cfg["frames"] // cfg["quoted_gpus"]      # per GPU
    else:
        frames = cfg["frames"]                            # total
    main = measure_problem(ctx, cams, frames, args.scaling, args.steps, args.warmup, sampler=True, parity=True,
                           keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, main.pop("outputs"))

    # ---- the public call: numpy arrays in, calibration out (N > 1: the 50k-frame problem sharded inside the call)
    import multicam_calibration_b200 as mcc
    from multicam_calibration_b200.synthetic import make_scene
    if world == 1 or args.scaling == "strong":
        api_scene = main["scene"]
    else:
        api_scene = make_scene(cams, frames, sigma=SIGMA, p_missing_view=P_MISSING, seed=0, shard=0)
    api = api_converge(ctx, api_scene)
    api_same = None
    if world == 1 and not args.no_cpu_baseline:
        api_same = api_converge(ctx, make_scene(cams, CPU_CONVERGE_FRAMES, sigma=SIGMA, p_missing_view=P_MISSING, seed=0))
    mcc.release_device_memory()
    torch.cuda.empty_cache()

    # ---- strong scaling of the same problem (weak runs at N > 1): `frames` in total, split over the ranks
    strong = None
    if world > 1 and args.scaling == "weak" and not args.no_extras:
        s = measure_problem(ctx, cams, frames, "strong", args.steps, args.warmup, e2e=False)
        ms_step = s["ms"] / args.steps
        per = s["kernels_ms_max"]
        strong = {"workload": workload_name(cams, frames, "strong", world, cfg["name"]), "frames_total": frames,
                  "frames_per_gpu": s["frames_local"], "observations_total": s["n_obs_total"],
                  "ms_per_step": ms_step, "value": s["n_obs_total"] / (ms_step * 1e-3), "unit": UNIT,
                  "kernels_ms": kernels_block(per), "collective": s["collective"],
                  "limiter": {"compute_ms": per[0] + per[1] + per[2], "finalize_allreduce_ms": per[3],
                              "note": "max over ranks per kernel; the reduced-system sum (finalize + all-reduce) does not shrink "
                                      "with the shard, the three compute kernels do"},
                  "ba_converge": s["converge"],
                  "efficiency_note": "strong efficiency at N GPUs = value / (N x the N=1 line's value)"}

    # ---- extras: configs[3] shard per GPU; configs[4] and K1 at N = 1
    extra = {}
    if not args.no_extras:
        if args.config != 3:
            c3 = CONFIGS[3]
            per_gpu = c3["frames"] // c3["quoted_gpus"]
            m3 = measure_problem(ctx, c3["cams"], per_gpu, "weak", max(5, min(args.steps, 30)), args.warmup, e2e=False)
            n3 = max(5, min(args.steps, 30))
            ms3 = m3["ms"] / n3
            extra["config3"] = {"workload": workload_name(c3["cams"], per_gpu, "weak", world, c3["name"] + (
                                    ": this is the full configuration" if world == c3["quoted_gpus"] else f": {world} of its 8 shards")),
                                "n_gpus": world, "frames_total": per_gpu * world, "observations_total": m3["n_obs_total"],
                                "ms_per_step": ms3, "value": m3["n_obs_total"] / (ms3 * 1e-3), "unit": UNIT, "steps": n3,
                                "kernels_ms": kernels_block(m3["kernels_ms"]), "collective": m3["collective"],
                                "ba_converge": m3["converge"]}
        if world == 1:
            peaks, peak_kind = measured_peaks()
            extra["config5"] = extra_geometry(ctx, peaks, peak_kind, args.points, not args.no_cpu_baseline)
            extra["k1_residuals"] = extra_k1(ctx, main["scene"], peaks, peak_kind, not args.no_cpu_baseline)

    fp64_peak = ctypes.c_double(0.0)
    line = None
    if rank == 0:
        ctx.native.check(ctx.lib.mcba_measure_fp64_peak(ctx.local, ctypes.byref(fp64_peak)))
        peaks, peak_kind = measured_peaks()
        ms_step = main["ms"] / args.steps
        value = main["n_obs_total"] / (ms_step * 1e-3)
        e = main["e2e"]
        collective = {None: "none (1 GPU)", "peer": "one kernel over NVLink peer memory (CUDA IPC, mcba_peer.cu)",
                      "nccl": "ncclAllReduce"}[main["collective"]]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(cams, frames, args.scaling, world, cfg["name"] if not (args.cams or args.frames) else "custom"),
                       "frames_per_gpu": main["frames_local"], "observations_total": main["n_obs_total"],
                       "sharding": f"frames x{world}; one sum of the packed reduced camera system per step",
                       "collective": collective,
                       "l2": "per step 168 MB of observations are read, 151 MB of hand-off and 173 MB of Z are written and "
                             "re-read (6 cameras x 50k frames): the working set exceeds the 126 MB L2, no flush needed",
                       "loss": LOSS, "lambda": LAMBDA},
            "clocks": main["clocks"],
            "roofline": roofline_block(main, main["frames_local"], peaks, peak_kind, fp64_peak.value),
            "kernels_ms": kernels_block(main["kernels_ms"]),
            "e2e": {"value": main["n_obs_total"] / (e["ms_pinned"] * 1e-3), "unit": UNIT, "h2d_bytes_per_step": e["h2d"],
                    "d2h_bytes_per_step": e["d2h"], "ms_per_step": e["ms_pinned"], "steps": e["steps"],
                    "call": "mcba_build_reduced_host (pinned host uvs, objpoints, x -> S, b, cost); at one rank the observations cross PCIe in 8 frame ranges, each evaluated while the next is in flight",
                    "pageable": {"value": main["n_obs_total"] / (e["ms_pageable"] * 1e-3), "ms_per_step": e["ms_pageable"],
                                 "call": "the same call on pageable numpy arrays (staged through mcba_upload's bounce buffers)"}},
            "gpu_launches": main["launches"],
            "ba_converge": dict(main["converge"], api=api),
        }
        if world > 1:
            line["kernels_ms_max_over_ranks"] = kernels_block(main["kernels_ms_max"])
            line["multi_gpu_parity"] = main.get("parity")
            if strong:
                line["strong"] = strong
        if extra:
            line["extra"] = extra
        if world == 1 and not args.no_cpu_baseline:
            base = cpu_baseline(steps=2, warmup=0, converge_frames=CPU_CONVERGE_FRAMES, cams=cams)
            line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "reference_recorded")}
            conv = base["converge"]
            conv["engine_same_sample"] = api_same
            line["cpu_baseline"]["converge"] = conv
    if world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()
    return line


def _quiet_stdout():
    """Route everything libraries print on fd 1 (e.g. NCCL's version banner) to stderr and return a
    file object on the real stdout: the contract is ONE JSON line on stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configs[k] preset (default 2)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the preset's frames per GPU (default); strong: the preset's frames in total, split over the GPUs")
    ap.add_argument("--frames", type=int, default=0, help="override the preset's frame count (per GPU: weak, total: strong)")
    ap.add_argument("--cams", type=int, default=0, help="override the preset's camera count")
    ap.add_argument("--points", type=int, default=1_000_000, help="keypoints of the configs[4] extra")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only: no strong / configs[3] / configs[4] / K1 blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one computed (rank 0: S, b, g_cam, cost and the "
                         "gradient [g_cam | g_pose] of its frames) as DIR/<name>.npy, float64, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs applies to the engine arm only")
    args.warmup = max(args.warmup, 3) if args.impl == "engine" else args.warmup
    out = _quiet_stdout()
    line = run_reference(args) if args.impl == "reference" else run_engine(args)
    if line is not None:
        out.write(json.dumps(line) + "\n")
        out.flush()


if __name__ == "__main__":
    main()
