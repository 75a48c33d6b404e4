"""torchrun --nproc-per-node N scripts/fixed_params_multigpu_check.py [frames]: the frame-sharded solve with camera
parameters held (intrinsics and camera 0's extrinsics) against the single-GPU masked solve of the same problem
(run by tests/test_fixed_parameters.py)."""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
import multicam_calibration_b200 as mcc
from multicam_calibration_b200 import distributed
from multicam_calibration_b200.synthetic import make_scene

local = int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
rank, world = dist.get_rank(), dist.get_world_size()
F = int(sys.argv[1]) if len(sys.argv) > 1 else 997
sc = make_scene(6, F, sigma=0.3, p_missing_view=0.2, seed=5)
x0 = sc.x0()
fixed = np.zeros((6, 12), dtype=bool)
fixed[:, :6] = True
fixed[0, 6:] = True
a, b = distributed.shard_bounds(F, world, rank)
x_loc = distributed.split_params(x0, 6, a, b)
kw = dict(ftol=1e-12, xtol=1e-12, verbose=0)
x, res = distributed.solve_sharded(sc.uvs[:, a:b], sc.objpoints, x_loc, fixed=fixed, **kw)
ok = True
if rank == 0:
    xs, rs = mcc.BAProblem(sc.uvs, sc.objpoints, device=local).solve(x0, fixed=fixed, **kw)
    d_cost = abs(rs.cost - res.cost) / rs.cost
    d_x = np.abs(xs - x).max()
    held = np.array_equal(x[:72][fixed.ravel()], x0[:72][fixed.ravel()])
    ok = d_cost < 1e-9 and d_x < 1e-6 and held and res.nfev == rs.nfev
    print(f"world={world} sharded: cost {res.cost:.9f} nfev {res.nfev} | single: cost {rs.cost:.9f} nfev {rs.nfev} | "
          f"rel dcost {d_cost:.2e} max|dx| {d_x:.2e} held entries unchanged {held} collective={res.collective}")
    print("FIXED_MULTIGPU_OK" if ok else "FIXED_MULTIGPU_FAIL")
flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
dist.broadcast(flag, src=0)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1.0 else 1)
