"""Opcode histogram of the hot kernels in libmcba.so (cuobjdump -sass; runs without a GPU):

    python scripts/sass_histogram.py > profiles/r02_sass_opcodes.json

Per kernel: total instructions and the counts of the opcodes that show what the kernel is made of --
FP64 vector (DFMA / DMUL / DADD), FP64 tensor (DMMA), bulk asynchronous copies and their barriers
(UBLKCP, SYNCS), memory (LDG / STG / LDS / STS / LDL / STL), shuffles, MUFU seeds, barriers."""
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "multicam_calibration_b200", "libmcba.so")
HOT = ["k2p_kernel", "k2c_ring_kernel", "k2c_pose_kernel", "k2c_rows_kernel", "sum_children_kernel", "k2_syrk_kernel", "finalize_kernel", "solve_reduced_kernel",
       "backsub_kernel", "sum_scalars_kernel", "peer_allreduce_kernel", "residual_chunks_kernel", "cost_kernel",
       "triangulate_kernel", "project_points_multi_kernel", "homography_transfer_kernel", "tile_observations_kernel",
       "frame_errors_kernel"]
SHOW = ["DFMA", "DMUL", "DADD", "DMMA", "DSETP", "MUFU", "UBLKCP", "SYNCS", "LDG", "STG", "LDS", "STS", "LDL", "STL", "SHFL",
        "BAR", "ATOMG", "RED", "MEMBAR", "FSEL", "IMAD"]


def main():
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    out, name, counts = {}, None, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                out[name] = counts
            name, counts = m.group(1), collections.Counter()
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and name:
            counts[m.group(1)] += 1
    if name:
        out[name] = counts
    demangle = subprocess.run(["cu++filt"] + list(out), capture_output=True, text=True).stdout.splitlines()
    names = dict(zip(out, demangle)) if len(demangle) == len(out) else {k: k for k in out}
    report = {}
    for mangled, counts in out.items():
        pretty = re.sub(r"\((?:int|bool)\)", "", names[mangled]).split("(")[0].replace("void ", "")
        if not any(h in pretty for h in HOT):
            continue
        rec = {"instructions": int(sum(counts.values()))}
        rec.update({op: int(counts[op]) for op in SHOW if counts.get(op)})
        report[pretty] = rec
    json.dump({"library": "multicam_calibration_b200/libmcba.so (sm_100a)", "kernels": dict(sorted(report.items()))},
              sys.stdout, indent=1)
    print()


if __name__ == "__main__":
    main()
