#!/usr/bin/env python3
"""Throughput of the batched arm Jacobian and manipulability (ForwardKinematics.jacobian_batch / manipulability,
the Jacobian kinds of csrc/fk.cu fk_transforms_kernel).  Prints one JSON line.

Workloads: {geometric, position} x {float32, float64}, the manipulability-only call in both dtypes, and fp64 geometric
with the manipulability beside it; angles seeded uniform in [-pi, pi].  Rows are sized so that angles plus outputs are
at least 4x the 126 MB L2, so every timed launch streams from and to HBM.

Per workload:
  - kernel time of `IkEngine.jacobian_device` from CUDA events after a warm-up (median of --reps), rows/s, bytes moved
    per row (angles in + outputs out) and the achieved GB/s;
  - the copy ceiling: a torch `fill_` of the outputs' size, timed the same way in the same process, and the kernel's
    fraction of it;
  - for reference, the fp64 joint origins (`fk_transforms_device`, what="joints") on the same rows: the FK chain with
    the fewest output bytes.
The alternative without this kernel: central differences over `fkine_device` (the device form of `fkine_batch`), eight
launches of all four matrices with theta_k +- h and the position columns differenced in torch, timed on the rows of the
fp64 geometric workload; its largest difference from the kernel's linear rows is recorded.  The host path
(`IkEngine.jacobian` into pinned memory) is timed for fp64 geometric and the fp64 manipulability."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fk_transforms_bench import event_seconds, gpu_info  # noqa: E402

L2_BYTES = 126 * 2 ** 20
TAIL = {"geometric": (6, 4), "position": (3, 4), None: ()}


def rows_for(b_row, max_rows):
    return int(min(max_rows, -(-4 * L2_BYTES // b_row)))


def run_device(args):
    import torch
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    rows = []
    cases = [(w, d, False) for w in ("geometric", "position") for d in (np.float32, np.float64)]
    cases += [(None, np.float32, True), (None, np.float64, True), ("geometric", np.float64, True)]
    for what, dtype, manip in cases:
        item = np.dtype(dtype).itemsize
        b_in = 4 * item
        b_jac = int(np.prod(TAIL[what])) * item if what else 0
        b_out = b_jac + (item if manip else 0)
        n = rows_for(b_in + b_out, args.max_rows)
        td = torch.float32 if dtype == np.float32 else torch.float64
        g = torch.Generator(device="cuda").manual_seed(1)
        ang = ((torch.rand(n, 4, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * np.pi).to(td)
        out = torch.empty((n,) + TAIL[what], dtype=td, device="cuda") if what else None
        w = torch.empty(n, dtype=td, device="cuda") if manip else None
        t = event_seconds(lambda: eng.jacobian_device(ang, out, what or "geometric", w), args.reps, args.warmup)
        fill = torch.empty(n * b_out // item, dtype=td, device="cuda")
        t_fill = event_seconds(lambda: fill.fill_(1.0), args.reps, args.warmup)
        del fill
        ang64 = ang.double()
        joints = torch.empty((n, 4, 3), dtype=torch.float64, device="cuda")
        t_joints = event_seconds(lambda: eng.fk_transforms_device(ang64, joints, "joints"), args.reps, args.warmup)
        del ang64, joints
        eng.stats_reset_torch()
        gbs = n * (b_in + b_out) / t / 1e9
        fill_gbs = n * b_out / t_fill / 1e9
        rows.append({
            "what": what or "manipulability only", "manipulability": manip, "dtype": np.dtype(dtype).name, "rows": n,
            "bytes_per_row_in": b_in, "bytes_per_row_out": b_out, "kernel_s": t, "rows_per_s": n / t,
            "achieved_gb_s": gbs, "fill_gb_s": fill_gbs, "fraction_of_fill": gbs / fill_gbs,
            "fk_joints_f64_rows_per_s_same_rows": n / t_joints,
        })
        del ang, out, w
    return rows


def run_central_differences(args):
    """The user's alternative on the rows of the fp64 geometric workload."""
    import torch
    from inversekinematicsann_b200.kinematics._shared import get_engine
    from inversekinematicsann_b200.kinematics.forward import ForwardKinematics
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    eng = get_engine()
    fk = ForwardKinematics(R.dh_matrix)
    n = rows_for(32 + 192, args.max_rows)
    h = 1e-6
    g = torch.Generator(device="cuda").manual_seed(1)
    ang = (torch.rand(n, 4, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * np.pi
    plus, minus = torch.empty_like(ang), torch.empty_like(ang)
    mp = torch.empty((n, 4, 4, 4), dtype=torch.float64, device="cuda")
    mm = torch.empty_like(mp)
    lin = torch.empty((n, 3, 4), dtype=torch.float64, device="cuda")

    def differences():
        for k in range(4):
            plus.copy_(ang)
            minus.copy_(ang)
            plus[:, k] += h
            minus[:, k] -= h
            fk.fkine_device(plus, mp)
            fk.fkine_device(minus, mm)
            torch.sub(mp[:, 3, :3, 3], mm[:, 3, :3, 3], out=lin[:, :, k])
        lin.div_(2 * h)

    t = event_seconds(differences, args.reps, args.warmup)
    jac = torch.empty((n, 6, 4), dtype=torch.float64, device="cuda")
    eng.jacobian_device(ang, jac, "geometric")
    err = float((lin - jac[:, :3]).abs().max())
    eng.stats_reset_torch()
    return {"rows": n, "h": h, "fk_launches_per_call": 8, "seconds": t, "rows_per_s": n / t,
            "max_abs_difference_from_kernel": err}


def run_host(args):
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    res = []
    for what, manip in (("geometric", False), (None, True)):
        b_out = 192 if what else 8
        n = rows_for(32 + b_out, args.max_rows)
        ang = np.random.default_rng(2).uniform(-np.pi, np.pi, (n, 4))
        out = eng.pinned_empty((n, 6, 4), np.float64) if what else None
        eng.jacobian(ang[: 1 << 16], what, manipulability=manip, out=out[: 1 << 16] if what else None)  # warm-up
        t0 = time.perf_counter()
        eng.jacobian(ang, what, manipulability=manip, out=out)
        t_host = time.perf_counter() - t0
        res.append({"what": what or "manipulability only", "dtype": "float64", "rows": n, "host_s": t_host,
                    "host_rows_per_s": n / t_host, "host_d2h_gb_s": n * b_out / t_host / 1e9})
        del ang, out
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--max-rows", type=int, default=1 << 27)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    res = gpu_info()
    res["workloads"] = run_device(args)
    res["central_differences_over_fkine"] = run_central_differences(args)
    res["host"] = run_host(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
