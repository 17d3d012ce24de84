#!/usr/bin/env python3
"""Throughput of the closed-form inverse kinematics (IkEngine.analytic_ik / analytic_ik_device, csrc/analytic.cu
analytic_ik_kernel), and AnalyticInverseKinematics.ikine_pose against FabrikInverseKinematics.ikine_pose.  Prints one
JSON line.

Device-resident, per kind (poses: 2 branches, positions with one pitch per row: 4 branches) and dtype (inputs and
angles of the same dtype, status written): rows sized so that inputs and outputs are at least 4x the 126 MB L2; kernel
time from CUDA events (median of --reps after --warmup); rows/s, bytes moved per row and GB/s, against a torch `fill_`
of the output's size timed the same way in the same process.  The host path (`analytic_ik` into NumPy arrays): rows/s.

ikine_pose on the workloads of tools/pose_bench.py (r07): (a) poses of random angles inside the workspace box and (d)
their positions with uniformly random rotations (generally no pose of this 4-joint arm): rows/s of the whole call (one
upload, seed, refinement, one download), the converged fraction, mean / p99 steps and percentiles of the final weighted
errors, for the closed-form seed and the FABRIK seed."""
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
from pose_bench import L2_BYTES, TOL, poses, random_rotations  # noqa: E402


def run_device(eng, fk, args):
    import torch
    rows = []
    for kind, branches in (("pose", 2), ("position", 4)):
        for dtype in (torch.float32, torch.float64):
            size = 4 if dtype == torch.float32 else 8
            b_in = (16 if kind == "pose" else 4) * size
            b_out = branches * 4 * size + 4
            n = int(min(args.max_rows, -(-4 * L2_BYTES // (b_in + b_out))))
            g = torch.Generator(device="cuda").manual_seed(3)
            th = (torch.rand(n, 4, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * np.pi
            T = fk.fkine_device(th)[:, 3].contiguous()
            if kind == "pose":
                x, pitch = T.to(dtype), None
            else:
                x, pitch = T[:, :3, 3].contiguous().to(dtype), th[:, 1:].sum(dim=1).to(dtype)
            del T, th
            out = torch.empty((n, branches, 4), dtype=dtype, device="cuda")
            st = torch.empty(n, dtype=torch.int32, device="cuda")
            t = event_seconds(lambda: eng.analytic_ik_device(x, pitch, out, st), args.reps, args.warmup)
            flat = out.view(-1)
            t_fill = event_seconds(lambda: flat.fill_(1.0), args.reps, args.warmup)
            gbs = n * (b_in + b_out) / t / 1e9
            rows.append({"kind": kind, "dtype": str(dtype).replace("torch.", ""), "rows": n, "bytes_per_row_in": b_in,
                         "bytes_per_row_out": b_out, "kernel_s": t, "rows_per_s": n / t, "achieved_gb_s": gbs,
                         "fill_of_output_gb_s": n * branches * 4 * size / t_fill / 1e9,
                         "fraction_of_fill_gb_s": gbs / (n * branches * 4 * size / t_fill / 1e9)})
            del x, pitch, out, st, flat
            torch.cuda.empty_cache()
    return rows


def run_host(eng, fk, args):
    import torch
    res = []
    n = args.host_rows
    th = (torch.rand(n, 4, device="cuda", dtype=torch.float64) * 2 - 1) * np.pi
    T = fk.fkine_device(th)[:, 3].contiguous().cpu().numpy()
    phi = th[:, 1:].sum(dim=1).cpu().numpy()
    for kind, x, pitch in (("pose", T, None), ("position", np.ascontiguousarray(T[:, :3, 3]), phi)):
        eng.analytic_ik(x[: 1 << 16], None if pitch is None else pitch[: 1 << 16])  # warm-up
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            eng.analytic_ik(x, pitch)
            times.append(time.perf_counter() - t0)
        res.append({"kind": kind, "dtype": "float64", "rows": n, "seconds": float(np.median(times)),
                    "rows_per_s": n / float(np.median(times))})
    return res


def ikine_pose_stats(ik, Th, reps):
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out, its, err = ik.ikine_pose(Th, as_array=True, return_iterations=True, return_fk_error=True)
        times.append(time.perf_counter() - t0)
    conv = err <= TOL
    t = float(np.median(times))
    return {"rows": int(Th.shape[0]), "seconds": t, "rows_per_s": Th.shape[0] / t,
            "fraction_converged": float(conv.mean()), "mean_steps": float(its.mean()),
            "p99_steps": float(np.percentile(its, 99)), "max_steps": int(its.max()),
            "fraction_at_step_0": float((its == 0).mean()),
            "final_error_p50_p90_p99_max": [float(v) for v in np.percentile(err, [50, 90, 99, 100])]}


def run_ikine_pose(fk, args):
    from inversekinematicsann_b200.kinematics.inverse import AnalyticInverseKinematics, FabrikInverseKinematics
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    _, T = poses(fk, args.pose_rows, 11)
    Tr = random_rotations(T, 12)
    work = {"a_poses_of_random_angles": T.cpu().numpy(), "d_random_rotations": Tr.cpu().numpy()}
    del T, Tr
    solvers = {"analytic": AnalyticInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits),
               "fabrik": FabrikInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)}
    res = []
    for wname, Th in work.items():
        for sname, ik in solvers.items():
            ik.ikine_pose(Th[:4096])  # warm-up
            r = ikine_pose_stats(ik, Th, args.pose_reps)
            r.update({"workload": wname, "seed": sname})
            res.append(r)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--max-rows", type=int, default=1 << 27)
    ap.add_argument("--host-rows", type=int, default=1 << 22)
    ap.add_argument("--pose-rows", type=int, default=1 << 20)
    ap.add_argument("--pose-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    from inversekinematicsann_b200.kinematics.forward import ForwardKinematics
    from inversekinematicsann_b200.kinematics._shared import get_engine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    res = gpu_info()
    fk = ForwardKinematics(R.dh_matrix)
    eng = get_engine()
    res["device"] = run_device(eng, fk, args)
    res["host"] = run_host(eng, fk, args)
    res["ikine_pose"] = run_ikine_pose(fk, args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
