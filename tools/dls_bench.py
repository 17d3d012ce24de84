#!/usr/bin/env python3
"""Throughput and convergence of the damped-least-squares refinement (InverseKinematics.refine / refine_device,
csrc/fk.cu dls_refine_kernel).  Prints one JSON line.

Targets are cube_random (the engine's generator) over the whole workspace box (0,-6,-3)+(6,12,9); "reachable" keeps
those within 6 m - 1e-6 of the shoulder (0, 0, 2), "out of reach" those beyond 6 m + 1e-3.  Rows are sized so that
targets, seeds, angles, iterations and errors (100 B per fp64 row) are at least 4x the 126 MB L2.  Every workload is
fp64 and device-resident, tol 1e-9:
  (a) FABRIK-seeded (`fabrik_solve_device`, tol 1e-3) refinement of reachable targets;
  (b) ANN-seeded (models/roboarm_b200_r01, float32 predictions widened) refinement of the same targets;
  (c) one broadcast seed, the DH table's seed row [0, pi/2, 0, 0] (the stretched arm, where Jv is rank-deficient);
  (d) FABRIK-seeded, half of the targets out of reach (these run to max_iter).
Per workload: kernel time from CUDA events (median of --reps windows after --warmup), rows/s, mean / p99 / max of the
step count, step-rows/s (sum of steps over the time) and the fraction converged; with per-row seeds also how far the
converged rows moved from their seeds (the largest joint, wrapped).

--sweep adds (a)-(c) on --sweep-rows rows for each damping in --dampings with max_iter 256, to choose the defaults
from the step-count distributions.

Baselines on the rows of (a): the same steps written the obvious way in torch (`jacobian_device` + `fkine_device(what=
"joints")` + a batched `torch.linalg.solve` in fp64, --torch-steps steps for every row), and FABRIK alone
(`fabrik_solve_device`).  The host path (`IkEngine.dls_refine` into pinned memory) is timed on (a).

--compare-lib PATH (another build of libikb200.so, e.g. the parent commit's): `ikb_fk_transforms_device` (fp64 joints and
matrices) and `ikb_jacobian_device` (fp64 position) of both builds on the same rows, timed alternately in one process,
with their outputs compared bit for bit."""
import argparse
import ctypes
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
ROW_BYTES = 24 + 32 + 32 + 4 + 8
SHOULDER = (0.0, 0.0, 2.0)
BOX_LEN, BOX_START = (6.0, 12.0, 9.0), (0.0, -6.0, -3.0)
TOL = 1e-9
MODEL = os.path.join(ROOT, "models", "roboarm_b200_r01.h5")


def targets(n, reach, seed):
    """n cube_random targets: reach=True within reach, False beyond it."""
    import torch
    from inversekinematicsann_b200.robot.position_generator import TrainingDataGenerator as Gen
    out, got, k = [], 0, 0
    while got < n:
        xyz = Gen.cube_random_device(1.0, *BOX_LEN, start=BOX_START, seed=seed + k, no_of_samples=2 * n,
                                     dtype="float64")
        d = torch.linalg.vector_norm(xyz - torch.tensor(SHOULDER, dtype=torch.float64, device="cuda"), dim=1)
        keep = xyz[d < 6.0 - 1e-6] if reach else xyz[d > 6.0 + 1e-3]
        out.append(keep)
        got += keep.shape[0]
        k += 1
    return torch.cat(out)[:n].contiguous()


class Setup:
    def __init__(self):
        from inversekinematicsann_b200.kinematics.inverse import AnnInverseKinematics, FabrikInverseKinematics
        from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
        self.fabrik = FabrikInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
        self.ann = AnnInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
        self.ann.load_model(MODEL)
        self.eng = self.fabrik._engine()
        assert self.ann._engine() is self.eng

    def fabrik_seeds(self, xyz):
        import torch
        out = torch.empty((xyz.shape[0], 4), dtype=torch.float64, device="cuda")
        self.eng.fabrik_solve_device(xyz, out)
        return out

    def ann_seeds(self, xyz):
        import torch
        eng = self.ann.ann._ensure_uploaded()
        out = torch.empty((xyz.shape[0], 4), dtype=torch.float32, device="cuda")
        eng.ann_solve_device(xyz, out, mode=self.ann.ann.mode)
        return out.double()

    def workloads(self, n, seed):
        import torch
        reach = targets(n, True, seed)
        far = targets(n // 2, False, seed + 1000)
        half = torch.cat([reach[: n - n // 2], far])
        half = half[torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))]
        dh_seed = torch.tensor([[0.0, np.pi / 2, 0.0, 0.0]], dtype=torch.float64, device="cuda")
        return {"a_fabrik_seeded": (reach, self.fabrik_seeds(reach)), "b_ann_seeded": (reach, self.ann_seeds(reach)),
                "c_broadcast_dh_seed": (reach, dh_seed),
                "d_half_out_of_reach": (half.contiguous(), self.fabrik_seeds(half.contiguous()))}


def refine_stats(eng, xyz, seed, damping, max_iter, args, timed=True):
    import torch
    n = xyz.shape[0]
    out = torch.empty((n, 4), dtype=torch.float64, device="cuda")
    iters = torch.empty(n, dtype=torch.int32, device="cuda")
    err = torch.empty(n, dtype=torch.float64, device="cuda")
    run = lambda: eng.dls_refine_device(xyz, seed, out, iters, err, damping=damping, tol=TOL, max_iter=max_iter)
    t = event_seconds(run, args.reps, args.warmup) if timed else None
    if not timed:
        run()
    torch.cuda.synchronize()
    it = iters.cpu().numpy()
    conv = (err <= TOL).cpu().numpy()
    res = {"rows": n, "damping": damping, "max_iter": max_iter, "mean_steps": float(it.mean()),
           "p99_steps": float(np.percentile(it, 99)), "p999_steps": float(np.percentile(it, 99.9)),
           "max_steps": int(it.max()), "fraction_converged": float(conv.mean()),
           "mean_steps_converged": float(it[conv].mean()) if conv.any() else None,
           "max_steps_converged": int(it[conv].max()) if conv.any() else None}
    if seed.shape[0] == n and conv.any():
        # how far a converged row moved from its seed (largest joint, wrapped to [-pi, pi]): whether it kept its branch
        moved = (torch.remainder(out - seed + np.pi, 2 * np.pi) - np.pi).abs().amax(dim=1).cpu().numpy()[conv]
        res.update({"move_p999_rad": float(np.percentile(moved, 99.9)), "move_max_rad": float(moved.max()),
                    "fraction_moved_over_0.5_rad": float((moved > 0.5).mean())})
    if timed:
        res.update({"kernel_s": t, "rows_per_s": n / t, "step_rows_per_s": float(it.sum(dtype=np.int64)) / t})
    eng.stats_reset_torch()
    return res, out


def run_sweep(s, args):
    w = s.workloads(args.sweep_rows, 7)
    res = []
    for damping in args.dampings:
        for name in ("a_fabrik_seeded", "b_ann_seeded", "c_broadcast_dh_seed"):
            xyz, seed = w[name]
            r, _ = refine_stats(s.eng, xyz, seed, damping, 256, args, timed=False)
            r["workload"] = name
            res.append(r)
    return res


def torch_dls(fk, eng, xyz, theta, damping, steps):
    """The obvious way: per step one Jacobian launch, one FK launch and a batched 3x3 solve in torch."""
    import torch
    n = xyz.shape[0]
    J = torch.empty((n, 3, 4), dtype=torch.float64, device="cuda")
    joints = torch.empty((n, 4, 3), dtype=torch.float64, device="cuda")
    eye = torch.eye(3, dtype=torch.float64, device="cuda") * (damping * damping)
    for _ in range(steps):
        eng.jacobian_device(theta, J, "position")
        fk.fkine_device(theta, joints, "joints")
        e = xyz - joints[:, 3]
        A = torch.bmm(J, J.transpose(1, 2)) + eye
        y = torch.linalg.solve(A, e)
        theta += torch.bmm(J.transpose(1, 2), y.unsqueeze(2)).squeeze(2)
    return theta


def run_main(s, args):
    import torch
    from inversekinematicsann_b200 import engine as E
    from inversekinematicsann_b200.kinematics.forward import ForwardKinematics
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    n = int(min(args.max_rows, -(-4 * L2_BYTES // ROW_BYTES)))
    w = s.workloads(n, 11)
    res = {"defaults": {"damping": E.DLS_DAMPING, "max_iter": E.DLS_MAX_ITER, "tol": TOL}, "workloads": []}
    for name, (xyz, seed) in w.items():
        r, _ = refine_stats(s.eng, xyz, seed, E.DLS_DAMPING, E.DLS_MAX_ITER, args)
        r["workload"] = name
        res["workloads"].append(r)
    xyz, seed = w["a_fabrik_seeded"]
    fk = ForwardKinematics(R.dh_matrix)
    theta = torch.empty_like(seed)
    t_torch = event_seconds(lambda: torch_dls(fk, s.eng, xyz, theta.copy_(seed), E.DLS_DAMPING, args.torch_steps),
                            args.reps, args.warmup)
    res["torch_obvious_way"] = {"rows": n, "steps": args.torch_steps, "seconds": t_torch,
                                "step_rows_per_s": n * args.torch_steps / t_torch}
    out = torch.empty_like(seed)
    t_fab = event_seconds(lambda: s.eng.fabrik_solve_device(xyz, out), args.reps, args.warmup)
    res["fabrik_alone"] = {"rows": n, "seconds": t_fab, "rows_per_s": n / t_fab}
    # host path: the same rows from and into host memory (pinned output)
    h_xyz, h_seed = xyz.cpu().numpy(), seed.cpu().numpy()
    h_out = s.eng.pinned_empty((n, 4), np.float64)
    s.eng.dls_refine(h_xyz[: 1 << 16], h_seed[: 1 << 16], out=h_out[: 1 << 16])  # warm-up
    t0 = time.perf_counter()
    s.eng.dls_refine(h_xyz, h_seed, out=h_out)
    t_host = time.perf_counter() - t0
    res["host_a_fabrik_seeded"] = {"rows": n, "host_s": t_host, "host_rows_per_s": n / t_host}
    return res


def run_compare(s, args):
    """fk_transforms and jacobian of this build and another, alternately on the same rows."""
    import torch
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    other = ctypes.CDLL(os.path.abspath(args.compare_lib))
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    other.ikb_engine_create.argtypes = [ctypes.POINTER(_native.IkbConfig), ctypes.POINTER(vp)]
    other.ikb_fk_transforms_device.argtypes = [vp, vp, i32, i64, i32, vp, vp]
    other.ikb_jacobian_device.argtypes = [vp, vp, i32, i64, i32, vp, vp, vp]
    lim = R.effector_workspace_limits
    cfg = _native.IkbConfig()
    cfg.dh[:] = np.asarray(R.dh_matrix, dtype=np.float64).reshape(-1).tolist()
    cfg.links[:] = list(R.links_lengths)
    cfg.limits[:] = [lim["x"][0], lim["x"][1], lim["y"][0], lim["y"][1], lim["z"][0], lim["z"][1]]
    cfg.tol, cfg.max_iter, cfg.device = 1e-3, 100, 0
    h = vp()
    if other.ikb_engine_create(ctypes.byref(cfg), ctypes.byref(h)) != 0:
        raise RuntimeError("the other build could not create an engine")
    eng = s.eng
    stream = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = []
    for kind, tail, b_out in (("fk_transforms joints", (4, 3), 96), ("fk_transforms matrices", (4, 4, 4), 512),
                              ("jacobian position", (3, 4), 96)):
        n = int(min(args.max_rows, -(-4 * L2_BYTES // (32 + b_out))))
        g = torch.Generator(device="cuda").manual_seed(5)
        ang = (torch.rand(n, 4, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * np.pi
        mine = torch.empty((n,) + tail, dtype=torch.float64, device="cuda")
        theirs = torch.empty_like(mine)
        if kind.startswith("fk"):
            what = _native.IKB_FK_JOINTS if "joints" in kind else _native.IKB_FK_MATRICES
            run_mine = lambda: eng.fk_transforms_device(ang, mine, "joints" if "joints" in kind else "matrices")
            run_theirs = lambda: other.ikb_fk_transforms_device(h, ang.data_ptr(), _native.IKB_F64, n, what,
                                                                theirs.data_ptr(), stream())
        else:
            run_mine = lambda: eng.jacobian_device(ang, mine, "position")
            run_theirs = lambda: other.ikb_jacobian_device(h, ang.data_ptr(), _native.IKB_F64, n,
                                                           _native.IKB_JAC_POSITION, theirs.data_ptr(), None, stream())
        t_mine, t_theirs = [], []
        for _ in range(args.ab_rounds):  # alternate, so that both see the same machine state
            t_mine.append(event_seconds(run_mine, args.reps, args.warmup))
            t_theirs.append(event_seconds(run_theirs, args.reps, args.warmup))
        torch.cuda.synchronize()
        res.append({"kernel": kind, "dtype": "float64", "rows": n,
                    "this_build_rows_per_s": [n / t for t in t_mine], "other_build_rows_per_s": [n / t for t in t_theirs],
                    "ratio_of_medians": float(np.median(t_theirs) / np.median(t_mine)),
                    "identical_bits": bool(torch.equal(mine.view(torch.int64), theirs.view(torch.int64)))})
        del ang, mine, theirs
    return {"other_build": args.compare_label, "rows": res}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--max-rows", type=int, default=1 << 27)
    ap.add_argument("--sweep", action="store_true", help="also the damping sweep")
    ap.add_argument("--sweep-rows", type=int, default=1 << 20)
    ap.add_argument("--dampings", type=float, nargs="+", default=[0.001, 0.002, 0.005, 0.01, 0.02, 0.05, 0.1, 0.2, 0.5])
    ap.add_argument("--torch-steps", type=int, default=4)
    ap.add_argument("--compare-lib", default=None, help="another build of libikb200.so to time alternately against")
    ap.add_argument("--compare-label", default="other build", help="what the other build is, for the JSON line")
    ap.add_argument("--ab-rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    res = gpu_info()
    s = Setup()
    if args.sweep:
        res["sweep"] = run_sweep(s, args)
    res.update(run_main(s, args))
    if args.compare_lib:
        res["compare"] = run_compare(s, args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
