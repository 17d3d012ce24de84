#!/usr/bin/env python3
"""Throughput and convergence of the damped-least-squares refinement onto poses (InverseKinematics.refine_pose /
ikine_pose, csrc/fk.cu dls_pose_refine_kernel).  Prints one JSON line.

Poses are fkine_batch of angles uniform in [-pi, pi]^4 whose effector lies inside the workspace box, so every one is
reachable.  Rows are sized so that poses, seeds, angles, iterations and errors (204 B per fp64 row) are at least 4x
the 126 MB L2.  Every workload is fp64 and device-resident, default weights (all ones), tol 1e-9:
  (a) FABRIK-seeded (`fabrik_solve_device` on the position column);
  (b) one broadcast seed, the DH table's seed row [0, pi/2, 0, 0] (the arm straight up, a singular pose);
  (c) ANN-seeded (models/roboarm_b200_r01, float32 predictions widened);
  (d) the positions of (a) with uniformly random rotations, FABRIK-seeded: generally not a pose of this 4-joint arm,
      so these run to max_iter;
  (e) weights (1, 1, 1, 0, 0, 0) on the rows and seeds of (a), and `dls_refine_device` on their positions.
Per workload: kernel time from CUDA events (median of --reps windows after --warmup), rows/s, mean / p99 / max of the
step count, step-rows/s (sum of steps over the time), the fraction converged and the fraction converged within
8, 16, ... steps.  For per-row seeds of poses of known angles, also how many seeds have theta_1 more than pi/2 from the
pose's own (the arm reaching back over its base, which puts the seed's orientation about pi off), how many of these
and of the others converge, and the final errors of the rows that do not.

--sweep adds (a)-(c) on --sweep-rows rows for each damping in --dampings with max_iter 256, to choose the defaults
from the step-count distributions.

Baseline on the rows of (a): the same steps written in torch (`fkine_device` + `jacobian_device` + the quaternion error
+ a batched `torch.linalg.solve` in fp64, --torch-steps steps for every row).

--compare-lib PATH (another build of libikb200.so, e.g. the parent commit's): `ikb_dls_refine_device` and
`ikb_fk_transforms_device` (fp64 matrices) of both builds on the same rows, timed alternately in one process, with
their outputs compared bit for bit."""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fk_transforms_bench import event_seconds, gpu_info  # noqa: E402

L2_BYTES = 126 * 2 ** 20
ROW_BYTES = 128 + 32 + 32 + 4 + 8
LIMITS = ((0.0, 6.0), (-6.0, 6.0), (-3.0, 6.0))
TOL = 1e-9
MODEL = os.path.join(ROOT, "models", "roboarm_b200_r01.h5")
POSITION_ONLY = (1.0, 1.0, 1.0, 0.0, 0.0, 0.0)


def poses(fk, n, seed):
    """(theta, T): n poses T = fkine_batch(theta), theta uniform in [-pi, pi]^4, whose position is inside the
    workspace box."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    out, ths, got = [], [], 0
    while got < n:
        th = (torch.rand(2 * n, 4, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * np.pi
        T = fk.fkine_device(th)[:, 3]
        p = T[:, :3, 3]
        ok = torch.ones(th.shape[0], dtype=torch.bool, device="cuda")
        for i, (lo, hi) in enumerate(LIMITS):
            ok &= (p[:, i] >= lo) & (p[:, i] <= hi)
        out.append(T[ok])
        ths.append(th[ok])
        got += int(ok.sum())
        del T
    return torch.cat(ths)[:n].contiguous(), torch.cat(out)[:n].contiguous()


def random_rotations(T, seed):
    """The positions of T with uniformly random rotations (unit quaternions from a 4-D normal)."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn(T.shape[0], 4, device="cuda", generator=g, dtype=torch.float64)
    w, x, y, z = (q / torch.linalg.vector_norm(q, dim=1, keepdim=True)).unbind(1)
    R = torch.stack([torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], -1),
                     torch.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)], -1),
                     torch.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1)], -2)
    out = T.clone()
    out[:, :3, :3] = R
    return out


class Setup:
    def __init__(self):
        from inversekinematicsann_b200.kinematics.inverse import AnnInverseKinematics, FabrikInverseKinematics
        from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
        self.fabrik = FabrikInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
        self.ann = AnnInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
        self.ann.load_model(MODEL)
        self.eng = self.fabrik._engine()
        self.fk = self.fabrik.fkine
        assert self.ann._engine() is self.eng

    def fabrik_seeds(self, T):
        import torch
        out = torch.empty((T.shape[0], 4), dtype=torch.float64, device="cuda")
        self.eng.fabrik_solve_device(T[:, :3, 3].contiguous(), out)
        return out

    def ann_seeds(self, T):
        import torch
        eng = self.ann.ann._ensure_uploaded()
        out = torch.empty((T.shape[0], 4), dtype=torch.float32, device="cuda")
        eng.ann_solve_device(T[:, :3, 3].contiguous(), out, mode=self.ann.ann.mode)
        return out.double()

    def workloads(self, n, seed, with_rotations=True):
        import torch
        th, T = poses(self.fk, n, seed)
        self.truth = th
        dh_seed = torch.tensor([[0.0, np.pi / 2, 0.0, 0.0]], dtype=torch.float64, device="cuda")
        w = {"a_fabrik_seeded": (T, self.fabrik_seeds(T)), "b_broadcast_dh_seed": (T, dh_seed),
             "c_ann_seeded": (T, self.ann_seeds(T))}
        if with_rotations:
            Tr = random_rotations(T, seed + 1)
            w["d_random_rotations"] = (Tr, self.fabrik_seeds(Tr))
        return w


def summary(it, conv, n, t):
    res = {"rows": n, "mean_steps": float(it.mean()), "p99_steps": float(np.percentile(it, 99)),
           "fraction_converged_within": {str(k): float((conv & (it <= k)).mean()) for k in (8, 16, 32, 64, 128, 256)
                                         if k <= it.max()},
           "p999_steps": float(np.percentile(it, 99.9)), "max_steps": int(it.max()),
           "fraction_converged": float(conv.mean()),
           "mean_steps_converged": float(it[conv].mean()) if conv.any() else None,
           "max_steps_converged": int(it[conv].max()) if conv.any() else None}
    if t is not None:
        res.update({"kernel_s": t, "rows_per_s": n / t, "step_rows_per_s": float(it.sum(dtype=np.int64)) / t})
    return res


def refine_stats(eng, T, seed, damping, max_iter, args, weights=None, timed=True, truth=None):
    import torch
    n = T.shape[0]
    out = torch.empty((n, 4), dtype=torch.float64, device="cuda")
    iters = torch.empty(n, dtype=torch.int32, device="cuda")
    err = torch.empty(n, dtype=torch.float64, device="cuda")
    run = lambda: eng.dls_pose_refine_device(T, seed, out, iters, err, weights=weights, damping=damping, tol=TOL,
                                             max_iter=max_iter)
    t = event_seconds(run, args.reps, args.warmup) if timed else None
    if not timed:
        run()
    torch.cuda.synchronize()
    conv = (err <= TOL).cpu().numpy()
    res = summary(iters.cpu().numpy(), conv, n, t)
    res.update({"damping": damping, "max_iter": max_iter})
    if truth is not None and seed.shape[0] == n:
        # theta_1 fixes the arm's vertical plane and the sign of its joint axes: a seed whose theta_1 is more than
        # pi/2 from the pose's own (the arm reaching back over its base) starts with the orientation about pi off
        flipped = ((torch.remainder(seed[:, 0] - truth[:, 0] + np.pi, 2 * np.pi) - np.pi).abs() > np.pi / 2).cpu().numpy()
        e = err.cpu().numpy()
        res.update({"fraction_seed_theta1_flipped": float(flipped.mean()),
                    "fraction_flipped_among_not_converged": float(flipped[~conv].mean()) if (~conv).any() else None,
                    "fraction_converged_of_flipped": float(conv[flipped].mean()) if flipped.any() else None,
                    "fraction_converged_of_not_flipped": float(conv[~flipped].mean()) if (~flipped).any() else None,
                    "err_not_converged_p10_p50_p90": [float(v) for v in np.percentile(e[~conv], [10, 50, 90])]
                    if (~conv).any() else None})
    eng.stats_reset_torch()
    return res


def run_sweep(s, args):
    w = s.workloads(args.sweep_rows, 7, with_rotations=False)
    res = []
    for damping in args.dampings:
        for name, (T, seed) in w.items():
            r = refine_stats(s.eng, T, seed, damping, 256, args, timed=False,
                             truth=s.truth if name != "b_broadcast_dh_seed" else None)
            r["workload"] = name
            res.append(r)
    return res


def torch_pose_steps(fk, eng, T, theta, damping, steps):
    """The obvious way: per step one FK launch, one Jacobian launch, the quaternion error and a batched 4x4 solve."""
    import torch
    n = T.shape[0]
    J = torch.empty((n, 6, 4), dtype=torch.float64, device="cuda")
    chain = torch.empty((n, 4, 4, 4), dtype=torch.float64, device="cuda")
    eye = torch.eye(4, dtype=torch.float64, device="cuda") * (damping * damping)
    Rd, pd = T[:, :3, :3], T[:, :3, 3]
    for _ in range(steps):
        fk.fkine_device(theta, chain, "matrices")
        eng.jacobian_device(theta, J, "geometric")
        M = torch.bmm(Rd, chain[:, 3, :3, :3].transpose(1, 2))
        tr = M[:, 0, 0] + M[:, 1, 1] + M[:, 2, 2]
        d = torch.stack([M[:, 2, 1] - M[:, 1, 2], M[:, 0, 2] - M[:, 2, 0], M[:, 1, 0] - M[:, 0, 1]], 1)
        diag = torch.stack([M[:, 0, 0], M[:, 1, 1], M[:, 2, 2]], 1)
        big = diag.argmax(1)
        use_tr = tr >= diag.amax(1)
        h_tr = torch.sqrt((1 + tr).clamp_min(0))
        i = big
        j, k = (i + 1) % 3, (i + 2) % 3
        ar = torch.arange(n, device="cuda")
        h = torch.sqrt((1 + M[ar, i, i] - M[ar, j, j] - M[ar, k, k]).clamp_min(0))
        qi = h
        qj = (M[ar, i, j] + M[ar, j, i]) / h
        qk = (M[ar, i, k] + M[ar, k, i]) / h
        sgn = torch.where(d[ar, i] < 0, -1.0, 1.0)
        eo_d = torch.zeros((n, 3), dtype=torch.float64, device="cuda")
        eo_d[ar, i], eo_d[ar, j], eo_d[ar, k] = qi * sgn, qj * sgn, qk * sgn
        eo = torch.where(use_tr[:, None], d / h_tr[:, None], eo_d)
        e = torch.cat([pd - chain[:, 3, :3, 3], eo], 1)
        A = torch.bmm(J.transpose(1, 2), J) + eye
        b = torch.bmm(J.transpose(1, 2), e.unsqueeze(2))
        theta += torch.linalg.solve(A, b).squeeze(2)
    return theta


def run_main(s, args):
    import torch
    from inversekinematicsann_b200 import engine as E
    n = int(min(args.max_rows, -(-4 * L2_BYTES // ROW_BYTES)))
    w = s.workloads(n, 11)
    res = {"defaults": {"weights": list(E.POSE_WEIGHTS), "damping": E.POSE_DAMPING, "max_iter": E.POSE_MAX_ITER,
                        "tol": TOL}, "workloads": []}
    for name, (T, seed) in w.items():
        r = refine_stats(s.eng, T, seed, E.POSE_DAMPING, E.POSE_MAX_ITER, args,
                         truth=s.truth if name in ("a_fabrik_seeded", "c_ann_seeded") else None)
        r["workload"] = name
        res["workloads"].append(r)
    T, seed = w["a_fabrik_seeded"]
    r = refine_stats(s.eng, T, seed, E.POSE_DAMPING, E.POSE_MAX_ITER, args, weights=POSITION_ONLY)
    r["workload"] = "e_position_weights"
    res["workloads"].append(r)
    xyz = T[:, :3, 3].contiguous()
    out = torch.empty_like(seed)
    iters = torch.empty(n, dtype=torch.int32, device="cuda")
    err = torch.empty(n, dtype=torch.float64, device="cuda")
    run = lambda: s.eng.dls_refine_device(xyz, seed, out, iters, err, damping=E.POSE_DAMPING, tol=TOL,
                                          max_iter=E.POSE_MAX_ITER)
    t = event_seconds(run, args.reps, args.warmup)
    r = summary(iters.cpu().numpy(), (err <= TOL).cpu().numpy(), n, t)
    r.update({"workload": "e_dls_refine_same_rows", "damping": E.POSE_DAMPING, "max_iter": E.POSE_MAX_ITER})
    res["workloads"].append(r)
    s.eng.stats_reset_torch()
    theta = torch.empty_like(seed)
    t_torch = event_seconds(lambda: torch_pose_steps(s.fk, s.eng, T, theta.copy_(seed), E.POSE_DAMPING,
                                                     args.torch_steps), args.reps, args.warmup)
    res["torch_obvious_way"] = {"rows": n, "steps": args.torch_steps, "seconds": t_torch,
                                "step_rows_per_s": n * args.torch_steps / t_torch}
    return res


def run_compare(s, args):
    """dls_refine and fk_transforms of this build and another, alternately on the same rows."""
    import torch
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    other = ctypes.CDLL(os.path.abspath(args.compare_lib))
    vp, i32, i64, dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
    other.ikb_engine_create.argtypes = [ctypes.POINTER(_native.IkbConfig), ctypes.POINTER(vp)]
    other.ikb_fk_transforms_device.argtypes = [vp, vp, i32, i64, i32, vp, vp]
    other.ikb_dls_refine_device.argtypes = [vp, vp, i32, i64, vp, i64, vp, i32, dbl, dbl, ctypes.c_int32, vp, vp, vp]
    lim = R.effector_workspace_limits
    cfg = _native.IkbConfig()
    cfg.dh[:] = np.asarray(R.dh_matrix, dtype=np.float64).reshape(-1).tolist()
    cfg.links[:] = list(R.links_lengths)
    cfg.limits[:] = [lim["x"][0], lim["x"][1], lim["y"][0], lim["y"][1], lim["z"][0], lim["z"][1]]
    cfg.tol, cfg.max_iter, cfg.device = 1e-3, 100, 0
    h = vp()
    if other.ikb_engine_create(ctypes.byref(cfg), ctypes.byref(h)) != 0:
        raise RuntimeError("the other build could not create an engine")
    from inversekinematicsann_b200 import engine as E
    eng = s.eng
    stream = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = []
    # dls_refine: FABRIK-seeded positions of poses (the rows of workload (a))
    n = int(min(args.max_rows, -(-4 * L2_BYTES // 100)))
    _, T = poses(s.fk, n, 21)
    xyz = T[:, :3, 3].contiguous()
    del T
    seed = torch.empty((n, 4), dtype=torch.float64, device="cuda")
    eng.fabrik_solve_device(xyz, seed)
    mine, theirs = torch.empty_like(seed), torch.empty_like(seed)
    run_mine = lambda: eng.dls_refine_device(xyz, seed, mine, damping=E.DLS_DAMPING, tol=TOL, max_iter=E.DLS_MAX_ITER)
    run_theirs = lambda: other.ikb_dls_refine_device(h, xyz.data_ptr(), _native.IKB_F64, n, seed.data_ptr(), n,
                                                     theirs.data_ptr(), _native.IKB_F64, E.DLS_DAMPING, TOL,
                                                     E.DLS_MAX_ITER, None, None, stream())
    jobs = [("dls_refine fabrik-seeded", n, run_mine, run_theirs, mine, theirs)]
    m = int(min(args.max_rows, -(-4 * L2_BYTES // (32 + 512))))
    g = torch.Generator(device="cuda").manual_seed(5)
    ang = (torch.rand(m, 4, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * np.pi
    cm, ct = torch.empty((m, 4, 4, 4), dtype=torch.float64, device="cuda"), torch.empty((m, 4, 4, 4), dtype=torch.float64,
                                                                                        device="cuda")
    jobs.append(("fk_transforms matrices", m, lambda: eng.fk_transforms_device(ang, cm, "matrices"),
                 lambda: other.ikb_fk_transforms_device(h, ang.data_ptr(), _native.IKB_F64, m, _native.IKB_FK_MATRICES,
                                                        ct.data_ptr(), stream()), cm, ct))
    for kind, rows, rm, rt, a, b in jobs:
        t_mine, t_theirs = [], []
        for _ in range(args.ab_rounds):  # alternate, so that both see the same machine state
            t_mine.append(event_seconds(rm, args.reps, args.warmup))
            t_theirs.append(event_seconds(rt, args.reps, args.warmup))
        torch.cuda.synchronize()
        res.append({"kernel": kind, "dtype": "float64", "rows": rows,
                    "this_build_rows_per_s": [rows / t for t in t_mine],
                    "other_build_rows_per_s": [rows / t for t in t_theirs],
                    "ratio_of_medians": float(np.median(t_theirs) / np.median(t_mine)),
                    "identical_bits": bool(torch.equal(a.view(torch.int64), b.view(torch.int64)))})
    eng.stats_reset_torch()
    return {"other_build": args.compare_label, "rows": res}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
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
