#!/usr/bin/env python3
"""Throughput of the batched cumulative DH transforms (ForwardKinematics.fkine_batch / joint_positions, csrc/fk.cu
fk_transforms_kernel).  Prints one JSON line.

Workloads: {matrices, joints} x {float32, float64}; angles seeded uniform in [-pi, pi].  Rows are sized so that angles
plus output are at least 4x the 126 MB L2, so every timed launch streams from and to HBM.

Per workload:
  - kernel time of `IkEngine.fk_transforms_device` from CUDA events after a warm-up (median of --reps), rows/s, bytes
    moved per row (angles in + output out) and the achieved GB/s;
  - the copy ceiling: a torch `fill_` of the output's size (write only) and a `copy_` of the output's size (read +
    write the same byte count), timed the same way in the same process; the kernel's fraction of each;
  - the host path (`IkEngine.fk_transforms` into a pinned output): rows/s and device-to-host GB/s of the output.
The "before": rows/s of a loop of single-pose `fkine` calls over --loop-poses poses, the only way to get all four
matrices of many poses without the batched path.

--compare-lib PATH loads another build of libikb200.so (the parent commit's, for example) and checks that its
`ikb_fk_chain_host` returns, pose for pose, the same bits as this build's batched path and the same status as this
build's `ikb_fk_chain_host`: 10^4 seeded poses, the engine's seed pose, poses at exactly +-2pi, NaN and poses outside
the range."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 * 2 ** 20


def row_bytes(what, dtype):
    item = np.dtype(dtype).itemsize
    return 4 * item, (64 if what == "matrices" else 12) * item


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.splitlines()[0]
        name, power, clock = [v.strip() for v in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError) as exc:
        return {"gpu_query_error": str(exc)}


def event_seconds(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(times))


def run_device(args):
    import torch
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    rows = []
    for what in ("matrices", "joints"):
        for dtype in (np.float32, np.float64):
            b_in, b_out = row_bytes(what, dtype)
            n = int(min(args.max_rows, -(-4 * L2_BYTES // (b_in + b_out))))
            td = torch.float32 if dtype == np.float32 else torch.float64
            g = torch.Generator(device="cuda").manual_seed(1)
            ang = ((torch.rand(n, 4, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * np.pi).to(td)
            tail = (4, 4, 4) if what == "matrices" else (4, 3)
            out = torch.empty((n,) + tail, dtype=td, device="cuda")
            t = event_seconds(lambda: eng.fk_transforms_device(ang, out, what), args.reps, args.warmup)
            flat = out.view(-1)
            src = torch.empty_like(flat).copy_(flat)
            t_fill = event_seconds(lambda: flat.fill_(1.0), args.reps, args.warmup)
            t_copy = event_seconds(lambda: flat.copy_(src), args.reps, args.warmup)
            del src
            out_bytes = n * b_out
            gbs = n * (b_in + b_out) / t / 1e9
            fill_gbs, copy_gbs = out_bytes / t_fill / 1e9, 2 * out_bytes / t_copy / 1e9
            # host path: the same rows from and into host memory (pinned output)
            h_ang = ang.cpu().numpy()
            h_out = eng.pinned_empty((n,) + tail, dtype)
            eng.fk_transforms(h_ang[: min(n, 1 << 16)], what, out=h_out[: min(n, 1 << 16)])  # warm-up
            t0 = time.perf_counter()
            _, st = eng.fk_transforms(h_ang, what, out=h_out)
            t_host = time.perf_counter() - t0
            rows.append({
                "what": what, "dtype": np.dtype(dtype).name, "rows": n, "bytes_per_row_in": b_in,
                "bytes_per_row_out": b_out, "kernel_s": t, "rows_per_s": n / t, "achieved_gb_s": gbs,
                "fill_gb_s": fill_gbs, "copy_gb_s": copy_gbs, "fraction_of_fill": gbs / fill_gbs,
                "fraction_of_copy": gbs / copy_gbs, "host_s": t_host, "host_rows_per_s": n / t_host,
                "host_d2h_gb_s": out_bytes / t_host / 1e9, "guard_fired": st.first_fk_angle_range >= 0,
            })
            del ang, out, flat, h_out
    # the "before": one pose per fkine call
    from inversekinematicsann_b200.kinematics.forward import ForwardKinematics
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    fk = ForwardKinematics(R.dh_matrix)
    poses = np.random.default_rng(2).uniform(-np.pi, np.pi, (args.loop_poses, 4))
    for p in poses[:100]:
        fk.fkine(list(p))
    t0 = time.perf_counter()
    for p in poses:
        fk.fkine(list(p))
    t_loop = time.perf_counter() - t0
    return {"workloads": rows, "fkine_loop": {"poses": args.loop_poses, "seconds": t_loop,
                                              "rows_per_s": args.loop_poses / t_loop}}


def compare_poses(seed_pose):
    rng = np.random.default_rng(3)
    two_pi = 2 * np.pi
    special = np.array([seed_pose,
                        [two_pi, -two_pi, two_pi, -two_pi], [-two_pi, 0.0, 0.0, two_pi],
                        [np.nan, 0.1, 0.2, 0.3], [0.1, np.nan, np.nan, 0.3],
                        [7.0, 0.0, 0.0, 0.0], [0.0, 0.0, -6.3, 0.0], [np.nextafter(two_pi, 7.0), 0.0, 0.0, 0.0]])
    return np.ascontiguousarray(np.vstack([special, rng.uniform(-np.pi, np.pi, (10_000, 4))]))


def run_compare(args):
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    dh = np.asarray(R.dh_matrix, dtype=np.float64)
    lim = R.effector_workspace_limits
    other = ctypes.CDLL(os.path.abspath(args.compare_lib))
    vp = ctypes.c_void_p
    other.ikb_engine_create.argtypes = [ctypes.POINTER(_native.IkbConfig), ctypes.POINTER(vp)]
    other.ikb_fk_chain_host.argtypes = [vp, vp, vp, ctypes.POINTER(ctypes.c_int)]
    cfg = _native.IkbConfig()
    cfg.dh[:] = dh.reshape(-1).tolist()
    cfg.links[:] = list(R.links_lengths)
    cfg.limits[:] = [lim["x"][0], lim["x"][1], lim["y"][0], lim["y"][1], lim["z"][0], lim["z"][1]]
    cfg.tol, cfg.max_iter, cfg.device = 1e-3, 100, 0
    h = vp()
    if other.ikb_engine_create(ctypes.byref(cfg), ctypes.byref(h)) != 0:
        raise RuntimeError("the other build could not create an engine")
    poses = compare_poses([0.0, dh[0, 1], dh[0, 2], dh[0, 3]])
    n = poses.shape[0]
    want = np.empty((n, 4, 4, 4))
    want_st = np.empty(n, dtype=np.int32)
    st = ctypes.c_int(0)
    for i in range(n):
        row = np.ascontiguousarray(poses[i])
        if other.ikb_fk_chain_host(h, row.ctypes.data, want[i].ctypes.data, ctypes.byref(st)) != 0:
            raise RuntimeError("the other build's ikb_fk_chain_host failed")
        want_st[i] = st.value
    with IkEngine(dh, R.links_lengths, R.effector_workspace_limits) as eng:
        got, stats = eng.fk_transforms(poses)
        got_st = np.array([eng.fk_chain(p)[1] for p in poses], dtype=np.int32)
        single = np.array([eng.fk_chain(p)[0] for p in poses[:200]])
    bad_rows = np.flatnonzero(want_st)
    same_bits = bool(np.array_equal(got.view(np.uint64), want.view(np.uint64)))
    return {"other_build": args.compare_label, "poses": n,
            "identical_bits": same_bits,
            "identical_bits_single_pose_path": bool(np.array_equal(single.view(np.uint64),
                                                                   want[:200].view(np.uint64))),
            "identical_status": bool(np.array_equal(got_st, want_st)),
            "out_of_range_rows": bad_rows.tolist(),
            "batched_first_fk_angle_range": stats.first_fk_angle_range,
            "first_matches": stats.first_fk_angle_range == (int(bad_rows[0]) if bad_rows.size else -1)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--max-rows", type=int, default=1 << 27)
    ap.add_argument("--loop-poses", type=int, default=10_000)
    ap.add_argument("--compare-lib", default=None, help="another build of libikb200.so to check bit for bit against")
    ap.add_argument("--compare-label", default="other build", help="what the other build is, for the JSON line")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    res = gpu_info()
    res.update(run_device(args))
    if args.compare_lib:
        res["compare"] = run_compare(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
