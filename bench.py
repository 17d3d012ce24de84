#!/usr/bin/env python
"""Headline benchmark: batched IK solves/s of the B200 engine (FABRIK + ANN) beside the CPU restatement.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Under torchrun (N > 1) every rank solves its own contiguous shard of the trajectory (weak scaling:
`--rows` FABRIK targets per GPU); rank 0 prints ONE JSON line.  A "step" is one pass of the hot path
(check_limits + FABRIK + fp64 angle extraction) over the rank's batch of synthetic cube_random targets,
inputs resident in HBM (`value`), or host-resident and pushed through the public
FabrikInverseKinematics.ikine() call (`e2e`).  The ANN path (config 2) rides in the same line under "ann".

`--impl reference` times the CPU restatement of the reference's algorithm (oracle/ik_oracle.c, all host
threads; the reference itself is pure Python and cannot travel to the GPU box) on bounded samples of the
same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "IK solves/sec (FABRIK, cube_random full workspace, tol 1e-3 / 100 iterations)"
UNIT = "solves/s"
WORKSPACE_BOX = ((6.0, 12.0, 9.0), (0.0, -6.0, -3.0))   # SURVEY 8d cfg 3 (W): len, start
INTERIOR_BOX = ((2.0, 4.0, 3.0), (1.0, -2.0, 1.0))      # SURVEY 8d cfg 3 (R)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline FABRIK loop (`value`); the secondary legs time "
                         "between 2 and 5 steps, or half of this")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="FABRIK targets per GPU (config 3)")
    ap.add_argument("--ann-rows", type=int, default=1_000_000, help="ANN targets per GPU (config 2)")
    ap.add_argument("--e2e-rows", type=int, default=0, help="host-resident rows per GPU for e2e (0 = --rows)")
    ap.add_argument("--ann-big-rows", type=int, default=125_000_000,
                    help="ANN targets per GPU for the config-4 leg (1e9 over 8 GPUs); 0 skips it")
    ap.add_argument("--skip-ann", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0; a fixed, seeded sample "
                         f"of at most {DUMP_ROWS} rows per array) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_ROWS = 1_500_000   # 24 MB of float32 [*, 4] angles per dumped array, 48 MB for both


def dump_rows(n):
    """The rows of an n-row output that --dump-outputs writes: all of them up to DUMP_ROWS, else the same seeded sample
    in every run, in ascending order."""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))


# ---- clocks -----------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self, t0, t1):
        rows = [r for t, r in self.samples if t0 <= t <= t1] or [r for _, r in self.samples[-3:]]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(rows[0][1]),
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows), "reasons": reasons}


# the same string in both arms' config (the reference arm solves a bounded sample of it per step)
WORKLOAD = ("BASELINE configs[2]: FABRIK on 100M cube_random targets per GPU, full workspace box (0,-6,-3)+(6,12,9) "
            "(GPU arm: device generator, Philox4x32-10, seed 1234+rank); configs[1] (ANN with the shipped .h5) cannot "
            "run as stated because the weights are absent -- see \"ann\"")


# ---- CPU arm (oracle port) -----------------------------------------------------------------------------
def host_points(n, box, seed):
    """Rows [0, n) of the GPU arm's rank-0 input: the device generator's Philox stream restated in NumPy
    (oracle/np_oracle.philox_cube_random), rounded to float32 as the device buffer is, widened to the float64 the
    C restatement computes in -- the same numbers the kernel reads."""
    from oracle import np_oracle
    ln, st = box
    return np_oracle.philox_cube_random(n, ln, st, seed, dtype=np.float32).astype(np.float64)


def cpu_fabrik_rate(sample_rows, box, seed=1234, repeats=1):
    """solves/s of the C restatement (OpenMP, all host threads) on `sample_rows` targets."""
    from oracle import c_oracle
    c_oracle.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1 to its workers
    pts = host_points(sample_rows, box, seed)
    c_oracle.fabrik_ikine(pts[:1000])
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        res = c_oracle.fabrik_ikine(pts)
        best = min(best, time.perf_counter() - t0)
    return sample_rows / best, c_oracle.num_threads(), float(res["iters"].mean())


def cpu_ann_rate(sample_rows, weights, biases, seed=1234):
    """solves/s of the NumPy fp32 restatement (BLAS threads = all host cores)."""
    from oracle import np_oracle
    from threadpoolctl import threadpool_limits
    pts = host_points(sample_rows, WORKSPACE_BOX, seed)
    with threadpool_limits(limits=os.cpu_count() or 1):
        np_oracle.mlp_predict(pts[:2048], weights, biases)
        t0 = time.perf_counter()
        np_oracle.mlp_predict(pts, weights, biases)
        return sample_rows / (time.perf_counter() - t0)


def calibrated_cpu_sample(box, target_seconds=12.0):
    rate, threads, _ = cpu_fabrik_rate(200_000, box, repeats=2)
    return int(max(100_000, min(20_000_000, rate * target_seconds))), threads


def run_reference_arm(args, rank):
    """The reference's own algorithm on the host cores: rank 0 only, bounded samples per step."""
    if rank != 0:
        return
    from oracle import c_oracle
    c_oracle.set_num_threads(os.cpu_count() or 1)
    sample, threads = calibrated_cpu_sample(WORKSPACE_BOX, target_seconds=6.0)
    pts = host_points(sample, WORKSPACE_BOX, 1234)
    for _ in range(max(1, min(args.warmup, 2))):
        c_oracle.fabrik_ikine(pts[: sample // 4])
    t0 = time.perf_counter()
    iters = 0.0
    for _ in range(args.steps):
        iters = float(c_oracle.fabrik_ikine(pts)["iters"].mean())
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "gpu_launches": 0,
        "config": {"workload": WORKLOAD, "rows_per_step": sample, "mean_iterations": iters,
                   "input": "rows [0, rows_per_step) of the GPU arm's rank-0 input (the same Philox4x32-10 stream, seed 1234, "
                            "restated in NumPy: float32 values widened to float64)",
                   "fabrik_precision": "fp64 (C restatement of the reference's Python floats)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} targets per step x {args.steps} steps, oracle/ik_oracle.c "
                                   f"(C restatement of fabrik.py + inverse.py, OpenMP); the reference is "
                                   f"pure Python (~4e2 solves/s/core on this workload, BASELINE.md) and is "
                                   f"not present on the GPU box"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---- GPU arm -----------------------------------------------------------------------------------------
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3  # timing rule: at least 3 warm-up steps

    import torch
    import torch.distributed as dist
    from inversekinematicsann_b200.engine import fabrik_algorithmic_flops
    from inversekinematicsann_b200.kinematics.inverse import AnnInverseKinematics, FabrikInverseKinematics
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    from inversekinematicsann_b200.sharding import PeerGather, ShardedFabrik, gather_rows, reduce_stats

    def bind_to_gpu_numa_node(index):
        """Pin this rank to the CPUs next to its GPU so that its pinned staging buffers are allocated on the
        local NUMA node (eight ranks otherwise share one node's memory controllers for all H2D/D2H traffic)."""
        try:
            import pynvml
            pynvml.nvmlInit()
            handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            words = (os.cpu_count() + 63) // 64
            mask = pynvml.nvmlDeviceGetCpuAffinity(handle, words)
            cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
            cpus &= os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
            return len(cpus)
        except Exception:
            return 0

    numa_cpus = bind_to_gpu_numa_node(local_rank) if world > 1 else 0
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        from datetime import timedelta
        dist.init_process_group("nccl", device_id=dev, timeout=timedelta(seconds=180))   # a hang fails fast

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(seconds):
        if world == 1:
            return seconds
        t = torch.tensor([seconds], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ik = FabrikInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits, device=local_rank)
    eng = ik._engine()
    n = args.rows

    def device_points(rows, box, seed):
        """cube_random (position_generator.py:48-55: start + len * U[0,1) per axis) generated on the device by
        csrc/generators.cu (Philox4x32-10), `rows` points."""
        from inversekinematicsann_b200.robot.position_generator import TrainingDataGenerator as Gen
        ln, st = box
        return Gen.cube_random_device(ln[0] * ln[1] * ln[2] / rows, ln[0], ln[1], ln[2], start=st, seed=seed,
                                      no_of_samples=rows, device=local_rank)

    def timed_device_loop(fn, steps, warmup):
        """K steps bracketed by barrier + synchronize, CUDA events on torch's current stream (the stream
        the kernels are launched on); returns (max-over-ranks seconds, wall t0, wall t1)."""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        w1 = time.perf_counter()
        return max_over_ranks(e0.elapsed_time(e1) * 1e-3), w0, w1

    def dump(name, t):
        """--dump-outputs: the dump_rows sample of rank 0's device output t, as DIR/<name>.npy"""
        if args.dump_outputs and rank == 0:
            rows = torch.from_numpy(dump_rows(t.shape[0])).to(t.device)
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.index_select(0, rows).cpu().numpy())

    PARITY_ROWS = 100_000

    def reduce_parity(block):
        """max / p99 -> maximum over ranks, counts -> sums, means -> row-weighted means (every rank checks the first
        PARITY_ROWS rows of ITS shard against the oracle on its own host cores)."""
        if world == 1:
            return block
        keys = sorted(block)
        mx = torch.tensor([block[k] for k in keys if k.startswith(("max_", "p99_"))], dtype=torch.float64, device=dev)
        sm = torch.tensor([block[k] for k in keys if k.startswith(("rows", "n_", "sum_"))], dtype=torch.float64, device=dev)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        out = dict(block)
        for k, v in zip([k for k in keys if k.startswith(("max_", "p99_"))], mx.tolist()):
            out[k] = v
        for k, v in zip([k for k in keys if k.startswith(("rows", "n_", "sum_"))], sm.tolist()):
            out[k] = v
        return out

    def finish_parity(block, tol):
        """counts / sums -> the fractions and means SURVEY 8d asks for"""
        rows = max(block["rows"] - block["n_excluded_degenerate"], 1)
        out = {"rows": int(block["rows"]), "excluded_degenerate": int(block["n_excluded_degenerate"]),
               "max_abs_dtheta": block["max_abs_dtheta"], "p99": block["p99_abs_dtheta"],
               f"frac_gt_{tol:g}": block["n_gt_tol"] / rows}
        if "n_k_mismatch" in block:
            out["k_mismatch_frac"] = block["n_k_mismatch"] / rows
        out["fk_err_ref_vs_engine"] = {"reference_mean": block["sum_fk_ref"] / rows, "engine_mean": block["sum_fk_eng"] / rows,
                                       "max_abs_diff": block["max_fk_diff"]}
        for k in ("max_abs_dtheta_vs_fp64", "max_abs_dtheta_vs_torch", "max_oracle_fp32_vs_fp64"):
            if k in block:
                out[k] = block[k]
        return out

    def fabrik_parity(xyz_dev, angles_dev, iters_dev, label):
        """The first PARITY_ROWS rows of THIS launch's inputs and outputs against the CPU oracle
        (oracle/ik_oracle.c = fabrik.py + inverse.py:54-139 restated): SURVEY 8d 'parity metrics to print'."""
        from oracle import c_oracle
        c_oracle.set_num_threads(os.cpu_count() or 1)
        m = min(PARITY_ROWS, xyz_dev.shape[0])
        pts = xyz_dev[:m].double().cpu().numpy()             # the float32 inputs, exactly as the kernel read them
        got = angles_dev[:m].double().cpu().numpy()
        got_k = iters_dev[:m].cpu().numpy()
        want = c_oracle.fabrik_ikine(pts)
        ok = np.isfinite(want["angles"]).all(axis=1) & np.isfinite(got).all(axis=1)
        d = np.abs(got - want["angles"])[ok].max(axis=1) if ok.any() else np.zeros(1)
        _, _, fk_ref = c_oracle.fk_positions(want["angles"][ok], targets=pts[ok])
        _, _, fk_eng = c_oracle.fk_positions(got[ok], targets=pts[ok])
        block = {"rows": m, "n_excluded_degenerate": int((~ok).sum()), "max_abs_dtheta": float(d.max()),
                 "p99_abs_dtheta": float(np.quantile(d, 0.99)), "n_gt_tol": int((d > 1e-4).sum()),
                 "n_k_mismatch": int((got_k[ok] != want["iters"][ok]).sum()),
                 "sum_fk_ref": float(fk_ref.sum()), "sum_fk_eng": float(fk_eng.sum()),
                 "max_fk_diff": float(np.abs(fk_ref - fk_eng).max())}
        out = finish_parity(reduce_parity(block), 1e-4)
        out["what"] = (f"{label}: rows [0, {m}) of every rank's shard, outputs of the full-size launch (float32 angles) vs "
                       f"oracle/ik_oracle.c on the same float32 inputs; bar 1e-4 rad, iteration counts exact")
        return out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # ---- FABRIK, device resident (value + roofline) ----------------------------------------------
    xyz = device_points(n, WORKSPACE_BOX, 1234 + rank)          # 1.2 GB >> 126 MB L2
    angles = torch.empty(n, 4, device=dev, dtype=torch.float32)
    eng.stats_reset_torch()
    eng.fabrik_solve_device(xyz, angles)
    one = eng.stats_fetch_torch()                               # per-launch iteration count (deterministic)
    launches0 = eng.launch_count
    secs, w0, w1 = timed_device_loop(lambda: eng.fabrik_solve_device(xyz, angles), args.steps, args.warmup)
    dump("fabrik_angles", angles)   # before the legs below overwrite `angles`
    gpu_launches = (eng.launch_count - launches0 - args.warmup) * world
    value = n * world * args.steps / secs
    total = reduce_stats(one)
    flops_per_launch = fabrik_algorithmic_flops(one.sum_iterations, n)
    launch_s = secs / args.steps
    peak_fp64 = eng.microbench_fma("f64")
    peak_fp64_theory = eng.theoretical_fma_peak("f64")
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6650.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        if t.get("rows") == n:
            traffic = t.get("dram_bytes_per_launch")
    roofline = {
        "kernel": "fabrik_split_kernel<double>", "bound": "fp64",
        "achieved": flops_per_launch / launch_s / 1e12, "peak": peak_fp64, "unit": "TFLOP/s",
        "frac": flops_per_launch / launch_s / 1e12 / peak_fp64,
        "peak_source": "measured live: DFMA-chain microbenchmark (ikb_microbench_fma); MEASURED_PEAKS.json has no "
                       "CUDA-core figure",
        "peak_theoretical": peak_fp64_theory, "frac_of_theoretical": flops_per_launch / launch_s / 1e12 / peak_fp64_theory,
        "peak_theoretical_source": "SMs x 64 fp64 lanes x 2 x max SM clock (cudaDevAttrClockRate)",
        "flops_per_launch": flops_per_launch, "flops_model": "114*sum_iterations + 126*rows (SURVEY 8d)",
        "launch_ms": launch_s * 1e3,
        "hbm": {"achieved": n * 28 / launch_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": n * 28 / launch_s / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if os.path.exists(peaks_path) else "fallback"},
        "traffic": traffic,
    }

    # parity of THIS launch's rows against the oracle (outside the timed region)
    it_full = torch.empty(n, device=dev, dtype=torch.int32)
    eng.fabrik_solve_device(xyz, angles, iters=it_full)
    parity = {"fabrik_workspace_box": fabrik_parity(xyz, angles, it_full, "cfg 3 (W) cube_random full workspace")}
    del it_full

    # opt-in fp32 iterate (the north star's FP32-pipe variant; outside the parity bar, see DESIGN.md section 3)
    secs32, _, _ = timed_device_loop(lambda: eng.fabrik_solve_device(xyz, angles, precision="f32"), max(2, args.steps // 2), 3)
    peak_fp32_k1 = eng.microbench_fma("f32")
    f32_mode = {"value": n * world * max(2, args.steps // 2) / secs32, "unit": UNIT,
                "fp32_frac": flops_per_launch / (secs32 / max(2, args.steps // 2)) / 1e12 / peak_fp32_k1,
                "peak_fp32_tflops": peak_fp32_k1,
                "note": "fp32 iterate + fp64 angle extraction; ~0.3 % of rows leave the 1e-4 rad band (tests/test_gpu_fabrik.py)"}
    eng.fabrik_solve_device(xyz, angles)  # restore the fp64 result for the FK error below
    # FK position error of the solved angles (K3), once, outside the timed loop
    err = torch.empty(n, device=dev, dtype=torch.float32)
    eng.stats_reset_torch()
    fk_secs, _, _ = timed_device_loop(lambda: eng.fk_device(angles, targets=xyz, err=err), 3, 1)
    eng.stats_reset_torch()
    eng.fk_device(angles, targets=xyz, err=err)
    fk_stats = reduce_stats(eng.stats_fetch_torch())
    reach = (xyz - torch.tensor([0.0, 0.0, 2.0], device=dev)).norm(dim=1) <= 6.0
    fk_error = {"mean_all": fk_stats.mean_fk_error,
                "median_reachable": float(err[reach][:20_000_000].median().item()),
                "reachable_fraction": float(reach.float().mean().item()),
                "fk_rows_per_s": n * world * 3 / fk_secs,
                "fk_hbm_frac": n * 32 * 3 / fk_secs / 1e9 / hbm_peak}
    # the same error as part of the solve call (ikb_fabrik_solve_device with fk_err_out): above 2^10 rows that is
    # K1 + K3 on one stream (the fused epilogue measured 2.2 ms extra at 100 M rows against 0.8 ms for K3), below it
    # K1's fused epilogue (one launch)
    fused_steps = max(2, args.steps // 2)
    fused_secs, _, _ = timed_device_loop(lambda: eng.fabrik_solve_device(xyz, angles, fk_err=err), fused_steps, 1)
    eng.stats_reset_torch()
    eng.fabrik_solve_device(xyz, angles, fk_err=err)
    fused_stats = reduce_stats(eng.stats_fetch_torch())
    small = 512
    s_xyz, s_ang, s_err = xyz[:small].contiguous(), angles[:small].contiguous(), err[:small].contiguous()
    s_plain, _, _ = timed_device_loop(lambda: eng.fabrik_solve_device(s_xyz, s_ang), 20, 3)
    s_fused, _, _ = timed_device_loop(lambda: eng.fabrik_solve_device(s_xyz, s_ang, fk_err=s_err), 20, 3)
    s_two, _, _ = timed_device_loop(lambda: (eng.fabrik_solve_device(s_xyz, s_ang),
                                             eng.fk_device(s_ang, targets=s_xyz, err=s_err)), 20, 3)
    fk_error["in_solve_call"] = {"ms_per_step": fused_secs / fused_steps * 1e3, "mean_all": fused_stats.mean_fk_error,
                                 "extra_ms_vs_plain_solve": (fused_secs / fused_steps - secs / args.steps) * 1e3,
                                 "separate_fk_kernel_ms": fk_secs / 3 * 1e3,
                                 "small_batch_512_us": {"plain": s_plain / 20 * 1e6, "fused_epilogue": s_fused / 20 * 1e6,
                                                         "two_launches": s_two / 20 * 1e6}}
    del s_xyz, s_ang, s_err

    # interior (fully reachable) box, secondary figure
    xyz_r = device_points(min(n, 50_000_000), INTERIOR_BOX, 99 + rank)
    ang_r = torch.empty(xyz_r.shape[0], 4, device=dev, dtype=torch.float32)
    eng.stats_reset_torch()
    eng.fabrik_solve_device(xyz_r, ang_r)
    one_r = eng.stats_fetch_torch()
    secs_r, _, _ = timed_device_loop(lambda: eng.fabrik_solve_device(xyz_r, ang_r), args.steps, 3)
    it_r = torch.empty(xyz_r.shape[0], device=dev, dtype=torch.int32)
    eng.fabrik_solve_device(xyz_r, ang_r, iters=it_r)
    parity["fabrik_interior_box"] = fabrik_parity(xyz_r, ang_r, it_r, "cfg 3 (R) cube_random reachable interior")
    del it_r
    interior = {"value": xyz_r.shape[0] * world * args.steps / secs_r, "unit": UNIT,
                "rows_per_gpu": xyz_r.shape[0], "mean_iterations": one_r.sum_iterations / xyz_r.shape[0],
                "fp64_frac": fabrik_algorithmic_flops(one_r.sum_iterations, xyz_r.shape[0]) /
                             (secs_r / args.steps) / 1e12 / peak_fp64}
    del xyz_r, ang_r, err

    # ---- the final result gather (north star: "NCCL is used only for the final result gather") -------
    gather = None
    if world > 1:
        sh = ShardedFabrik(ik)
        n_total = n * world
        full = torch.empty(n_total, 4, device=dev, dtype=torch.float32) if rank == 0 else None
        g_steps = max(2, min(args.steps, 5))
        GATHER_CHUNK = 1 << 24   # rows per K1 launch when chunks are shipped while the next one is solved
        only_secs, _, _ = timed_device_loop(lambda: gather_rows(angles, n_total, dst=0, out=full), g_steps, 2)
        both_secs, _, _ = timed_device_loop(
            lambda: sh.ikine_device(xyz, angles, n_total=n_total, gather_dst=0, gather_out=full, check=False,
                                    chunk_rows=GATHER_CHUNK, gather_mode="nccl"), g_steps, 2)
        # every shard must have landed at its own rows of rank 0's buffer
        probe = torch.zeros(world, dtype=torch.float64, device=dev)
        probe[rank] = angles[:4096].double().sum() + angles[-4096:].double().sum()
        dist.all_reduce(probe, op=dist.ReduceOp.SUM)
        order_ok = None
        if rank == 0:
            got = torch.stack([full[r * n: r * n + 4096].double().sum() + full[(r + 1) * n - 4096: (r + 1) * n].double().sum()
                               for r in range(world)])
            order_ok = bool(torch.equal(got, probe))
        # the same with copy-engine pushes into rank 0's buffer (symmetric memory): no NCCL kernels next to K1
        peer = None
        try:
            pg = PeerGather(n_total, 4, torch.float32, dev, dst=0)
            p2p_secs, _, _ = timed_device_loop(
                lambda: sh.ikine_device(xyz, angles, n_total=n_total, gather_dst=0, check=False, chunk_rows=GATHER_CHUNK,
                                        peer_gather=pg), g_steps, 2)
            probe2 = torch.zeros(world, dtype=torch.float64, device=dev)
            probe2[rank] = angles[:4096].double().sum() + angles[-4096:].double().sum()
            dist.all_reduce(probe2, op=dist.ReduceOp.SUM)
            ok2 = None
            if rank == 0:
                got2 = torch.stack([pg.buf[r * n: r * n + 4096].double().sum() + pg.buf[(r + 1) * n - 4096: (r + 1) * n].double().sum()
                                    for r in range(world)])
                ok2 = bool(torch.equal(got2, probe2))
            peer = {"overlapped_ms": p2p_secs / g_steps * 1e3,
                    "solve_plus_gather_over_solve": (p2p_secs / g_steps) / (secs / args.steps), "order_verified": ok2,
                    "how": "PeerGather: finished 16 Mi-row chunks pushed into rank 0's buffer (torch symmetric memory mapped "
                           "over NVLink) with device-to-device copies on a side stream -- copy engines, no SMs"}
            del pg
        except Exception as exc:   # symmetric memory unavailable on this box / torch build
            peer = {"unavailable": f"{type(exc).__name__}: {exc}"[:300]}
        moved = (world - 1) * n * 16
        gather = {"rows_total": n_total, "dst": 0, "bytes_into_dst": moved,
                  "ms": only_secs / g_steps * 1e3, "GBps_into_dst": moved / (only_secs / g_steps) / 1e9,
                  "solve_ms": secs / args.steps * 1e3, "overlapped_ms": both_secs / g_steps * 1e3,
                  "solve_plus_gather_over_solve": (both_secs / g_steps) / (secs / args.steps),
                  "order_verified": order_ok, "copy_engine_push": peer,
                  "chunk_rows": GATHER_CHUNK,
                  "how": "ShardedFabrik.ikine_device: K1 per 16 Mi-row chunk, finished chunks shipped to rank 0 with NCCL "
                         "send/recv (point-to-point, received in place) while the next chunk is solved; `ms` is the "
                         "same gather after the solve, not overlapped.  All other ranks' rows converge on ONE GPU, so "
                         "the gather is bound by that GPU's NVLink ingest: (N-1) x 1.6 GB at GBps_into_dst"}
        del full

    # ---- FABRIK end to end: host buffers through the public ikine() call --------------------------
    # page-locked buffers from the library (cudaHostAlloc by this rank after its CPU binding: NUMA-local, not portable)
    m = args.e2e_rows or n
    h_in, h_out = eng.pinned_empty((m, 3), np.float32), eng.pinned_empty((m, 4), np.float32)
    torch.from_numpy(h_in).copy_(xyz[:m])
    del xyz, angles
    e2e_steps = max(2, min(args.steps, 5))
    for _ in range(2):
        ik.ikine(h_in, out=h_out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ik.ikine(h_in, out=h_out)          # H2D + solve + D2H, synchronous at the API boundary
    torch.cuda.synchronize()
    e2e_secs = max_over_ranks(time.perf_counter() - t0)
    # copy ceiling: the same buffers through the same 3-slot pipeline with the kernels removed, all ranks at once
    eng.copy_pipeline(h_in, h_out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.copy_pipeline(h_in, h_out)
    copy_secs = max_over_ranks(time.perf_counter() - t0)
    legs = {}
    for name, src, dst in (("h2d_only", h_in, None), ("d2h_only", None, h_out)):
        eng.copy_pipeline(src, dst)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            eng.copy_pipeline(src, dst)
        leg_secs = max_over_ranks(time.perf_counter() - t0)
        legs[name] = (m * world * e2e_steps * (12 if src is not None else 16)) / leg_secs / 1e9
    e2e = {"value": m * world * e2e_steps / e2e_secs, "unit": UNIT,
           "h2d_bytes_per_step": m * 12 * world, "d2h_bytes_per_step": m * 16 * world,
           "rows_per_gpu": m, "steps": e2e_steps,
           "api": "FabrikInverseKinematics.ikine(float32 ndarray, out=pinned float32 ndarray)",
           "copy_ceiling": {"value": m * world * e2e_steps / copy_secs, "unit": UNIT,
                            "what": "ikb_copy_pipeline_host: the same pinned buffers, chunking and 3 streams per GPU, "
                                    "kernels removed, all ranks concurrently",
                            "aggregate_GBps_both_directions": m * world * e2e_steps * 28 / copy_secs / 1e9,
                            "h2d_alone_GBps": legs["h2d_only"], "d2h_alone_GBps": legs["d2h_only"]},
           "frac_of_copy_ceiling": copy_secs / e2e_secs,
           "pinned_memory": "ikb_host_alloc (cudaHostAlloc, default flags) by each rank"}
    del h_in, h_out

    # ---- ANN (config 2) -------------------------------------------------------------------------------
    ann_block = None
    if not args.skip_ann:
        from inversekinematicsann_b200 import models  # synthetic weights (the shipped .h5 is absent) + shipped scalers
        ann = AnnInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits, device=local_rank)
        trained = os.path.join(os.path.dirname(os.path.abspath(__file__)), "models", "roboarm_b200_r01")
        if os.path.exists(trained + ".npz"):
            ann.load_model(trained + ".h5")    # reference file convention (ann.py:78-85); weights come from the .npz
            weights_note = ("models/roboarm_b200_r01: the reference architecture trained by tools/train_fabrik_model.py "
                            "on FABRIK-labelled targets (the reference's own .h5 is missing from its tree, so parity "
                            "with Keras stays unpinned)")
        else:
            W, b = models.synthetic_weights()
            ann.ann.set_model(W, b, models.SHIPPED_MEAN_X, models.SHIPPED_SCALE_X, models.SHIPPED_MEAN_Y,
                              models.SHIPPED_SCALE_Y)
            weights_note = "synthetic seeded Glorot (no trained model under models/; parity unpinned)"
        W, b = ann.ann.model.kernels, ann.ann.model.biases
        aeng = ann.ann._ensure_uploaded()
        an = args.ann_rows
        # configs[1]: random_dist points = position_generator.random_distribution(n, limits, 'normal', std_dev=0.5)
        # (per-axis truncated normal around 0 inside the workspace box), generated on the device (csrc/generators.cu)
        from inversekinematicsann_b200.robot.position_generator import TrainingDataGenerator as Gen
        axyz = Gen.random_distribution_device(an, R.effector_workspace_limits, 'normal', 0.5, seed=4321 + rank,
                                              device=local_rank)
        aout = torch.empty(an, 4, device=dev, dtype=torch.float32)
        a_steps = max(2, min(args.steps, 5))
        bf16_peak = json.load(open(peaks_path)).get("bf16_tflops", 1590.0) if os.path.exists(peaks_path) else 1590.0
        flops = 2.0 * aeng.mlp_macs_per_row * an
        modes = {}
        for mode in ("fp16x3_ts", "fp16x3", "fp32"):
            a_launch0 = aeng.launch_count
            a_secs, _, _ = timed_device_loop(lambda: aeng.ann_solve_device(axyz, aout, mode=mode), a_steps, 3)
            gpu_launches += (aeng.launch_count - a_launch0 - 3) * world
            modes[mode] = a_secs / a_steps
            if mode == "fp16x3_ts":     # the default mode, the one `ann.value` reports
                dump("ann_angles", aout)
        # parity of the default mode's launch on the bench's own rows: NumPy fp32 / fp64 restatements of ann.py:70-76
        # and an independent torch-CPU fp32 evaluation (oracle/torch_oracle.py); FK error with the oracle's FK
        aeng.ann_solve_device(axyz, aout, mode="fp16x3_ts")
        from oracle import c_oracle, np_oracle, torch_oracle
        from threadpoolctl import threadpool_limits
        pm = min(PARITY_ROWS, an)
        p_pts = axyz[:pm].double().cpu().numpy()
        p_got = aout[:pm].cpu().numpy()
        sc = (ann.ann.x_data_skaler.mean_, ann.ann.x_data_skaler.scale_, ann.ann.y_data_skaler.mean_,
              ann.ann.y_data_skaler.scale_)
        with threadpool_limits(limits=os.cpu_count() or 1):
            p32 = np_oracle.mlp_predict(p_pts, W, b, *sc, dtype=np.float32)
            p64 = np_oracle.mlp_predict(p_pts, W, b, *sc, dtype=np.float64)
        pt32 = torch_oracle.mlp_predict_fresh_process(p_pts, W, b, *sc)
        d32 = np.abs(p_got.astype(np.float64) - p32).max(axis=1)
        _, _, fk_ref = c_oracle.fk_positions(p32.astype(np.float64), targets=p_pts)
        _, _, fk_eng = c_oracle.fk_positions(p_got.astype(np.float64), targets=p_pts)
        a_par = finish_parity(reduce_parity({
            "rows": pm, "n_excluded_degenerate": 0, "max_abs_dtheta": float(d32.max()),
            "p99_abs_dtheta": float(np.quantile(d32, 0.99)), "n_gt_tol": int((d32 > 1e-5).sum()),
            "max_abs_dtheta_vs_fp64": float(np.abs(p_got - p64).max()),
            "max_abs_dtheta_vs_torch": float(np.abs(p_got.astype(np.float64) - pt32).max()),
            "max_oracle_fp32_vs_fp64": float(np.abs(p32 - p64).max()),
            "sum_fk_ref": float(fk_ref.sum()), "sum_fk_eng": float(fk_eng.sum()),
            "max_fk_diff": float(np.abs(fk_ref - fk_eng).max())}), 1e-5)
        a_par["what"] = (f"cfg 2 random_dist: rows [0, {pm}) of every rank's shard, mlp_tc2_kernel output vs the NumPy fp32 "
                         f"restatement (max_abs_dtheta, p99, frac), vs its fp64 form and vs torch-CPU fp32 F.linear+tanh; bar "
                         f"1e-5 rad vs fp32.  Checker weights = this repo's trained network: parity with Keras itself is "
                         f"UNPINNED (the reference's .h5 is absent from its tree)")
        parity["ann_random_dist"] = a_par
        del p32, p64, pt32
        a_in, a_res = aeng.pinned_empty((an, 3), np.float32), aeng.pinned_empty((an, 4), np.float32)
        torch.from_numpy(a_in).copy_(axyz)
        ann.ikine(a_in, out=a_res)
        barrier()
        t0 = time.perf_counter()
        for _ in range(a_steps):
            ann.ikine(a_in, out=a_res)      # default mode = fp16x3_ts
        ae2e = max_over_ranks(time.perf_counter() - t0)
        del a_in, a_res
        peak_fp32 = aeng.microbench_fma("f32")
        tc_s = modes["fp16x3_ts"]
        # FK round trip of the predictions (BASELINE metric: mean FK position error), on the rows FABRIK can reach
        a_err = torch.empty(an, device=dev, dtype=torch.float32)
        aeng.ann_solve_device(axyz, aout, mode="fp16x3_ts", fk_err=a_err)   # error from the kernel's own output stage
        fused_a_secs, _, _ = timed_device_loop(
            lambda: aeng.ann_solve_device(axyz, aout, mode="fp16x3_ts", fk_err=a_err), a_steps, 1)
        f_ang = torch.empty(an, 4, device=dev, dtype=torch.float32)
        f_it = torch.empty(an, device=dev, dtype=torch.int32)
        f_err = torch.empty(an, device=dev, dtype=torch.float32)
        eng.fabrik_solve_device(axyz, f_ang, iters=f_it)
        eng.fk_device(f_ang, targets=axyz, err=f_err)
        reach = (f_it < 100) & (f_err <= 1e-2)
        ann_fk = {"rows_reachable": int(reach.sum()), "ann_mean": float(a_err[reach].double().mean()),
                  "ann_median": float(a_err[reach].median()), "fabrik_mean_same_rows": float(f_err[reach].double().mean()),
                  "angle_abs_diff_vs_fabrik_mean": float((aout[reach] - f_ang[reach]).abs().double().mean()),
                  "fused_ms_per_step": fused_a_secs / a_steps * 1e3,
                  "note": "rows of the workspace sample that FABRIK solves to <= 1e-2 (the population the model was "
                          "trained on); errors come from the ANN kernel's fused FK epilogue"}
        del a_err, f_ang, f_it, f_err
        ann_traffic = None
        tpath2 = os.path.join(ROOT, "profiles", "k2_ts_traffic.json")
        if os.path.exists(tpath2):
            t2 = json.load(open(tpath2))
            if t2.get("rows") == an:
                ann_traffic = t2.get("dram_bytes_per_launch", t2.get("dram_bytes_read", 0) + t2.get("dram_bytes_write", 0))
        # executed tensor-core work: 3 partial products (x_hi w_hi, x_lo w_hi, x_hi w_lo) on the 512-padded layers
        hp = 128 * ((max(aeng.mlp_dims[1:-1]) + 127) // 128)
        executed = 3 * 2.0 * hp * hp * (len(aeng.mlp_dims) - 3) * an
        ann_block = {
            "metric": "IK solves/sec (ANN 3->12x500 tanh->4, fused scaler+MLP+scaler)", "value": an * world / tc_s,
            "unit": UNIT, "rows_per_gpu": an, "ms_per_step": tc_s * 1e3, "dtype": "f16x2-split inputs, f32 accumulate",
            "workload": "BASELINE configs[1]: 1M random_dist points (truncated normal, std 0.5, workspace limits) per GPU, "
                        "float32 [n,3] in HBM -> float32 [n,4]",
            "mode": "IKB_MLP_FP16X3_TS: tcgen05 kind::f16, hi/lo split of activations and weights, x_hi as TMEM A operand, fp32 accumulators in TMEM",
            "weights": weights_note, "fk_error": ann_fk,
            "e2e": {"value": an * world * a_steps / ae2e, "unit": UNIT, "h2d_bytes_per_step": an * 12 * world,
                    "d2h_bytes_per_step": an * 16 * world},
            "roofline": {"kernel": "mlp_tc2_kernel", "bound": "tensor", "achieved": flops / tc_s / 1e12, "peak": bf16_peak,
                         "unit": "TFLOP/s", "frac": flops / tc_s / 1e12 / bf16_peak,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if os.path.exists(peaks_path) else "fallback",
                         "flops_per_row": 2 * aeng.mlp_macs_per_row,
                         "executed_tensor_tflops": executed / tc_s / 1e12, "executed_frac": executed / tc_s / 1e12 / bf16_peak,
                         "note": "fp32-grade results need 3 fp16 partial products per algorithmic MAC, so frac <= 1/3 by construction",
                         "traffic": ann_traffic},
            "fp16x3_ss": {"value": an * world / modes["fp16x3"], "unit": UNIT, "kernel": "mlp_tc_kernel",
                          "roofline": {"bound": "tensor", "achieved": flops / modes["fp16x3"] / 1e12, "peak": bf16_peak,
                                       "unit": "TFLOP/s", "frac": flops / modes["fp16x3"] / 1e12 / bf16_peak}},
            "fp32_simt": {"value": an * world / modes["fp32"], "unit": UNIT, "kernel": "mlp_simt_kernel",
                          "roofline": {"bound": "fp32", "achieved": flops / modes["fp32"] / 1e12, "peak": peak_fp32,
                                       "unit": "TFLOP/s", "frac": flops / modes["fp32"] / 1e12 / peak_fp32}},
        }
        # BASELINE config 4: 125 M uniform workspace targets per GPU (1e9 on 8 GPUs), predictions + FK round trip,
        # the per-GPU (sum, count) reduced across ranks; same kernel, the error comes from its fused epilogue
        del axyz, aout
        big = args.ann_big_rows
        if big > 0:
            bxyz = device_points(big, WORKSPACE_BOX, 777 + rank)
            bout = torch.empty(big, 4, device=dev, dtype=torch.float32)
            aeng.stats_reset_torch()
            b_secs, _, _ = timed_device_loop(lambda: aeng.ann_solve_device(bxyz, bout, mode="fp16x3_ts", fk_stats=True), 2, 1)
            b_stats = reduce_stats(aeng.stats_fetch_torch())
            gpu_launches += 2 * world
            ann_block["config4_fk_round_trip"] = {
                "value": big * world * 2 / b_secs, "unit": UNIT, "rows_per_gpu": big, "rows_total": big * world,
                "ms_per_step": b_secs / 2 * 1e3, "mean_fk_error_all_rows": b_stats.mean_fk_error,
                "rows_in_error_mean": b_stats.n_fk_error // 3,
                "roofline_frac": 2.0 * aeng.mlp_macs_per_row * big / (b_secs / 2) / 1e12 / bf16_peak,
                "note": "uniform over the whole workspace box, 37 % of which FABRIK (and hence the training set) cannot "
                        "reach, so the all-rows mean is dominated by unreachable targets; see fk_error for reachable rows"}
            del bxyz, bout
        if rank == 0 and not args.skip_cpu:
            rows = 100_000
            ann_block["cpu_baseline"] = {"value": cpu_ann_rate(rows, W, b), "unit": UNIT, "cores": os.cpu_count(),
                                         "kind": "port", "sample": f"{rows} targets, NumPy fp32 restatement of ann.py:70-76 "
                                                                   f"(BLAS threads = host cores); Keras is not installed"}

    clocks = None
    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(w0, w1)

    # ---- the other BASELINE configs as drop-in latency / wire-path figures (rank 0, not part of `value`) ----
    extras = None
    if rank == 0:
        from inversekinematicsann_b200 import wire
        from inversekinematicsann_b200.robot.position_generator import TrainingDataGenerator as G
        spring = G.spring(50, 2, 3, 6)                      # configs[0]: cli.py --shape spring example (cli.py:195)
        ik.ikine(spring)
        t0 = time.perf_counter()
        for _ in range(20):
            ik.ikine(spring)                                # list in, list out, exactly the CLI's call
        spring_ms = (time.perf_counter() - t0) / 20 * 1e3
        circ = G.circle_device(2, 10_000_000, (2, 0, 2), dtype="float32").cpu().numpy()   # configs[4]
        body = wire.encode_binary_request(circ)
        wire.handle_request(ik, body, zero_copy=True)
        t0 = time.perf_counter()
        for _ in range(3):
            reply = wire.handle_request(ik, body, zero_copy=True)
        broker_s = (time.perf_counter() - t0) / 3
        t0 = time.perf_counter()
        reply_bytes = wire.handle_request(ik, body)          # independent bytes copy of the reply
        broker_copy_s = time.perf_counter() - t0
        # parity of the reply's first rows (cfg 5 circle) against the oracle
        from oracle import c_oracle
        c_oracle.set_num_threads(os.cpu_count() or 1)
        dec = wire.decode_binary_reply(reply)
        c_want = c_oracle.fabrik_ikine(circ[:PARITY_ROWS].astype(np.float64))
        c_d = np.abs(dec["angles"][:PARITY_ROWS].astype(np.float64) - c_want["angles"]).max(axis=1)
        parity["broker_circle"] = {"rows": int(c_d.shape[0]), "max_abs_dtheta": float(c_d.max()),
                                   "p99": float(np.quantile(c_d, 0.99)), "frac_gt_0.0001": float((c_d > 1e-4).mean()),
                                   "what": "cfg 5: first rows of the IKB1 reply (float32) for the 10 M-point circle vs "
                                           "oracle/ik_oracle.c, rank 0"}
        extras = {"cli_spring_50_points_ms": spring_ms,
                  "cli_spring_reference_ms": "~30 (1 678 solves/s, BASELINE.md)",
                  "broker_binary_10M_circle": {"value": 10_000_000 / broker_s, "unit": UNIT,
                                               "request_bytes": len(body), "reply_bytes": len(reply),
                                               "reply_dtype": str(dec["angles"].dtype),
                                               "with_bytes_copy_of_reply": 10_000_000 / broker_copy_s,
                                               "path": "wire.handle_request(IKB1 payload, zero_copy=True) = decode (view of the "
                                                       "pageable request body) + ikine(out=pinned reply arena) + 16-byte header; "
                                                       "1 GPU"}}
        del reply, dec, reply_bytes
    # cfg 5 as BASELINE words it: one 10 M-point request served by the N-GPU sharded engine (all ranks take part)
    if world > 1:
        sh5 = ShardedFabrik(ik)
        req = G5 = None
        if rank == 0:
            req = wire.decode_binary_request(body)
            G5 = eng.pinned_empty((req.shape[0], 4), np.float32)
        sh5.ikine_from_root(req, root=0, out=G5)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            sh5.ikine_from_root(req, root=0, out=G5)
        sharded_s = max_over_ranks(time.perf_counter() - t0) / 3
        if rank == 0:
            same = bool(np.array_equal(G5, wire.decode_binary_reply(wire.handle_request(ik, body, zero_copy=True))["angles"]))
            extras["broker_sharded_10M_circle"] = {
                "value": 10_000_000 / sharded_s, "unit": UNIT, "n_gpus": world, "identical_to_one_gpu_reply": same,
                "path": "ShardedFabrik.ikine_from_root: request H2D on rank 0, shards to the other GPUs and angles back over "
                        "NCCL send/recv, D2H into a pinned reply on rank 0",
                "note": "one request crosses PCIe once, on rank 0's link (120 MB in, 160 MB out): that link bounds the "
                        "path, the 0.5 ms solve does not, so N GPUs cannot beat one for a single request of this size"}

    cpu_baseline = None
    if rank == 0 and not args.skip_cpu:
        sample, threads = calibrated_cpu_sample(WORKSPACE_BOX)
        rate, threads, mean_it = cpu_fabrik_rate(sample, WORKSPACE_BOX)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"the first {sample} rows of this run's rank-0 input (mean {mean_it:.1f} iterations), "
                                  f"oracle/ik_oracle.c = C restatement of fabrik.py/inverse.py with OpenMP on all host "
                                  f"threads; the pure-Python reference runs ~4e2 solves/s/core on this workload "
                                  f"(BASELINE.md) and does not exist on the GPU box"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "rows_per_gpu": n, "input": "float32 [n,3] AoS in HBM (1.2 GB per GPU, > 126 MB L2: no flush needed)",
                       "output": "float32 [n,4]", "fabrik_precision": "fp64 iterate + fp64 angle extraction",
                       "mean_iterations": total.sum_iterations / (n * world),
                       "iteration_capped_fraction": total.n_iter_capped / (n * world),
                       "sharding": f"contiguous ranges, {world} rank(s), no data-path collective in `value` "
                                   f"(the final gather to rank 0 is timed separately under \"gather\")",
                       "rank_cpu_affinity": numa_cpus or "unchanged"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(gpu_launches), "roofline": roofline,
            "parity": parity, "gather": gather,
            "cpu_baseline": cpu_baseline, "fk_error": fk_error, "fabrik_interior_box": interior,
            "fabrik_f32_mode": f32_mode, "ann": ann_block,
            "other_configs": extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
