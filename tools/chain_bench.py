#!/usr/bin/env python3
"""Throughput of Fabrik.calculate on J-point chains (csrc/fabrik_chain.cu).  Prints one JSON line.

Workloads: unit links, J in --js; goals uniform in a ball about S of radius 1.25 (J - 1) (about half of them
reachable) and 0.9 (J - 1) (all reachable); the straight seed chain (n_init = 1) or a random chain per row
(n_init = n).  Rows per workload are sized to 4x the 126 MB L2, so every timed call streams from HBM.

Per workload: kernel time of `IkEngine.fabrik_chain_device` from CUDA events after a warm-up (median of --reps), chains
per second, the summed passes, algorithmic fp64 TFLOP/s (32 J - 14 flops per pass) against the measured fp64 FMA rate
of `ikb_microbench_fma`, the bytes a row moves and which bound applies.  The fp64-pipe instructions of the kernel
instantiation come from its SASS (cuobjdump): the IEEE division and square root sequences cost far more than the one
flop each counts for.

--compare-lib PATH times the same workloads through the host entry point of this build and of another build of
libikb200.so, alternating, with kernel times from torch.profiler, and checks that both builds compute the same chains.
A build without `ikb_fabrik_chain_host` runs only J = 4, through `ikb_fabrik_calculate_host`."""
import argparse
import ctypes
import json
import os
import re
import shutil
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 * 2 ** 20


def flops_per_pass(J):
    return 32 * J - 14


def bytes_per_row(J, per_row):
    return 24 + 24 * J * per_row + 24 * J + 4


def workload_rows(J, per_row, cap):
    return int(min(cap, max(1 << 16, 4 * L2_BYTES // bytes_per_row(J, per_row))))


def make_inputs(J, n, radius, per_row, seed):
    rng = np.random.default_rng(seed)
    links = np.ones(J)
    if per_row:
        init = rng.standard_normal((n, J, 3)).cumsum(axis=1)
        S = init[:, 0]
    else:
        init = np.zeros((J, 3))
        init[:, 2] = np.arange(J, dtype=np.float64)
        S = np.zeros((1, 3))
    u = rng.standard_normal((n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    goals = S + u * (radius * max(J - 1, 1) * rng.uniform(0, 1, (n, 1)) ** (1 / 3))
    return links, np.ascontiguousarray(init), np.ascontiguousarray(goals)


def gpu_info():
    info = {}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.splitlines()[0]
        name, power, clock = [v.strip() for v in out.split(",")]
        info = {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError) as exc:
        info = {"gpu_query_error": str(exc)}
    return info


def sass_fp64_counts(lib_path, J, jreg):
    """fp64-pipe instructions of the kernel instantiation that runs J points: {opcode: count} or None."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        return None
    inst = J if J <= jreg else 0
    sass = subprocess.run([tool, "-sass", lib_path], capture_output=True, text=True).stdout
    m = re.search(r"Function : (\S*fabrik_chain_kernelILi%dE\S*)\n(.*?)(?=\n\s*Function : |\Z)" % inst, sass, re.S)
    if not m:
        return None
    counts = {}
    for op in re.findall(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9.]+)", m.group(2)):
        base = op.split(".")[0]
        if base in ("DFMA", "DADD", "DMUL", "DSETP", "DMNMX") or op.startswith(("MUFU.RSQ64H", "MUFU.RCP64H")):
            counts[base if base != "MUFU" else op] = counts.get(base if base != "MUFU" else op, 0) + 1
    counts["total"] = sum(counts.values())
    return counts


def run_device(args, workloads, jreg):
    import torch
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    fma = eng.microbench_fma("f64")
    results = []
    for J, radius, per_row in workloads:
        n = workload_rows(J, per_row, args.max_rows)
        links, init, goals = make_inputs(J, n, radius, per_row, seed=J)
        d_init = torch.from_numpy(init).cuda()
        d_goals = torch.from_numpy(goals).cuda()
        out = torch.empty((n, J, 3), dtype=torch.float64, device="cuda")
        iters = torch.empty(n, dtype=torch.int32, device="cuda")
        for _ in range(args.warmup):
            eng.fabrik_chain_device(links, 1e-3, 100, d_init, d_goals, out, iters)
        times = []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.fabrik_chain_device(links, 1e-3, 100, d_init, d_goals, out, iters)
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b) * 1e-3)
        t = float(np.median(times))
        sum_k = int(iters.sum().item())
        flops = sum_k * flops_per_pass(J)
        tflops = flops / t / 1e12
        bpr = bytes_per_row(J, per_row)
        hbm_s = n * bpr / 7.7e12
        fp64_s = flops / (fma * 1e12)
        results.append({
            "J": J, "radius": radius, "n_init": "n" if per_row else 1, "rows": n, "seconds": t,
            "chains_per_s": n / t, "sum_passes": sum_k, "mean_passes": sum_k / n,
            "fp64_tflops_algorithmic": tflops, "fraction_of_fma_microbench": tflops / fma,
            "bytes_per_row": bpr, "bound": "fp64" if fp64_s > hbm_s else "hbm",
            "instantiation": "registers" if J <= jreg else "local memory",
            "sass_fp64": sass_fp64_counts(_native.LIB_PATH, J, jreg),
        })
        del d_init, d_goals, out, iters
    return {"fma_microbench_fp64_tflops": fma, "workloads": results}


class _Build:
    """One libikb200.so and an engine of it with unit links (so that the 4-point entry point solves the same rows)."""

    def __init__(self, path):
        from inversekinematicsann_b200 import _native
        from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
        self.path = path
        self.lib = ctypes.CDLL(path)
        self.chain = hasattr(self.lib, "ikb_fabrik_chain_host")
        vp, i64 = ctypes.c_void_p, ctypes.c_int64
        self.lib.ikb_engine_create.argtypes = [ctypes.POINTER(_native.IkbConfig), ctypes.POINTER(vp)]
        self.lib.ikb_fabrik_calculate_host.argtypes = [vp, vp, i64, vp, i64, vp, vp, ctypes.POINTER(_native.IkbStats)]
        if self.chain:
            self.lib.ikb_fabrik_chain_host.argtypes = [vp, ctypes.c_int32, vp, ctypes.c_double, ctypes.c_int32, vp,
                                                       i64, vp, i64, vp, vp, ctypes.POINTER(_native.IkbStats)]
        cfg = _native.IkbConfig()
        cfg.dh[:] = np.asarray(R.dh_matrix, dtype=np.float64).reshape(-1).tolist()
        cfg.links[:] = [1.0] * 4
        lim = R.effector_workspace_limits
        cfg.limits[:] = [lim["x"][0], lim["x"][1], lim["y"][0], lim["y"][1], lim["z"][0], lim["z"][1]]
        cfg.tol, cfg.max_iter, cfg.device = 1e-3, 100, 0
        self.h = vp()
        if self.lib.ikb_engine_create(ctypes.byref(cfg), ctypes.byref(self.h)) != 0:
            raise RuntimeError(f"{path}: engine creation failed")

    def solve(self, links, init, goals):
        from inversekinematicsann_b200 import _native
        n, J = goals.shape[0], links.shape[0]
        out = np.empty((n, J, 3))
        it = np.empty(n, dtype=np.int32)
        s = _native.IkbStats()
        n_init = 1 if init.ndim == 2 else n
        if self.chain:
            rc = self.lib.ikb_fabrik_chain_host(self.h, J, links.ctypes.data, 1e-3, 100, init.ctypes.data, n_init,
                                                goals.ctypes.data, n, out.ctypes.data, it.ctypes.data, ctypes.byref(s))
        else:
            assert J == 4
            rc = self.lib.ikb_fabrik_calculate_host(self.h, init.ctypes.data, n_init, goals.ctypes.data, n,
                                                    out.ctypes.data, it.ctypes.data, ctypes.byref(s))
        if rc != 0:
            raise RuntimeError(f"{self.path}: solve failed ({rc})")
        return out, it


def kernel_seconds(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    us = 0.0
    for e in prof.key_averages():
        if "fabrik" in e.key:
            us += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return us * 1e-6, res


def run_compare(args, workloads):
    from inversekinematicsann_b200 import _native
    import torch
    torch.cuda.init()
    this, other = _Build(_native.LIB_PATH), _Build(os.path.abspath(args.compare_lib))
    rows = []
    for J, radius, per_row in workloads:
        if not other.chain and J != 4:
            continue
        n = workload_rows(J, per_row, args.max_rows)
        links, init, goals = make_inputs(J, n, radius, per_row, seed=J)
        for b in (this, other):
            b.solve(links, init, goals)  # warm-up
        t = {this.path: [], other.path: []}
        res = {}
        for _ in range(args.reps):
            for b in (other, this):
                s, res[b.path] = kernel_seconds(lambda: b.solve(links, init, goals))
                t[b.path].append(s)
        same = (np.array_equal(res[this.path][0], res[other.path][0]) and
                np.array_equal(res[this.path][1], res[other.path][1]))
        t_this, t_other = float(np.median(t[this.path])), float(np.median(t[other.path]))
        rows.append({"J": J, "radius": radius, "n_init": "n" if per_row else 1, "rows": n,
                     "kernel_s_this": t_this, "kernel_s_other": t_other, "speedup": t_other / t_this,
                     "kernel_s_this_all": t[this.path], "kernel_s_other_all": t[other.path], "same_output": same})
    return {"this_build": "this tree", "other_build": args.compare_label, "workloads": rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--js", default=None, help="comma-separated chain lengths (default 4,6,8,16,J_REG+1,64)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--max-rows", type=int, default=1 << 23)
    ap.add_argument("--jreg", type=int, default=32, help="largest J with a register-resident instantiation")
    ap.add_argument("--compare-lib", default=None, help="another build of libikb200.so to time against")
    ap.add_argument("--compare-label", default="other build", help="what the other build is, for the JSON line")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    js = [int(v) for v in args.js.split(",")] if args.js else [4, 6, 8, 16, args.jreg + 1, 64]
    workloads = [(J, r, p) for J in js for r in (1.25, 0.9) for p in (False, True)]
    res = gpu_info()
    if args.compare_lib:
        res.update(run_compare(args, workloads))
    else:
        res.update(run_device(args, workloads, args.jreg))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
