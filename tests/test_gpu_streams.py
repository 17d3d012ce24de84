"""The device entry points on torch's current stream, and launches on several streams against one engine.

Every device entry point is documented as enqueued on torch's current stream.  The first tests hold an entry point's
inputs back on a side stream (decoys until a ~30 ms sleep on that stream has passed, then the real rows): a launch on
any other stream would read the decoys, or have its outputs cloned before it wrote them.

The persistent kernels (K1, fabrik_chain_kernel, dls_refine_kernel) take their rows from a work counter of the engine's
ring of 16.  Launches on different streams may overlap, so a counter must not be reset for a new launch while the
last launch that used it still runs; the other tests overlap a long launch with the 16th ring-using call after it on
another stream, and 48 launches over three streams."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SLEEP_CYCLES = 60_000_000  # torch.cuda._sleep: ~30 ms at the B200's ~2 GHz SM clock
RING = 16                  # kCounterRing of csrc/capi.cu
STAT_COUNTS = ("n_solved", "sum_iterations", "n_iter_capped", "first_out_of_limits", "first_zero_division",
               "first_domain_error", "first_fk_angle_range", "n_fk_error")  # sum_fk_error is a float sum: order-dependent
CHAIN_LINKS = [2.0, 2.0, 2.0, 2.0]
CHAIN_INIT = [[0.0, 0.0, 0.0], [0.0, 0.0, 2.0], [0.0, 0.0, 4.0], [0.0, 0.0, 6.0]]
SHOULDER = np.array([0.0, 0.0, 2.0])


def _torch():
    import torch
    return torch


def _bits(t):
    torch = _torch()
    return t.view({torch.float64: torch.int64, torch.float32: torch.int32, torch.int32: torch.int32}[t.dtype])


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and _torch().equal(_bits(a), _bits(b))


def _counts(st):
    return {f: getattr(st, f) for f in STAT_COUNTS}


def _cuda(a, dtype=None):
    torch = _torch()
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


def _targets(n, seed, reach=None):
    """n points of the workspace box; reach=False keeps those more than 6.05 m from the shoulder (out of reach)."""
    rng = np.random.default_rng(seed)
    out = []
    while sum(len(o) for o in out) < n:
        p = rng.uniform((0.0, -6.0, -3.0), (6.0, 6.0, 6.0), size=(2 * n + 64, 3))
        if reach is False:
            p = p[np.linalg.norm(p - SHOULDER, axis=1) > 6.05]
        out.append(p)
    return np.vstack(out)[:n]


def _angles(n, seed):
    return np.random.default_rng(seed).uniform(-np.pi, np.pi, size=(n, 4))


def _far_goals(n, seed):
    """Chain goals 10-20 m from the chain's base: out of reach of its 6 m."""
    rng = np.random.default_rng(seed)
    u = rng.standard_normal((n, 3))
    return u / np.linalg.norm(u, axis=1, keepdims=True) * rng.uniform(10.0, 20.0, (n, 1))


@pytest.fixture(scope="module")
def eng():
    """An engine of its own (the shared one's model and statistics belong to other tests), with a network loaded."""
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    from oracle import np_oracle
    e = IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    W, b = np_oracle.synthetic_mlp(seed=5, dims=np_oracle.LAYER_DIMS)
    e.mlp_load(W, b, np_oracle.SHIPPED_MEAN_X, np_oracle.SHIPPED_SCALE_X, np_oracle.SHIPPED_MEAN_Y,
               np_oracle.SHIPPED_SCALE_Y)
    yield e
    _torch().cuda.synchronize()
    e.close()


# ---- (a) every device entry point runs on the caller's stream -------------------------------------------------------
def _plain(eng, inputs, launch):
    """launch(*copies of inputs) on the default stream -> (clones of its outputs, statistics of the call)."""
    torch = _torch()
    torch.cuda.synchronize()
    eng.stats_reset()
    outs = launch(*[t.clone() for t in inputs])
    got = [o.clone() for o in outs]
    torch.cuda.synchronize()
    return got, eng.stats_fetch()


def _late_inputs(eng, real, decoy, launch):
    """launch(*bufs) on a fresh side stream, where bufs hold `decoy` until a ~30 ms sleep on that stream has passed and
    `real` after it -> (clones of the outputs taken on that stream, statistics fetched on that stream)."""
    torch = _torch()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        eng.stats_reset_torch()
        bufs = [d.clone() for d in decoy]
        torch.cuda._sleep(SLEEP_CYCLES)
        for b, r in zip(bufs, real):
            b.copy_(r)
        outs = launch(*bufs)
        got = [o.clone() for o in outs]
        st = eng.stats_fetch_torch()
    s.synchronize()
    return got, st


def _check_on_caller_stream(eng, real, launch):
    """The entry point's outputs and statistics on a side stream with late inputs equal a plain call's, bit for bit; the
    decoys (the real rows rolled by a third) give other outputs or statistics, so a launch that read them would be
    seen."""
    torch = _torch()
    decoy = [torch.roll(t, shifts=t.shape[0] // 3 + 1, dims=0).contiguous() for t in real]
    want, st_want = _plain(eng, real, launch)
    got, st_got = _late_inputs(eng, real, decoy, launch)
    for i, (w, g) in enumerate(zip(want, got)):
        assert _same_bits(w, g), f"output {i} differs from the plain call's"
    assert _counts(st_got) == _counts(st_want)
    wrong, st_wrong = _plain(eng, decoy, launch)
    assert any(not _same_bits(w, d) for w, d in zip(want, wrong)) or _counts(st_wrong) != _counts(st_want), \
        "the decoys must give other results"
    return st_want


@pytest.mark.parametrize("n", [1000, 70_000], ids=["fused_fk", "k3_fk"])
@pytest.mark.parametrize("out_dtype", ["float32", "float64"])
@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_fabrik_solve_device_on_caller_stream(eng, precision, out_dtype, n):
    """n <= 1024 takes K1 with the fused FK error, larger n K1 then K3 on the same stream."""
    torch = _torch()
    dt = getattr(torch, out_dtype)

    def launch(xyz):
        out = torch.empty((xyz.shape[0], 4), dtype=dt, device="cuda")
        it = torch.empty(xyz.shape[0], dtype=torch.int32, device="cuda")
        err = torch.empty(xyz.shape[0], dtype=dt, device="cuda")
        eng.fabrik_solve_device(xyz, out, iters=it, precision=precision, fk_err=err, fk_stats=True)
        return out, it, err

    st = _check_on_caller_stream(eng, [_cuda(_targets(n, 1))], launch)
    assert st.n_solved == n and st.n_fk_error > 0


@pytest.mark.parametrize("mode", ["fp16x3_ts", "fp16x3", "fp32"])
def test_ann_solve_device_on_caller_stream(eng, mode):
    torch = _torch()

    def launch(xyz):
        out = torch.empty((xyz.shape[0], 4), dtype=torch.float32, device="cuda")
        err = torch.empty(xyz.shape[0], dtype=torch.float32, device="cuda")
        eng.ann_solve_device(xyz, out, mode=mode, fk_err=err, fk_stats=True)
        return out, err

    _check_on_caller_stream(eng, [_cuda(_targets(5000, 2))], launch)


def test_fk_device_error_ring_on_caller_stream(eng):
    """float32 angles and targets, errors only, >= 4 trips per warp slot: fk_error_stream_kernel (the cp.async ring)
    plus the pair kernel on the last 37 rows."""
    torch = _torch()
    n = 400_037

    def launch(angles, targets):
        err = torch.empty(angles.shape[0], dtype=torch.float32, device="cuda")
        eng.fk_device(angles, targets=targets, err=err)
        return (err,)

    _check_on_caller_stream(eng, [_cuda(_angles(n, 3), torch.float32), _cuda(_targets(n, 4), torch.float32)], launch)


def test_fk_device_positions_on_caller_stream(eng):
    torch = _torch()

    def launch(angles):
        pos = torch.empty((angles.shape[0], 3), dtype=torch.float64, device="cuda")
        eng.fk_device(angles, pos=pos)
        return (pos,)

    _check_on_caller_stream(eng, [_cuda(_angles(5000, 5))], launch)


@pytest.mark.parametrize("what,dtype", [("matrices", "float64"), ("joints", "float32")])
def test_fk_transforms_device_on_caller_stream(eng, what, dtype):
    torch = _torch()

    def launch(angles):
        tail = (4, 4, 4) if what == "matrices" else (4, 3)
        out = torch.empty((angles.shape[0],) + tail, dtype=angles.dtype, device="cuda")
        eng.fk_transforms_device(angles, out, what=what)
        return (out,)

    _check_on_caller_stream(eng, [_cuda(_angles(3000, 6), getattr(torch, dtype))], launch)


@pytest.mark.parametrize("what,dtype", [("geometric", "float64"), ("position", "float32")])
def test_jacobian_device_on_caller_stream(eng, what, dtype):
    torch = _torch()

    def launch(angles):
        rows = 6 if what == "geometric" else 3
        jac = torch.empty((angles.shape[0], rows, 4), dtype=angles.dtype, device="cuda")
        manip = torch.empty(angles.shape[0], dtype=angles.dtype, device="cuda")
        eng.jacobian_device(angles, jac, what=what, manip=manip)
        return jac, manip

    _check_on_caller_stream(eng, [_cuda(_angles(3000, 7), getattr(torch, dtype))], launch)


@pytest.mark.parametrize("in_place", [False, True], ids=["per_row_seeds", "in_place"])
def test_dls_refine_device_on_caller_stream(eng, in_place):
    torch = _torch()

    def launch(xyz, seed):
        n = xyz.shape[0]
        out = seed if in_place else torch.empty_like(seed)
        it = torch.empty(n, dtype=torch.int32, device="cuda")
        err = torch.empty(n, dtype=seed.dtype, device="cuda")
        eng.dls_refine_device(xyz, seed, out, iters=it, err=err)
        return out, it, err

    st = _check_on_caller_stream(eng, [_cuda(_targets(4000, 8)), _cuda(_angles(4000, 9))], launch)
    assert st.n_solved == 4000


def test_fabrik_chain_device_on_caller_stream(eng):
    torch = _torch()
    n = 3000
    rng = np.random.default_rng(10)
    init = np.cumsum(rng.standard_normal((n, 4, 3)), axis=1)

    def launch(init, goals):
        out = torch.empty((goals.shape[0], 4, 3), dtype=torch.float64, device="cuda")
        it = torch.empty(goals.shape[0], dtype=torch.int32, device="cuda")
        eng.fabrik_chain_device(CHAIN_LINKS, 1e-3, 100, init, goals, out, it)
        return out, it

    st = _check_on_caller_stream(eng, [_cuda(init), _cuda(rng.uniform(-5.0, 5.0, (n, 3)))], launch)
    assert st.n_solved == n


def test_check_limits_device_on_caller_stream(eng):
    """One offender among the real rows, another at a different row among the decoys; the statistics are fetched on
    the calling stream."""
    xyz = _targets(5000, 11)
    xyz[1234, 2] = 7.0
    st = _check_on_caller_stream(eng, [_cuda(xyz)], lambda t: (eng.check_limits_device(t) or ()))
    assert st.first_out_of_limits == 1234


GENERATOR_CASES = {  # kind -> (params as the *_device forms of TrainingDataGenerator build them, rows, seed)
    "circle": (0, [1.5, 2.0, 0.5, 1.0], 100_003, 0),
    "spring": (1, [4.0, 3.0, 2.0, 100_003], 100_003, 0),
    "cube": (2, [0.1, 5.0, 4.0, 5.0, 0.5, -2.0, 0.0, 50, 40], 50 * 40 * 50, 0),
    "cube_random": (3, [6.0, 12.0, 9.0, 0.0, -6.0, -3.0], 100_003, 99),
    "normal": (4, [0.0, 6.0, -6.0, 6.0, -3.0, 6.0, 0.5], 100_003, 7),
}


@pytest.mark.parametrize("kind", sorted(GENERATOR_CASES))
def test_generators_on_caller_stream(kind):
    """_generate allocates its output on the current stream: a block freed on a side stream while a NaN fill of it
    still waits behind a sleep there is handed out again, so a launch on any other stream would be overwritten."""
    torch = _torch()
    from inversekinematicsann_b200.robot.position_generator import _generate
    code, params, n, seed = GENERATOR_CASES[kind]
    want = _generate(code, params, n, seed=seed)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        block = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        torch.cuda._sleep(SLEEP_CYCLES)
        block.fill_(float("nan"))
        ptr = block.data_ptr()
        del block
        out = _generate(code, params, n, seed=seed)
        got = out.clone()
    s.synchronize()
    assert out.data_ptr() == ptr, "the caching allocator did not hand the freed block out again"
    assert torch.isfinite(want).all()
    assert _same_bits(got, want)


# ---- (b) the 16th ring-using call after a long launch, on another stream --------------------------------------------
def _elapsed(fn):
    """Seconds of fn()'s launches on the current stream (CUDA events), after one warm-up call."""
    torch = _torch()
    fn()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / 1e3


class _Call:
    """One ring-using device call: run() allocates its outputs on the current stream, enqueues the call and returns
    (n, outputs); outputs[1] holds the per-row iteration counts."""

    def __init__(self, eng, kind, n, seed, max_iter=None, far=False, in_place=False):
        torch = _torch()
        self.eng, self.kind, self.n, self.max_iter, self.in_place = eng, kind, n, max_iter, in_place
        if kind == "fabrik":
            self.xyz = _cuda(_targets(n, seed))
        elif kind == "chain":
            self.init = _cuda(np.array(CHAIN_INIT))
            self.goals = _cuda(_far_goals(n, seed) if far else np.random.default_rng(seed).uniform(-5.0, 5.0, (n, 3)))
        elif kind == "dls":
            self.xyz = _cuda(_targets(n, seed, reach=False if far else None))
            self.seed = _cuda(_angles(n, seed + 1))
        else:
            raise ValueError(kind)
        self.torch = torch

    def run(self):
        torch, n, eng = self.torch, self.n, self.eng
        it = torch.empty(n, dtype=torch.int32, device="cuda")
        if self.kind == "fabrik":
            out = torch.empty((n, 4), dtype=torch.float64, device="cuda")
            eng.fabrik_solve_device(self.xyz, out, iters=it)
            return out, it
        if self.kind == "chain":
            out = torch.empty((n, 4, 3), dtype=torch.float64, device="cuda")
            eng.fabrik_chain_device(CHAIN_LINKS, 1e-3, self.max_iter or 100, self.init, self.goals, out, it)
            return out, it
        out = self.seed.clone() if self.in_place else torch.empty_like(self.seed)
        err = torch.empty(n, dtype=torch.float64, device="cuda")
        eng.dls_refine_device(self.xyz, out if self.in_place else self.seed, out, iters=it, err=err,
                              max_iter=self.max_iter)
        return out, it, err


def _long_call(eng, variant):
    """A launch of 3 CTAs whose rows are all out of reach, with max_iter sized for ~50 ms: its warps fetch rows again
    only when their first rows finish, long after the calls behind it on the other stream."""
    if variant == "chain":
        n, m0 = 3 * 256, 2000  # 256 threads per CTA, a row per lane
        call = _Call(eng, "chain", n, 21, max_iter=m0, far=True)
    else:
        n, m0 = 3 * 64, 500    # 256 threads per CTA, a row per quad
        call = _Call(eng, "dls", n, 21, max_iter=m0, far=True, in_place=True)
    t = _elapsed(call.run)
    call.max_iter = int(min(2 ** 30, max(m0, m0 * 0.05 / t)))
    return call


@pytest.mark.parametrize("variant", ["chain", "dls"])
def test_ring_reuse_across_streams(eng, variant):
    """Stream A runs one long launch; stream B then makes 15 short ring-using calls and a 16th, which takes A's counter
    of the ring.  Every call's outputs equal its solo run's bits, and the engine's statistics count each row once."""
    torch = _torch()
    a = _long_call(eng, variant)
    kinds = ["fabrik", "chain", "dls"]
    rng = np.random.default_rng(22)
    calls_b = [_Call(eng, kinds[i % 3], int(rng.integers(64, 1001)), 100 + i) for i in range(RING - 1)]
    calls_b.append(_Call(eng, variant, 64, 200, far=True, in_place=variant == "dls"))
    assert calls_b[-1].n < a.n
    calls = [a] + calls_b

    solo = []
    for c in calls:
        torch.cuda.synchronize()
        solo.append([o.clone() for o in c.run()])
    t_a = _elapsed(a.run)
    assert t_a > 0.02, f"the long launch takes {t_a * 1e3:.1f} ms: too short to overlap the calls behind it"

    torch.cuda.synchronize()
    eng.stats_reset()
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(sa):
        out_a = a.run()
    with torch.cuda.stream(sb):
        out_b = [c.run() for c in calls_b]
    torch.cuda.synchronize()
    st = eng.stats_fetch()

    for i, (want, got) in enumerate(zip(solo, [out_a] + out_b)):
        for j, (w, g) in enumerate(zip(want, got)):
            assert _same_bits(w, g), f"call {i} ({calls[i].kind}, n={calls[i].n}): output {j} differs from its solo run"
    assert st.n_solved == sum(c.n for c in calls), (st.n_solved, [c.n for c in calls])
    assert st.sum_iterations == sum(int(s[1].sum()) for s in solo)


# ---- (c) many launches over three streams --------------------------------------------------------------------------
def test_many_launches_over_three_streams(eng):
    """48 launches of K1, the chain kernel, DLS, the network and FK on 1e4-1e6 rows, round-robin over three streams (so
    that ring-using calls j and j + 16 land on different streams): every output equals its solo run's bits, and the
    statistics equal those of the solo runs."""
    torch = _torch()
    rng = np.random.default_rng(31)
    N = 1_000_000
    xyz = _cuda(_targets(N, 32))
    xyz32 = xyz.float()
    ang = _cuda(_angles(N, 33))
    ang32 = ang.float()
    init = _cuda(np.array(CHAIN_INIT))
    modes = ["fp16x3_ts", "fp16x3", "fp32"]
    kinds = ["fabrik", "chain", "dls", "ann", "fk"]

    def make(i):
        kind = kinds[i % len(kinds)]
        n = int(np.exp(rng.uniform(np.log(1e4), np.log(1e6))))
        lo = int(rng.integers(0, N - n + 1))
        sl = slice(lo, lo + n)

        def run():
            it = torch.empty(n, dtype=torch.int32, device="cuda")
            if kind == "fabrik":
                out = torch.empty((n, 4), dtype=torch.float32 if i % 2 else torch.float64, device="cuda")
                eng.fabrik_solve_device(xyz[sl], out, iters=it, precision="f32" if i % 4 == 1 else "f64")
                return out, it
            if kind == "chain":
                out = torch.empty((n, 4, 3), dtype=torch.float64, device="cuda")
                eng.fabrik_chain_device(CHAIN_LINKS, 1e-3, 100, init, xyz[sl], out, it)
                return out, it
            if kind == "dls":
                out = torch.empty((n, 4), dtype=torch.float64, device="cuda")
                eng.dls_refine_device(xyz[sl], ang[sl], out, iters=it)
                return out, it
            if kind == "ann":
                out = torch.empty((n, 4), dtype=torch.float32, device="cuda")
                eng.ann_solve_device(xyz[sl], out, mode=modes[(i // len(kinds)) % 3])
                return (out,)
            if i % 2:
                err = torch.empty(n, dtype=torch.float32, device="cuda")
                eng.fk_device(ang32[sl], targets=xyz32[sl], err=err)
                return (err,)
            pos = torch.empty((n, 3), dtype=torch.float64, device="cuda")
            eng.fk_device(ang[sl], pos=pos)
            return (pos,)

        return kind, n, run

    calls = [make(i) for i in range(48)]
    torch.cuda.synchronize()
    eng.stats_reset()
    solo = []
    for _, _, run in calls:
        solo.append([o.clone() for o in run()])
        torch.cuda.synchronize()
    st_solo = eng.stats_fetch()
    ring = [(k, n, s) for (k, n, _), s in zip(calls, solo) if k in ("fabrik", "chain", "dls")]
    assert st_solo.n_solved == sum(n for _, n, _ in ring)
    assert st_solo.sum_iterations == sum(int(s[1].sum()) for _, _, s in ring)

    eng.stats_reset()
    streams = [torch.cuda.Stream() for _ in range(3)]
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    outs = []
    for i, (_, _, run) in enumerate(calls):
        with torch.cuda.stream(streams[i % 3]):
            outs.append(run())
    torch.cuda.synchronize()
    st = eng.stats_fetch()
    for i, (want, got) in enumerate(zip(solo, outs)):
        for j, (w, g) in enumerate(zip(want, got)):
            assert _same_bits(w, g), f"launch {i} ({calls[i][0]}, n={calls[i][1]}): output {j} differs from its solo run"
    assert _counts(st) == _counts(st_solo)
