"""Every device entry point writes exactly rows [0, n) of each output it is given: nothing before, nothing after, nothing
left unwritten.

The kernels work in units larger than a row -- 128-row ANN tiles, K3's row pairs and 64-row ring trips with an odd-row
tail, K1's parked and refilled rows, 64-row fk_transforms tiles -- and the host entry points go through staging
buffers, where a stray write would land in unused memory.  Here each output is the middle of a larger buffer filled
with a NaN bit pattern no kernel computes; after the call the bands on either side must hold that pattern bit for bit
and no element of the output may still hold it.  Outputs start 4, 8 and 12 bytes past 16-byte alignment wherever the
entry point accepts such a start; entry points that store rows as 16-byte vectors refuse them."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PAT32 = 0x7FBADBAD               # a NaN payload no arithmetic produces (hardware NaNs are 0x7FFFFFFF / 0x7FC00000)
PAT64 = 0x7FF4DEADBEEFBAD1
BAND = 1024                       # guard bytes on each side
N_SMALL = [1, 2, 3, 63, 64, 65, 127, 128, 129]


def _n_big():
    """Large enough for K3's ring (4 CTAs x 8 warps x 64 rows per SM) with a ragged tail, and for 16 ANN tiles per
    persistent CTA."""
    import torch
    return 4 * torch.cuda.get_device_properties(0).multi_processor_count * 8 * 64 + 37


class Guarded:
    """A `shape` tensor of `dtype` placed `offset` bytes past a 16-byte boundary inside a pattern-filled buffer."""

    def __init__(self, shape, dtype, offset=0):
        import torch
        isz = torch.empty((), dtype=dtype).element_size()
        assert offset % isz == 0
        self.count = int(np.prod(shape))
        self.start = (BAND + offset) // isz
        self.end = self.start + self.count
        self.pat = PAT32 if isz == 4 else PAT64
        itype = torch.int32 if isz == 4 else torch.int64
        self.raw = torch.full((self.end + BAND // isz,), self.pat, dtype=itype, device="cuda")
        assert self.raw.data_ptr() % 256 == 0
        self.t = self.raw[self.start:self.end].view(dtype).view(shape)
        assert self.t.data_ptr() % 16 == offset

    def check(self, tag, written=True):
        import torch
        torch.cuda.synchronize()
        r = self.raw
        assert bool((r[:self.start] == self.pat).all()), f"{tag}: write before the output"
        assert bool((r[self.end:] == self.pat).all()), f"{tag}: write past the output"
        inside = r[self.start:self.end] == self.pat
        if written:
            assert not bool(inside.any()), f"{tag}: {int(inside.sum())} elements left unwritten"
        else:
            assert bool(inside.all()), f"{tag}: written although the call was refused"


def _offsets(isz):
    return [o for o in (0, 4, 8, 12) if o % isz == 0]


def _cases(isz):
    """(n, offset) pairs: every small n at every offset, the large n aligned and at one misaligned start."""
    return [(n, o) for n in N_SMALL for o in _offsets(isz)] + [(_n_big(), 0), (_n_big(), _offsets(isz)[-1])]


def _points(n, dtype, seed=0):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    lo = torch.tensor([0.0, -6.0, -3.0], device="cuda", dtype=torch.float64)
    span = torch.tensor([6.0, 12.0, 9.0], device="cuda", dtype=torch.float64)
    return (torch.rand(n, 3, device="cuda", generator=g, dtype=torch.float64) * span + lo).to(dtype)


@pytest.fixture(scope="module")
def eng():
    from inversekinematicsann_b200.kinematics._shared import get_engine
    return get_engine()


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_fabrik_solve_device_bounds(eng, dtype):
    import torch
    dt = getattr(torch, dtype)
    isz = 4 if dtype == "float32" else 8
    for n, off in _cases(isz):
        xyz = _points(n, dt, seed=n)
        out = Guarded((n, 4), dt, 0)
        it = Guarded((n,), torch.int32, _offsets(4)[(n + 1) % 4])
        err = Guarded((n,), dt, off)
        eng.fabrik_solve_device(xyz, out.t, iters=it.t, fk_err=err.t)
        for g, what in ((out, "out"), (it, "iters"), (err, "fk_err")):
            g.check(f"fabrik {dtype} n={n} off={off} {what}")


@pytest.mark.parametrize("mode", ["fp16x3_ts", "fp16x3", "fp32"])
def test_ann_solve_device_bounds(mode):
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    from oracle import np_oracle
    W, b = np_oracle.synthetic_mlp(seed=12, dims=[3, 200, 200, 4])
    eng = IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    try:
        eng.mlp_load(W, b, np_oracle.SHIPPED_MEAN_X, np_oracle.SHIPPED_SCALE_X, np_oracle.SHIPPED_MEAN_Y,
                     np_oracle.SHIPPED_SCALE_Y)
        for n, off in _cases(4):
            xyz = _points(n, torch.float32, seed=n)
            out = Guarded((n, 4), torch.float32, 0)
            err = Guarded((n,), torch.float32, off)
            eng.ann_solve_device(xyz, out.t, mode=mode, fk_err=err.t)
            out.check(f"ann {mode} n={n} out")
            err.check(f"ann {mode} n={n} off={off} fk_err")
            only = Guarded((n, 4), torch.float32, 0)
            eng.ann_solve_device(xyz, only.t, mode=mode)
            only.check(f"ann {mode} n={n} out without fk_err")
            assert torch.equal(only.t, out.t)
    finally:
        eng.close()


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_fk_device_bounds(eng, dtype):
    """Error only (fp32: the ring, the pair kernel, or -- 4 / 12 bytes off -- the generic kernel) and positions with
    error (the generic kernel)."""
    import torch
    dt = getattr(torch, dtype)
    isz = 4 if dtype == "float32" else 8
    for n, off in _cases(isz):
        g = torch.Generator(device="cuda").manual_seed(n)
        ang = (torch.rand(n, 4, device="cuda", generator=g, dtype=torch.float64) * 12 - 6).to(dt)
        tgt = _points(n, dt, seed=n)
        err = Guarded((n,), dt, off)
        eng.fk_device(ang, targets=tgt, err=err.t)
        err.check(f"fk {dtype} n={n} off={off} err only")
        pos = Guarded((n, 3), dt, off)
        err2 = Guarded((n,), dt, _offsets(isz)[0])
        eng.fk_device(ang, targets=tgt, pos=pos.t, err=err2.t)
        pos.check(f"fk {dtype} n={n} off={off} pos")
        err2.check(f"fk {dtype} n={n} err with pos")
        pos_only = Guarded((n, 3), dt, off)
        eng.fk_device(ang, pos=pos_only.t)
        pos_only.check(f"fk {dtype} n={n} off={off} pos only")
        assert torch.equal(pos_only.t, pos.t)


@pytest.mark.parametrize("what", ["matrices", "joints"])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_fk_transforms_device_bounds(eng, dtype, what):
    import torch
    dt = getattr(torch, dtype)
    isz = 4 if dtype == "float32" else 8
    tail = (4, 4, 4) if what == "matrices" else (4, 3)
    for n, off in _cases(isz):
        g = torch.Generator(device="cuda").manual_seed(n)
        ang = (torch.rand(n, 4, device="cuda", generator=g, dtype=torch.float64) * 12 - 6).to(dt)
        out = Guarded((n,) + tail, dt, off)
        eng.fk_transforms_device(ang, out.t, what=what)
        out.check(f"fk_transforms {dtype} {what} n={n} off={off}")


@pytest.mark.parametrize("J", [4, 7])
def test_fabrik_chain_device_bounds(eng, J):
    import torch
    links = np.full(J, 1.5)
    init = torch.zeros(J, 3, dtype=torch.float64, device="cuda")
    init[:, 2] = torch.arange(1, J + 1, dtype=torch.float64, device="cuda") * 1.5
    for n, off in _cases(8):
        goals = _points(n, torch.float64, seed=n)
        out = Guarded((n, J, 3), torch.float64, off)
        it = Guarded((n,), torch.int32, _offsets(4)[n % 4])
        eng.fabrik_chain_device(links, 1e-3, 50, init, goals, out.t, iters=it.t)
        out.check(f"chain J={J} n={n} off={off} out")
        it.check(f"chain J={J} n={n} iters")


def _generate_into(eng, kind, params, n, out, seed=7, row_offset=0):
    import torch
    from inversekinematicsann_b200 import _native
    p = (ctypes.c_double * len(params))(*[float(v) for v in params])
    code = _native.IKB_F32 if out.dtype == torch.float32 else _native.IKB_F64
    stream = ctypes.c_void_p(torch.cuda.current_stream(eng.device).cuda_stream)
    eng._check(eng._lib.ikb_generate_device(eng._handle, kind, p, len(params), int(n), int(row_offset), out.data_ptr(),
                                            code, ctypes.c_uint64(seed), stream), "ikb_generate_device")


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_generator_device_bounds(eng, dtype):
    """The kernel behind every TrainingDataGenerator.*_device shape, writing into a guarded buffer; the rows must be the
    ones the public function returns."""
    import torch
    from inversekinematicsann_b200.robot import position_generator as pg
    dt = getattr(torch, dtype)
    isz = 4 if dtype == "float32" else 8
    kinds = {pg.GEN_CIRCLE: [2.0, 1.0, 0.5, -0.5], pg.GEN_CUBE: [0.5, 2.5, 3.5, 4.0, 0.0, -1.0, 1.0, 5, 7],
             pg.GEN_CUBE_RANDOM: [6, 12, 9, 0, -6, -3], pg.GEN_NORMAL: [0, 6, -6, 6, -3, 6, 0.5]}
    for n, off in _cases(isz):
        for kind, params in list(kinds.items()) + [(pg.GEN_SPRING, [1.0, 2.0, 3.0, n])]:
            out = Guarded((n, 3), dt, off)
            _generate_into(eng, kind, params, n, out.t)
            out.check(f"generator {kind} {dtype} n={n} off={off}")
            want = pg._generate(kind, params, n, dtype=dtype, seed=7)
            assert torch.equal(out.t, want), (kind, n)


def test_vector_row_outputs_refuse_misaligned_starts(eng):
    """ANN and FABRIK angles are stored, and K3 angles loaded, as 16-byte vectors per row: a start 4, 8 or 12 bytes
    off is refused before anything is launched, and the buffer stays untouched."""
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    from oracle import np_oracle
    n = 65
    xyz = _points(n, torch.float32)
    ann = IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    try:
        W, b = np_oracle.synthetic_mlp(seed=1, dims=[3, 64, 4])
        ann.mlp_load(W, b, np_oracle.SHIPPED_MEAN_X, np_oracle.SHIPPED_SCALE_X, np_oracle.SHIPPED_MEAN_Y,
                     np_oracle.SHIPPED_SCALE_Y)
        for off in (4, 8, 12):
            out = Guarded((n, 4), torch.float32, off)
            with pytest.raises(ValueError, match="16-byte aligned"):
                ann.ann_solve_device(xyz, out.t)
            out.check(f"ann off={off}", written=False)
    finally:
        ann.close()
    for dtype, offs in (("float32", (4, 8, 12)), ("float64", (8,))):
        dt = getattr(torch, dtype)
        for off in offs:
            out = Guarded((n, 4), dt, off)
            with pytest.raises(ValueError, match="16-byte aligned"):
                eng.fabrik_solve_device(xyz, out.t)
            out.check(f"fabrik {dtype} off={off}", written=False)
            ang = Guarded((n, 4), dt, off)
            ang.t.zero_()
            with pytest.raises(ValueError, match="16-byte aligned"):
                eng.fk_device(ang.t, targets=xyz.to(dt), err=torch.empty(n, dtype=dt, device="cuda"))
