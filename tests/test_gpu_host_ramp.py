"""The host pipelines (ikb_*_host) past their ramp, and long enough that stages share work counters.

A host call of more than 4 stages (16 Mi rows) starts with two short stages, 512 Ki and 2 Mi rows, before the 4 Mi
ones (host_chunk_rows in csrc/capi.cu).  Each stage runs on one of three slot streams with its global row offset, and
a call of 18 stages gives stage j and stage j + 16 the same counter of the engine's ring on different streams.  The
outputs must equal the device path's on the same rows, bit for bit, and every row must be counted once."""
import numpy as np
import pytest

STAGE = 1 << 22                               # kHostChunkRows of csrc/capi.cu
RAMP_N = 4 * STAGE + (1 << 20) + 37           # stages of 512 Ki, 2 Mi, 4 Mi, 4 Mi, 4 Mi and 2.5 Mi + 37 rows
LONG_N = (1 << 19) + (1 << 21) + 15 * STAGE + 12_345  # 18 stages
B1, B2 = STAGE // 8, STAGE // 8 + STAGE // 2  # first rows of the second and third stage: 512 Ki and 2.5 Mi


def host_chunk_rows(lo, n):
    """Rows of the pipeline stage that starts at row lo (restated from csrc/capi.cu)."""
    m = STAGE
    if n > 4 * STAGE:
        if lo == 0:
            m = STAGE // 8
        elif lo == STAGE // 8:
            m = STAGE // 2
    return min(m, n - lo)


def stages(n):
    out, lo = [], 0
    while lo < n:
        m = host_chunk_rows(lo, n)
        out.append((lo, m))
        lo += m
    return out


def test_restated_ramp():
    assert [m for _, m in stages(RAMP_N)] == [1 << 19, 1 << 21, STAGE, STAGE, STAGE, (1 << 21) + (1 << 19) + 37]
    assert [lo for lo, _ in stages(RAMP_N)][1:3] == [B1, B2]
    assert len(stages(LONG_N)) == 18 and stages(LONG_N)[-1][1] == 12_345
    assert [m for _, m in stages(4 * STAGE)] == [STAGE] * 4  # no ramp up to 4 stages


def _same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    u = {8: np.uint64, 4: np.uint32}[a.dtype.itemsize]
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(u), b.view(u))


def _box_rows(n, cols, seed):
    """n rows in the workspace box (cols=3, float32) or n angle rows in [-pi, pi) (cols=4, float32), drawn on the GPU."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = torch.rand(n, cols, generator=g, device="cuda")
    if cols == 3:
        return u.mul_(torch.tensor([6.0, 12.0, 9.0], device="cuda")).add_(torch.tensor([0.0, -6.0, -3.0], device="cuda"))
    return u.mul_(2 * np.pi).sub_(np.pi)


@pytest.fixture(scope="module")
def eng():
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    from oracle import np_oracle
    e = IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    W, b = np_oracle.synthetic_mlp(seed=3, dims=np_oracle.LAYER_DIMS)
    e.mlp_load(W, b, np_oracle.SHIPPED_MEAN_X, np_oracle.SHIPPED_SCALE_X, np_oracle.SHIPPED_MEAN_Y,
               np_oracle.SHIPPED_SCALE_Y)
    yield e
    torch.cuda.synchronize()
    e.close()


@pytest.fixture(scope="module")
def ramp_rows():
    """(targets, angles) of RAMP_N rows: float32 on the device and their host copies."""
    xyz = _box_rows(RAMP_N, 3, 41)
    ang = _box_rows(RAMP_N, 4, 42)
    return xyz, xyz.cpu().numpy(), ang, ang.cpu().numpy()


def _device_stats(eng, fn):
    import torch
    torch.cuda.synchronize()
    eng.stats_reset()
    fn()
    torch.cuda.synchronize()
    return eng.stats_fetch()


@pytest.mark.gpu
def test_fabrik_solve_host_ramp(eng, ramp_rows):
    import torch
    xyz, xyz_h, _, _ = ramp_rows
    n = RAMP_N
    l0 = eng.launch_count
    out, st, it, err = eng.fabrik_solve(xyz_h, out_dtype=np.float32, return_iters=True, return_fk_error=True)
    assert eng.launch_count - l0 == 2 * len(stages(n))  # K1, then K3 for the errors, per stage
    out_d = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    it_d = torch.empty(n, dtype=torch.int32, device="cuda")
    err_d = torch.empty(n, dtype=torch.float32, device="cuda")
    st_d = _device_stats(eng, lambda: eng.fabrik_solve_device(xyz, out_d, iters=it_d, fk_err=err_d))
    assert _same_bits(out, out_d.cpu().numpy())
    assert np.array_equal(it, it_d.cpu().numpy())
    assert _same_bits(err, err_d.cpu().numpy())
    assert st.n_solved == st_d.n_solved == n
    assert st.sum_iterations == st_d.sum_iterations == int(it.sum(dtype=np.int64))
    assert st.n_iter_capped == st_d.n_iter_capped and st.first_out_of_limits == -1


@pytest.mark.gpu
def test_check_limits_host_ramp(eng, ramp_rows):
    xyz, xyz_h, _, _ = ramp_rows
    l0 = eng.launch_count
    assert eng.check_limits(xyz_h) == -1
    assert eng.launch_count - l0 == len(stages(RAMP_N))
    assert _device_stats(eng, lambda: eng.check_limits_device(xyz)).first_out_of_limits == -1


@pytest.mark.gpu
def test_fk_host_ramp(eng, ramp_rows):
    import torch
    xyz, xyz_h, ang, ang_h = ramp_rows
    n = RAMP_N
    l0 = eng.launch_count
    pos, err, st = eng.fk(ang_h, targets=xyz_h, want_pos=True, want_err=True)
    assert eng.launch_count - l0 == len(stages(n))
    pos_d = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    err_d = torch.empty(n, dtype=torch.float32, device="cuda")
    st_d = _device_stats(eng, lambda: eng.fk_device(ang, targets=xyz, pos=pos_d, err=err_d))
    assert _same_bits(pos, pos_d.cpu().numpy()) and _same_bits(err, err_d.cpu().numpy())
    assert st.n_fk_error == st_d.n_fk_error == n and st.first_fk_angle_range == -1


@pytest.mark.gpu
def test_ann_solve_host_ramp(eng, ramp_rows):
    import torch
    xyz, xyz_h, _, _ = ramp_rows
    n = RAMP_N
    l0 = eng.launch_count
    out, st, err = eng.ann_solve(xyz_h, mode="fp16x3_ts", return_fk_error=True)
    assert eng.launch_count - l0 == len(stages(n))  # the FK error is part of the network kernel's output stage
    out_d = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    err_d = torch.empty(n, dtype=torch.float32, device="cuda")
    _device_stats(eng, lambda: eng.ann_solve_device(xyz, out_d, mode="fp16x3_ts", fk_err=err_d))
    assert _same_bits(out, out_d.cpu().numpy()) and _same_bits(err, err_d.cpu().numpy())
    assert st.first_out_of_limits == -1


# offenders just before and after the ramp's stage boundaries; the lowest is the first row of a later stage, so only a
# stage that reports its global row offset names it
OFFENDERS = {"after_512Ki": [B1, B1 + 1, B2 - 1, B2], "after_2.5Mi": [B2, B2 + 2, B2 + STAGE - 1, B2 + STAGE + 1]}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(OFFENDERS))
def test_first_offender_is_a_global_row(eng, ramp_rows, case):
    _, xyz_h, _, ang_h = ramp_rows
    rows = OFFENDERS[case]
    xyz = xyz_h.copy()
    xyz[rows, 0] = -1.0  # x < 0: outside the workspace box
    assert eng.check_limits(xyz) == rows[0]
    _, st = eng.fabrik_solve(xyz, out_dtype=np.float32)
    assert st.first_out_of_limits == rows[0]
    ang = ang_h.copy()
    ang[rows, 1] = 7.0  # > 2 pi
    _, _, st = eng.fk(ang)
    assert st.first_fk_angle_range == rows[0]


@pytest.mark.gpu
def test_fabrik_solve_host_18_stages(eng):
    """Stages j and j + 16 take the same counter of the ring and run on different slot streams.  Needs ~2 GB of host
    memory for the float32 targets and angles."""
    import torch
    n = LONG_N
    xyz = _box_rows(n, 3, 43)
    l0 = eng.launch_count
    out, st, it = eng.fabrik_solve(xyz.cpu().numpy(), out_dtype=np.float32, return_iters=True)
    assert eng.launch_count - l0 == len(stages(n)) == 18
    out_d = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    it_d = torch.empty(n, dtype=torch.int32, device="cuda")
    st_d = _device_stats(eng, lambda: eng.fabrik_solve_device(xyz, out_d, iters=it_d))
    for lo, m in stages(n):
        assert _same_bits(out[lo:lo + m], out_d[lo:lo + m].cpu().numpy()), f"stage at row {lo}"
        assert np.array_equal(it[lo:lo + m], it_d[lo:lo + m].cpu().numpy()), f"stage at row {lo}"
    assert st.n_solved == st_d.n_solved == n
    assert st.sum_iterations == st_d.sum_iterations == int(it.sum(dtype=np.int64))
