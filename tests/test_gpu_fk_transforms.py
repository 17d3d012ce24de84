"""Batched cumulative DH transforms (ForwardKinematics.fkine_batch / joint_positions / fkine_device, csrc/fk.cu).

The batched kernel is also the single-pose path (ikb_fk_chain_host is the kernel at n = 1), so a row's bits must not
depend on the batch, the chunking, the entry point or the output layout it comes out of."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TWISTED_DH = [[0, np.pi / 2, 0, 0], [2, 0.5, -0.25, 0.1], [0.3, 2, 1.5, 2.5], [np.pi / 2, 0.3, -0.2, 0.1]]
MSG = "Forward Kinematics exception, robot joints angles limits are (-2pi, 2pi)"


def _robot():
    from inversekinematicsann_b200.robot.robot import SixDOFRobot
    return SixDOFRobot


def _fk(dh=None):
    from inversekinematicsann_b200.kinematics.forward import ForwardKinematics
    return ForwardKinematics(_robot().dh_matrix if dh is None else dh)


def _angles(n, seed, dtype=np.float64):
    return np.random.default_rng(seed).uniform(-np.pi, np.pi, size=(n, 4)).astype(dtype)


def _chunk_rows(slot_rows, out_row_bytes):
    # capi.cu: a host chunk holds as many rows as the 32 bytes per slot row of the output staging buffer
    return slot_rows * 32 // out_row_bytes


def _slot_rows(n):
    # capi.cu ensure_slots: the next power of two >= n, at least 1024, at most 4 Mi
    want = 1024
    while want < n and want < 1 << 22:
        want <<= 1
    return want


# ---- 1. matrices, fp64 ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", ["robot", "twisted"])
def test_matrices_match_oracle_and_single_pose_bits(table):
    from oracle import c_oracle
    dh = None if table == "robot" else TWISTED_DH
    dh_arr = np.array(_robot().dh_matrix if dh is None else dh, dtype=np.float64)
    fk = _fk(dh)
    ang = _angles(20_000, 1 if table == "robot" else 2)
    T, chain = fk.fkine_batch(ang)
    assert chain.shape == (20_000, 4, 4, 4) and chain.dtype == np.float64
    for i in range(ang.shape[0]):
        st, want = c_oracle.fk_chain(ang[i], dh=dh_arr)
        assert st == 0
        assert np.abs(chain[i] - want).max() <= 1e-12, i
    for i in range(2_000):  # the single-pose path is the same kernel at n = 1
        t4, mats = fk.fkine(list(ang[i]))
        assert np.array_equal(np.array(mats), chain[i]) and np.array_equal(t4, T[i]), i
    assert np.shares_memory(T, chain) and np.array_equal(T, chain[:, 3])
    assert np.array_equal(chain[:, :, 3, :], np.broadcast_to([0.0, 0.0, 0.0, 1.0], (20_000, 4, 4)))
    assert not np.signbit(chain[:, :, 3, :]).any()


# ---- 2. joints layout ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_joints_are_column_three_of_the_matrices(dtype):
    fk = _fk()
    ang = _angles(20_011, 3, dtype)
    _, chain = fk.fkine_batch(ang)
    joints = fk.joint_positions(ang)
    assert joints.shape == (20_011, 4, 3) and joints.dtype == dtype
    assert np.array_equal(joints, chain[:, :, :3, 3])
    if dtype == np.float64:
        assert np.abs(joints[:, 3] - fk.fkine_positions(ang)).max() <= 1e-12


# ---- 3. float32 ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("what", ["matrices", "joints"])
def test_float32_is_the_fp64_result_rounded_once(what):
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    a32 = _angles(30_000, 4, np.float32)
    got, _ = eng.fk_transforms(a32, what)
    want, _ = eng.fk_transforms(a32.astype(np.float64), what)
    assert got.dtype == np.float32 and np.array_equal(got, want.astype(np.float32))


# ---- 4. batch independence, chunks, entry points, alignment ------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 31, 127, 129, 64 * 37 + 17])
@pytest.mark.parametrize("what", ["matrices", "joints"])
def test_row_permutation(n, what):
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    rng = np.random.default_rng(n)
    ang = _angles(n, n + 5)
    a, sa = eng.fk_transforms(ang, what)
    perm = rng.permutation(n)
    b, _ = eng.fk_transforms(ang[perm], what)
    assert a.shape == ((n, 4, 4, 4) if what == "matrices" else (n, 4, 3))
    assert np.array_equal(b, a[perm]) and sa.first_fk_angle_range == -1
    if n:
        single, _ = eng.fk_transforms(ang[n - 1:], what)
        assert np.array_equal(single[0], a[n - 1])


def test_host_chunks_equal_the_device_path():
    """A fresh engine, so that its staging slots are sized by this call alone: 800 000 fp64 rows give 1 Mi slot rows,
    chunks of 64 Ki rows at 512 B per row -- 13 chunks, one launch each."""
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    n = 800_000
    ang = _angles(n, 6)
    with IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits) as eng:
        for what, row_bytes in (("matrices", 512), ("joints", 96)):
            chunks = -(-n // _chunk_rows(_slot_rows(n), row_bytes))
            assert chunks >= 3
            before = eng.launch_count
            host, st = eng.fk_transforms(ang, what)
            assert eng.launch_count - before == chunks and st.first_fk_angle_range == -1
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                d_ang = torch.from_numpy(ang).cuda()
                out = torch.empty(host.shape, dtype=torch.float64, device="cuda")
                eng.fk_transforms_device(d_ang, out, what)
            s.synchronize()
            assert np.array_equal(out.cpu().numpy(), host), what


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("what", ["matrices", "joints"])
def test_unaligned_output_view(dtype, what):
    """An output that starts one element into its storage (4 or 8 bytes: not 16-byte aligned) takes the element-store
    path and gets the same bits; the elements around it are untouched."""
    import torch
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    td = getattr(torch, dtype)
    n = 64 * 5 + 3
    ang = torch.from_numpy(_angles(n, 7, np.dtype(dtype))).cuda()
    tail = (4, 4, 4) if what == "matrices" else (4, 3)
    width = int(np.prod(tail))
    aligned = torch.empty((n,) + tail, dtype=td, device="cuda")
    eng.fk_transforms_device(ang, aligned, what)
    base = torch.full((n * width + 2,), -7.0, dtype=td, device="cuda")
    view = base[1:1 + n * width].view((n,) + tail)
    assert view.data_ptr() % 16 != 0
    eng.fk_transforms_device(ang, view, what)
    torch.cuda.synchronize()
    assert torch.equal(view, aligned)
    assert base[0].item() == -7.0 and base[-1].item() == -7.0


# ---- 5. angle guard ------------------------------------------------------------------------------------------------
def test_guard_lowest_row_across_host_chunks():
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.robot.robot import OutOfRobotReachException
    R = _robot()
    n = 300_000  # 512 Ki slot rows: chunks of 32 Ki fp64 matrix rows
    chunk = _chunk_rows(_slot_rows(n), 512)
    ang = _angles(n, 8)
    with IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits) as eng:
        clean, _ = eng.fk_transforms(ang)
        ang[2 * chunk + 5, 1] = -6.5       # after the second chunk boundary
        ang[2 * chunk - 3, 3] = 7.0        # before it: the lowest
        ang[7 * chunk + 1, 0] = np.inf
        for what in ("matrices", "joints"):
            out, st = eng.fk_transforms(ang, what)
            assert st.first_fk_angle_range == 2 * chunk - 3, what
        out, _ = eng.fk_transforms(ang)
        keep = np.ones(n, dtype=bool)
        keep[[2 * chunk - 3, 2 * chunk + 5, 7 * chunk + 1]] = False
        assert np.array_equal(out[keep], clean[keep])   # offending rows are written, the others unchanged
        assert np.isfinite(out[2 * chunk - 3]).all()
    fk = _fk()
    with pytest.raises(OutOfRobotReachException) as exc:
        fk.fkine_batch(ang[: 2 * chunk])
    assert str(exc.value) == MSG
    with pytest.raises(OutOfRobotReachException) as exc:
        fk.joint_positions(np.array([[0.1, 0.2, 0.3, 0.4], [0.0, 0.0, 6.3, 0.0]]))
    assert str(exc.value) == MSG


def test_guard_bounds_inclusive_and_nan_passes():
    from inversekinematicsann_b200.kinematics._shared import get_engine
    fk = _fk()
    edge = np.array([[2 * np.pi, -2 * np.pi, 0.0, 0.0], [0.0, 0.0, -2 * np.pi, 2 * np.pi],
                     [np.nan, 0.1, 0.2, 0.3], [0.1, 0.2, 0.3, np.nan]])
    T, chain = fk.fkine_batch(edge)
    assert np.isfinite(chain[:2]).all() and np.isnan(chain[2]).any() and np.isnan(chain[3]).any()
    _, st = get_engine().fk_transforms(np.nextafter(edge[:1], np.inf))  # just above 2 pi
    assert st.first_fk_angle_range == 0
    # float32 angles are widened exactly before the test: float32(2 pi) = 6.2831855 lies above 2 pi, the float32
    # just below it passes
    inside = np.nextafter(np.float32(2 * np.pi), np.float32(0))
    fk.joint_positions(np.array([[inside, -inside, 0, 0], [np.nan, 0, 0, 0]], dtype=np.float32))
    _, st = get_engine().fk_transforms(edge.astype(np.float32))
    assert st.first_fk_angle_range == 0


def test_device_guard_accumulates_in_the_statistics():
    import torch
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    fk = _fk()
    ang = torch.from_numpy(_angles(10_000, 9)).cuda()
    eng.stats_reset_torch()
    fk.fkine_device(ang)
    assert eng.stats_fetch_torch().first_fk_angle_range == -1
    bad = ang.clone()
    bad[6_001, 2] = 6.4
    bad[9_999, 0] = -6.4
    fk.fkine_device(bad[6_000:], what="joints")   # row 1 of this call
    fk.fkine_device(bad)                          # row 6 001 of this one: the block keeps the lowest, 1
    assert eng.stats_fetch_torch().first_fk_angle_range == 1
    eng.stats_reset_torch()


def test_seed_chain_leaves_the_statistics_clean():
    """The engine's seed chain runs through the same kernel at creation; a seed pose outside [-2pi, 2pi] must not show
    up in the first call's statistics."""
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    dh = np.array(R.dh_matrix, dtype=np.float64)
    dh[0, 2] = 7.0
    with IkEngine(dh, R.links_lengths, R.effector_workspace_limits) as eng:
        assert eng.stats_fetch().first_fk_angle_range == -1
        _, status = eng.fk_chain([0.0, 7.0, 0.0, 0.0])
        assert status == 1
        _, status = eng.fk_chain([0.0, 2 * np.pi, 0.0, np.nan])
        assert status == 0


# ---- 6. composition with Fabrik ------------------------------------------------------------------------------------
def test_joint_positions_feed_fabrik_on_the_device():
    import torch
    from inversekinematicsann_b200.kinematics.fabrik import Fabrik
    from inversekinematicsann_b200.kinematics.inverse import FabrikInverseKinematics
    R = _robot()
    rng = np.random.default_rng(10)
    pts = rng.uniform([0, -6, -3], [6, 6, 6], size=(5_000, 3))
    ik = FabrikInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    angles = ik.ikine(pts, as_array=True)
    ok = np.isfinite(angles).all(axis=1)
    angles, pts = angles[ok], pts[ok]
    fk = _fk()
    goals = pts[::-1].copy()
    d_joints = fk.fkine_device(torch.from_numpy(angles).cuda(), what="joints")
    assert d_joints.shape == (angles.shape[0], 4, 3) and d_joints.dtype == torch.float64
    f = Fabrik(R.links_lengths)
    dev = f.calculate_device(d_joints, torch.from_numpy(goals).cuda())
    host, _ = f.calculate_batch(fk.joint_positions(angles), goals)
    assert np.array_equal(dev.cpu().numpy(), host)


# ---- 7. rejection --------------------------------------------------------------------------------------------------
def test_arguments_rejected_before_launch():
    import torch
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.kinematics._shared import get_engine
    eng = get_engine()
    n = 8
    ang = torch.zeros(n, 4, dtype=torch.float64, device="cuda")
    out = torch.empty(n, 4, 4, 4, dtype=torch.float64, device="cuda")
    before = eng.launch_count
    bad_device = [
        (TypeError, ang.cpu(), out, "matrices"),
        (TypeError, ang, out.cpu(), "matrices"),
        (ValueError, ang, out.float(), "matrices"),
        (ValueError, ang, torch.empty(n, 4, 3, dtype=torch.float64, device="cuda"), "matrices"),
        (ValueError, ang, out, "joints"),
        (ValueError, ang, torch.empty(n + 1, 4, 4, 4, dtype=torch.float64, device="cuda"), "matrices"),
        (ValueError, ang, torch.empty(4, 4, 4, n, dtype=torch.float64, device="cuda").permute(3, 0, 1, 2), "matrices"),
        (ValueError, ang, out, "positions"),
        (ValueError, torch.zeros(n, 3, dtype=torch.float64, device="cuda"), out, "matrices"),
        (ValueError, torch.zeros(n, 4, dtype=torch.float64, device="cuda").t().contiguous().t(), out, "matrices"),
    ]
    for exc, a, o, what in bad_device:
        with pytest.raises(exc):
            eng.fk_transforms_device(a, o, what)
    host = np.zeros((n, 4))
    ro = np.empty((n, 4, 4, 4))
    ro.flags.writeable = False
    bad_host = [
        (ValueError, host, ro, "matrices"),
        (TypeError, host, np.empty((n, 4, 4, 4), dtype=np.float32), "matrices"),
        (ValueError, host, np.empty((n, 4, 3)), "matrices"),
        (ValueError, host, np.empty((n, 4, 4, 4))[:, ::-1], "matrices"),
        (ValueError, np.zeros((n, 3)), None, "matrices"),
        (ValueError, host, None, "T"),
        (TypeError, host, torch.empty(n, 4, 4, 4, dtype=torch.float64), "matrices"),
    ]
    for exc, a, o, what in bad_host:
        with pytest.raises(exc):
            eng.fk_transforms(a, what, out=o)
    assert eng.launch_count == before
    lib, h = eng._lib, eng._handle
    p, q = host.ctypes.data, ro.ctypes.data
    for fn, last in ((lib.ikb_fk_transforms_host, None), (lib.ikb_fk_transforms_device, None)):
        assert fn(h, p, _native.IKB_F64, -1, _native.IKB_FK_MATRICES, q, last) == _native.IKB_ERR_INVALID
        assert fn(h, p, _native.IKB_F64, n, 2, q, last) == _native.IKB_ERR_INVALID
        assert fn(h, p, 5, n, _native.IKB_FK_JOINTS, q, last) == _native.IKB_ERR_INVALID
        assert fn(h, None, _native.IKB_F64, n, _native.IKB_FK_JOINTS, q, last) == _native.IKB_ERR_INVALID
        assert fn(h, p, _native.IKB_F64, n, _native.IKB_FK_JOINTS, None, last) == _native.IKB_ERR_INVALID
        assert fn(h, p + 4, _native.IKB_F64, n, _native.IKB_FK_JOINTS, q, last) == _native.IKB_ERR_INVALID
        assert fn(None, p, _native.IKB_F64, n, _native.IKB_FK_JOINTS, q, last) == _native.IKB_ERR_INVALID
        assert fn(h, None, _native.IKB_F64, 0, _native.IKB_FK_JOINTS, None, last) == _native.IKB_OK
    assert eng.launch_count == before
    st = _native.IkbStats()
    assert lib.ikb_fk_transforms_host(h, p, _native.IKB_F64, 0, 0, None, ctypes.byref(st)) == _native.IKB_OK
    assert st.first_fk_angle_range == -1
