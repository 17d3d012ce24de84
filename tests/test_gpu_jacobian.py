"""Batched arm Jacobians and manipulability (ForwardKinematics.jacobian / jacobian_batch / manipulability /
jacobian_device, the Jacobian kinds of fk_transforms_kernel in csrc/fk.cu).

The kernel builds on fkine_batch's chain, so its axes are fkine_batch's bits, and its linear rows and w are the bits of
a NumPy restatement in the operation order include/ikb200.h states.  Independent checks: central differences of the C
oracle's FK and, for the robot's own table, the closed form of its planar tail."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TWISTED_DH = [[0, np.pi / 2, 0, 0], [2, 0.5, -0.25, 0.1], [0.3, 2, 1.5, 2.5], [np.pi / 2, 0.3, -0.2, 0.1]]
MSG = "Forward Kinematics exception, robot joints angles limits are (-2pi, 2pi)"
TABLES = ["robot", "twisted"]
SUBSETS = ((0, 1, 2), (0, 1, 3), (0, 2, 3), (1, 2, 3))


def _robot():
    from inversekinematicsann_b200.robot.robot import SixDOFRobot
    return SixDOFRobot


def _dh(table):
    return _robot().dh_matrix if table == "robot" else TWISTED_DH


def _fk(table="robot"):
    from inversekinematicsann_b200.kinematics.forward import ForwardKinematics
    return ForwardKinematics(_dh(table))


def _eng(table="robot"):
    from inversekinematicsann_b200.kinematics._shared import get_engine
    return get_engine(dh_matrix=_dh(table))


def _angles(n, seed, dtype=np.float64):
    return np.random.default_rng(seed).uniform(-np.pi, np.pi, size=(n, 4)).astype(dtype)


def _slot_rows(n):
    # capi.cu ensure_slots: the next power of two >= n, at least 1024, at most 4 Mi
    want = 1024
    while want < n and want < 1 << 22:
        want <<= 1
    return want


def _chunk_rows(slot_rows, jac_row_bytes):
    # capi.cu ikb_jacobian_host: min(S, 32 S / B), S rows without a Jacobian output
    return slot_rows if jac_row_bytes is None else min(slot_rows, slot_rows * 32 // jac_row_bytes)


def _same_bits(a, b):
    """Equal bit for bit, except that any NaN equals any NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    nan = np.isnan(a)
    u = np.uint64 if a.dtype == np.float64 else np.uint32
    return bool(np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(u), b[~nan].view(u)))


# ---- the NumPy restatement (operation order of include/ikb200.h) -------------------------------------------------
def np_linear(chain):
    """Linear rows (n, 3, 4) from fkine_batch's matrices (n, 4, 4, 4): z_{i-1} x (p_4 - p_{i-1})."""
    n = chain.shape[0]
    z = np.empty((n, 4, 3))
    p = np.empty((n, 5, 3))
    z[:, 0] = (0.0, 0.0, 1.0)
    z[:, 1:] = chain[:, :3, :3, 2]
    p[:, 0] = 0.0
    p[:, 1:] = chain[:, :, :3, 3]
    d = p[:, 4:5] - p[:, :4]
    lin = np.empty((n, 3, 4))
    lin[:, 0] = z[..., 1] * d[..., 2] - z[..., 2] * d[..., 1]
    lin[:, 1] = z[..., 2] * d[..., 0] - z[..., 0] * d[..., 2]
    lin[:, 2] = z[..., 0] * d[..., 1] - z[..., 1] * d[..., 0]
    return lin


def np_geometric(chain):
    jac = np.empty((chain.shape[0], 6, 4))
    jac[:, :3] = np_linear(chain)
    jac[:, 3:, 0] = (0.0, 0.0, 1.0)
    jac[:, 3:, 1:] = np.transpose(chain[:, :3, :3, 2], (0, 2, 1))
    return jac


def np_manip(lin):
    s = []
    for a, b, c in SUBSETS:
        A, B, C = lin[:, :, a], lin[:, :, b], lin[:, :, c]
        m0 = B[:, 1] * C[:, 2] - B[:, 2] * C[:, 1]
        m1 = B[:, 2] * C[:, 0] - B[:, 0] * C[:, 2]
        m2 = B[:, 0] * C[:, 1] - B[:, 1] * C[:, 0]
        det = (A[:, 0] * m0 + A[:, 1] * m1) + A[:, 2] * m2
        s.append(det * det)
    return np.sqrt((s[0] + s[1]) + (s[2] + s[3]))


# ---- 1. bits against FK ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", TABLES)
def test_bits_against_fkine_batch(table):
    fk = _fk(table)
    ang = _angles(20_000, 11 if table == "robot" else 12)
    _, chain = fk.fkine_batch(ang)
    jac = fk.jacobian_batch(ang)
    assert jac.shape == (20_000, 6, 4) and jac.dtype == np.float64
    assert np.array_equal(jac[:, 3:, 0], np.broadcast_to([0.0, 0.0, 1.0], (20_000, 3)))
    assert not np.signbit(jac[:, 3:, 0]).any()
    for i in range(2, 5):
        assert _same_bits(np.ascontiguousarray(jac[:, 3:, i - 1]), np.ascontiguousarray(chain[:, i - 2, :3, 2]))
    assert _same_bits(jac[:, :3], np_linear(chain))
    assert _same_bits(jac, np_geometric(chain))
    _, w, st = _eng(table).jacobian(ang, "geometric", manipulability=True)
    assert st.first_fk_angle_range == -1
    assert _same_bits(w, np_manip(np_linear(chain)))


# ---- 2. independent oracle ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", TABLES)
def test_central_differences_of_the_c_oracle(table):
    from oracle import c_oracle
    dh = np.array(_dh(table), dtype=np.float64)
    ang = _angles(400, 21 if table == "robot" else 22, np.float64) * 0.9
    jac = _fk(table).jacobian_batch(ang)
    h = 1e-6
    worst_lin = worst_z = 0.0
    for n_row in range(ang.shape[0]):
        st, mats = c_oracle.fk_chain(ang[n_row], dh=dh)
        assert st == 0
        z = np.vstack([[0.0, 0.0, 1.0], mats[:3, :3, 2]])
        worst_z = max(worst_z, np.abs(jac[n_row, 3:].T - z).max())
        for k in range(4):
            a, b = ang[n_row].copy(), ang[n_row].copy()
            a[k] += h
            b[k] -= h
            pa = c_oracle.fk_chain(a, dh=dh)[1][3, :3, 3]
            pb = c_oracle.fk_chain(b, dh=dh)[1][3, :3, 3]
            worst_lin = max(worst_lin, np.abs((pa - pb) / (2 * h) - jac[n_row, :3, k]).max())
    assert worst_lin <= 1e-7, worst_lin
    assert worst_z <= 1e-12, worst_z


# ---- 3. closed form of the robot's table -------------------------------------------------------------------------
def _closed_form(ang):
    t1 = ang[:, 0]
    phi = np.cumsum(ang[:, 1:], axis=1)                        # phi_2, phi_3, phi_4
    rk = 2 * np.cumsum(np.cos(phi)[:, ::-1], axis=1)[:, ::-1]  # r_k = 2 sum_{j >= k} cos phi_j, k = 2..4
    hk = 2 * np.cumsum(np.sin(phi)[:, ::-1], axis=1)[:, ::-1]
    r = rk[:, 0]
    lin = np.empty((ang.shape[0], 3, 4))
    lin[:, :, 0] = r[:, None] * np.stack([-np.sin(t1), np.cos(t1), np.zeros_like(t1)], axis=1)
    for k in range(3):
        lin[:, :, k + 1] = np.stack([-hk[:, k] * np.cos(t1), -hk[:, k] * np.sin(t1), rk[:, k]], axis=1)
    pairs = sum((hk[:, k] * rk[:, l] - hk[:, l] * rk[:, k]) ** 2 for k in range(3) for l in range(k + 1, 3))
    return lin, np.abs(r) * np.sqrt(pairs)


def test_closed_form_on_the_robot_table():
    eng = _eng()
    ang = _angles(20_000, 31)
    jac, w, _ = eng.jacobian(ang, "position", manipulability=True)
    lin, w_cf = _closed_form(ang)
    assert np.abs(jac - lin).max() <= 1e-12
    assert np.abs(w - w_cf).max() <= 1e-12 * max(1.0, np.abs(w_cf).max())
    assert (w > 0).all()
    stretched = ang.copy()
    stretched[:, 2:] = 0.0
    seed = np.array([[0.0, np.pi / 2, 0.0, 0.0]])
    _, w0, _ = eng.jacobian(np.vstack([seed, stretched]), None, manipulability=True)
    assert (w0 >= 0).all() and w0.max() <= 1e-12, w0.max()


# ---- 4. layouts agree ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", TABLES)
def test_layouts_and_float32_agree(table):
    eng = _eng(table)
    ang = _angles(30_011, 41)
    geo, w_geo, _ = eng.jacobian(ang, "geometric", manipulability=True)
    pos, w_pos, _ = eng.jacobian(ang, "position", manipulability=True)
    none, w_only, _ = eng.jacobian(ang, None, manipulability=True)
    geo_plain, no_w, _ = eng.jacobian(ang)
    assert none is None and no_w is None
    assert _same_bits(pos, np.ascontiguousarray(geo[:, :3])) and _same_bits(geo_plain, geo)
    assert _same_bits(w_only, w_geo) and _same_bits(w_only, w_pos)
    a32 = ang.astype(np.float32)
    wide = a32.astype(np.float64)
    for what in ("geometric", "position"):
        j32, w32, _ = eng.jacobian(a32, what, manipulability=True)
        j64, w64, _ = eng.jacobian(wide, what, manipulability=True)
        assert j32.dtype == np.float32 and w32.dtype == np.float32
        assert _same_bits(j32, j64.astype(np.float32)) and _same_bits(w32, w64.astype(np.float32))
    _, w32, _ = eng.jacobian(a32, None, manipulability=True)
    _, w64, _ = eng.jacobian(wide, None, manipulability=True)
    assert _same_bits(w32, w64.astype(np.float32))


# ---- 5. batch independence -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", TABLES)
def test_batch_independence(table):
    fk, eng = _fk(table), _eng(table)
    big = _angles(100_003, 51)
    ref, w_ref, _ = eng.jacobian(big, "geometric", manipulability=True)
    for i in (0, 1, 64, 99_999, 100_002):
        assert _same_bits(fk.jacobian(big[i]), ref[i])
        assert _same_bits(fk.jacobian(list(big[i])), ref[i])
    rng = np.random.default_rng(52)
    for n in (1, 63, 64, 65, 129, 100_003):
        sel = rng.choice(big.shape[0], size=n, replace=False)
        for what in ("geometric", "position", None):
            j, w, _ = eng.jacobian(big[sel], what, manipulability=True)
            assert _same_bits(w, w_ref[sel]), (n, what)
            if what is not None:
                assert _same_bits(j, ref[sel] if what == "geometric" else np.ascontiguousarray(ref[sel, :3])), (n, what)


def test_empty_batch_launches_nothing():
    eng = _eng()
    fk = _fk()
    before = eng.launch_count
    assert fk.jacobian_batch(np.empty((0, 4))).shape == (0, 6, 4)
    assert fk.jacobian_batch(np.empty((0, 4), np.float32), "position").shape == (0, 3, 4)
    assert fk.manipulability(np.empty((0, 4))).shape == (0,)
    import torch
    d = torch.empty((0, 4), dtype=torch.float64, device="cuda")
    assert tuple(fk.jacobian_device(d).shape) == (0, 6, 4)
    assert fk.jacobian_device(d, what=None, manip_out=torch.empty(0, dtype=torch.float64, device="cuda")) is None
    assert eng.launch_count == before


# ---- 6. host and device --------------------------------------------------------------------------------------------
def test_host_chunks_equal_the_device_path():
    """A fresh engine, so that its staging slots are sized by this call alone."""
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    n = 800_000
    ang = _angles(n, 61)
    with IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits) as eng:
        for what, row_bytes in (("geometric", 192), ("position", 96)):
            for manip in (False, True):
                chunks = -(-n // _chunk_rows(_slot_rows(n), row_bytes))
                assert chunks >= 3
                before = eng.launch_count
                host, w, st = eng.jacobian(ang, what, manipulability=manip)
                assert eng.launch_count - before == chunks and st.first_fk_angle_range == -1
                s = torch.cuda.Stream()
                with torch.cuda.stream(s):
                    d_ang = torch.from_numpy(ang).cuda()
                    out = torch.empty(host.shape, dtype=torch.float64, device="cuda")
                    d_w = torch.empty(n, dtype=torch.float64, device="cuda") if manip else None
                    eng.jacobian_device(d_ang, out, what, d_w)
                s.synchronize()
                assert _same_bits(out.cpu().numpy(), host), (what, manip)
                if manip:
                    assert _same_bits(d_w.cpu().numpy(), w)
        # without a Jacobian a chunk holds a whole slot: 4 Mi slot rows at most, so 4 Mi + 5 rows make two chunks
        n2 = (1 << 22) + 5
        ang2 = _angles(n2, 62, np.float32)
        before = eng.launch_count
        _, w2, _ = eng.jacobian(ang2, None, manipulability=True)
        assert eng.launch_count - before == 2
        d_w = torch.empty(n2, dtype=torch.float32, device="cuda")
        eng.jacobian_device(torch.from_numpy(ang2).cuda(), None, "geometric", d_w)
        torch.cuda.synchronize()
        assert _same_bits(d_w.cpu().numpy(), w2)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("what", ["geometric", "position"])
def test_unaligned_outputs(dtype, what):
    """Outputs 4, 8 or 12 bytes off 16-byte alignment (as far as the element size allows) take the element-store path
    and get the same bits; the elements around them are untouched."""
    import torch
    eng = _eng()
    td = getattr(torch, dtype)
    item = np.dtype(dtype).itemsize
    n = 64 * 5 + 3
    ang = torch.from_numpy(_angles(n, 71, np.dtype(dtype))).cuda()
    tail = (6, 4) if what == "geometric" else (3, 4)
    width = int(np.prod(tail))
    ref = torch.empty((n,) + tail, dtype=td, device="cuda")
    ref_w = torch.empty(n, dtype=td, device="cuda")
    eng.jacobian_device(ang, ref, what, ref_w)
    for off_bytes in (4, 8, 12):
        if off_bytes % item:
            continue
        off = off_bytes // item
        base = torch.full((n * width + 2 * off + 8,), -7.0, dtype=td, device="cuda")
        assert base.data_ptr() % 16 == 0
        view = base[off:off + n * width].view((n,) + tail)
        wbase = torch.full((n + 2 * off,), -7.0, dtype=td, device="cuda")
        wview = wbase[off:off + n]
        eng.jacobian_device(ang, view, what, wview)
        torch.cuda.synchronize()
        assert torch.equal(view, ref) and torch.equal(wview, ref_w), off_bytes
        assert (base[:off] == -7.0).all() and (base[off + n * width:] == -7.0).all()
        assert (wbase[:off] == -7.0).all() and (wbase[off + n:] == -7.0).all()


def test_device_outputs_stay_inside_guard_bands():
    import torch
    eng = _eng()
    GUARD = 64
    pattern = {torch.float32: 0x7FC0BEEF, torch.float64: 0x7FF8DEADBEEF0001}
    for td, npd in ((torch.float32, np.float32), (torch.float64, np.float64)):
        ubits = torch.int32 if td == torch.float32 else torch.int64
        for n in list(range(1, 130)):
            ang = torch.from_numpy(_angles(n, 1000 + n, npd)).cuda()
            for what, width in (("geometric", 24), ("position", 12), (None, 0)):
                jb = torch.full((n * width + 2 * GUARD,), pattern[td], dtype=ubits, device="cuda").view(td)
                wb = torch.full((n + 2 * GUARD,), pattern[td], dtype=ubits, device="cuda").view(td)
                jac = jb[GUARD:GUARD + n * width].view((n, width // 4, 4)) if what else None
                eng.jacobian_device(ang, jac, what or "geometric", wb[GUARD:GUARD + n])
                torch.cuda.synchronize()
                jbits, wbits = jb.view(ubits), wb.view(ubits)
                for bits, inner in ((jbits, n * width), (wbits, n)):
                    assert (bits[:GUARD] == pattern[td]).all() and (bits[GUARD + inner:] == pattern[td]).all(), (n, what)
                assert not (wbits[GUARD:GUARD + n] == pattern[td]).any()
                if what:
                    assert not (jbits[GUARD:GUARD + n * width] == pattern[td]).any()


# ---- 7. guard ------------------------------------------------------------------------------------------------------
def _guard_poses():
    two_pi = 2 * np.pi
    rows = [[two_pi, -two_pi, 0.1, 0.2], [0.1, 0.2, -two_pi, two_pi],               # inside
            [np.nextafter(two_pi, 0), 0, 0, np.nextafter(-two_pi, 0)],             # inside
            [np.nan, 0.1, 0.2, 0.3], [0.1, 0.2, 0.3, np.nan],                        # NaN passes
            [np.nextafter(two_pi, 7.0), 0, 0, 0], [0, np.nextafter(-two_pi, -7.0), 0, 0],  # outside
            [0, 0, float(np.float32(two_pi)), 0], [np.inf, 0, 0, 0], [0, 0, 0, -np.inf]]
    bad = [False, False, False, False, False, True, True, True, True, True]
    return np.array(rows), np.array(bad)


@pytest.mark.parametrize("table", TABLES)
def test_guard_rows_written_and_lowest_reported(table):
    from inversekinematicsann_b200.robot.robot import OutOfRobotReachException
    eng = _eng(table)
    fk = _fk(table)
    rows, bad = _guard_poses()
    chain, _ = eng.fk_transforms(rows)
    want = np_geometric(chain)
    jac, w, st = eng.jacobian(rows, "geometric", manipulability=True)
    assert st.first_fk_angle_range == int(np.flatnonzero(bad)[0])
    assert _same_bits(jac, want) and _same_bits(w, np_manip(want[:, :3]))
    assert np.isfinite(jac[:3]).all() and np.isfinite(jac[5:8]).all()
    for i in np.flatnonzero(bad):
        _, _, st = eng.jacobian(rows[i:i + 1], None, manipulability=True)
        assert st.first_fk_angle_range == 0, i
        _, _, st = eng.jacobian(np.vstack([rows[:3], rows[i:i + 1]]), "position")
        assert st.first_fk_angle_range == 3, i
    # float32 angles are tested after widening: float32(2 pi) is outside, the float just below it inside
    inside = np.nextafter(np.float32(2 * np.pi), np.float32(0))
    f32 = np.array([[inside, -inside, 0, 0], [np.nan, 0, 0, 0], [0, np.float32(2 * np.pi), 0, 0]], dtype=np.float32)
    _, _, st = eng.jacobian(f32, "geometric", manipulability=True)
    assert st.first_fk_angle_range == 2
    fk.jacobian_batch(f32[:2])
    fk.manipulability(f32[:2])
    for call in (lambda: fk.jacobian_batch(rows), lambda: fk.jacobian_batch(rows, "position"),
                 lambda: fk.manipulability(rows[5:6]), lambda: fk.jacobian(rows[9]), lambda: fk.jacobian_batch(f32)):
        with pytest.raises(OutOfRobotReachException) as exc:
            call()
        assert str(exc.value) == MSG


def test_guard_lowest_row_across_host_chunks():
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    n = 300_000
    chunk = _chunk_rows(_slot_rows(n), 192)
    ang = _angles(n, 81)
    with IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits) as eng:
        clean, w_clean, _ = eng.jacobian(ang, "geometric", manipulability=True)
        ang[2 * chunk + 5, 1] = -6.5
        ang[2 * chunk - 3, 3] = 7.0        # the lowest, just before a chunk boundary
        ang[3 * chunk + 1, 0] = np.inf
        for what in ("geometric", "position", None):
            _, _, st = eng.jacobian(ang, what, manipulability=True)
            assert st.first_fk_angle_range == 2 * chunk - 3, what
        out, w, _ = eng.jacobian(ang, "geometric", manipulability=True)
        keep = np.ones(n, dtype=bool)
        keep[[2 * chunk - 3, 2 * chunk + 5, 3 * chunk + 1]] = False
        assert _same_bits(out[keep], clean[keep]) and _same_bits(w[keep], w_clean[keep])
        assert np.isfinite(out[2 * chunk - 3]).all() and np.isfinite(w[2 * chunk - 3])


def test_device_guard_accumulates_in_the_statistics():
    import torch
    eng = _eng()
    fk = _fk()
    ang = torch.from_numpy(_angles(10_000, 91)).cuda()
    eng.stats_reset_torch()
    fk.jacobian_device(ang)
    assert eng.stats_fetch_torch().first_fk_angle_range == -1
    bad = ang.clone()
    bad[6_001, 2] = 6.4
    bad[9_999, 0] = -np.inf
    w = torch.empty(4_000, dtype=torch.float64, device="cuda")
    fk.jacobian_device(bad[6_000:], what=None, manip_out=w)  # row 1 of this call
    fk.jacobian_device(bad, what="position")                 # row 6 001 of this one: the block keeps the lowest, 1
    assert eng.stats_fetch_torch().first_fk_angle_range == 1
    eng.stats_reset_torch()


# ---- arguments on the GPU -------------------------------------------------------------------------------------------
def test_arguments_rejected_before_launch():
    import torch
    from inversekinematicsann_b200 import _native
    eng = _eng()
    n = 8
    ang = torch.zeros(n, 4, dtype=torch.float64, device="cuda")
    out = torch.empty(n, 6, 4, dtype=torch.float64, device="cuda")
    w = torch.empty(n, dtype=torch.float64, device="cuda")
    before = eng.launch_count
    bad_device = [
        (TypeError, ang.cpu(), out, "geometric", None),
        (TypeError, ang, out.cpu(), "geometric", None),
        (ValueError, ang, out.float(), "geometric", None),
        (ValueError, ang, out, "position", None),
        (ValueError, ang, torch.empty(n + 1, 6, 4, dtype=torch.float64, device="cuda"), "geometric", None),
        (ValueError, ang, torch.empty(6, 4, n, dtype=torch.float64, device="cuda").permute(2, 0, 1), "geometric", None),
        (ValueError, ang, out, "matrices", None),
        (ValueError, ang, None, "geometric", None),
        (ValueError, ang, None, "geometric", w.float()),
        (ValueError, ang, None, "geometric", w.view(n, 1)),
        (ValueError, ang, None, "geometric", torch.empty(2 * n, dtype=torch.float64, device="cuda")[::2]),
        (TypeError, ang, None, "geometric", w.cpu()),
        (ValueError, torch.zeros(n, 3, dtype=torch.float64, device="cuda"), out, "geometric", None),
    ]
    for exc, a, o, what, m in bad_device:
        with pytest.raises(exc):
            eng.jacobian_device(a, o, what, m)
    host = np.zeros((n, 4))
    ro = np.empty((n, 6, 4))
    ro.flags.writeable = False
    bad_host = [
        (ValueError, host, ro, "geometric", False),
        (TypeError, host, np.empty((n, 6, 4), dtype=np.float32), "geometric", False),
        (ValueError, host, np.empty((n, 3, 4)), "geometric", False),
        (ValueError, host, np.empty((n, 6, 8))[:, :, ::2], "geometric", False),
        (ValueError, np.zeros((n, 3)), None, "geometric", False),
        (ValueError, host, None, "matrices", True),
        (ValueError, host, None, None, False),
        (ValueError, host, np.empty((n, 6, 4)), None, True),
        (TypeError, host, torch.empty(n, 6, 4, dtype=torch.float64), "geometric", False),
    ]
    for exc, a, o, what, m in bad_host:
        with pytest.raises(exc):
            eng.jacobian(a, what, manipulability=m, out=o)
    assert eng.launch_count == before
    lib, h = eng._lib, eng._handle
    p, q = host.ctypes.data, ro.ctypes.data
    G, P, F64 = _native.IKB_JAC_GEOMETRIC, _native.IKB_JAC_POSITION, _native.IKB_F64
    for fn in (lib.ikb_jacobian_host, lib.ikb_jacobian_device):
        assert fn(h, p, F64, -1, G, q, q, None) == _native.IKB_ERR_INVALID
        assert fn(h, p, F64, n, 2, q, None, None) == _native.IKB_ERR_INVALID
        assert fn(h, p, 5, n, P, q, None, None) == _native.IKB_ERR_INVALID
        assert fn(h, p, F64, n, G, None, None, None) == _native.IKB_ERR_INVALID
        assert fn(h, None, F64, n, G, q, None, None) == _native.IKB_ERR_INVALID
        assert fn(h, p + 4, F64, n, G, q, None, None) == _native.IKB_ERR_INVALID
        assert fn(h, p, F64, n, G, q + 4, None, None) == _native.IKB_ERR_INVALID
        assert fn(h, p, F64, n, G, None, q + 4, None) == _native.IKB_ERR_INVALID
        assert fn(None, p, F64, n, G, q, None, None) == _native.IKB_ERR_INVALID
        assert fn(h, None, F64, 0, G, None, q, None) == _native.IKB_OK
    assert eng.launch_count == before
    st = _native.IkbStats()
    assert lib.ikb_jacobian_host(h, p, F64, 0, G, q, None, ctypes.byref(st)) == _native.IKB_OK
    assert st.first_fk_angle_range == -1
