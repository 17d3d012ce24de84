"""Closed-form inverse kinematics (AnalyticInverseKinematics, IkEngine.analytic_ik / analytic_ik_device,
csrc/analytic.cu) against the NumPy restatement of include/ikb200.h (test_analytic_args.analytic_ik), against the GPU's
own forward kinematics, on degenerate rows, and across its entry points."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OFFSET_DH = [[0, 0, 0, 0], [0.7, 0.3, -0.1, 0.25], [0.4, 2.0, 1.5, 0.8], [-np.pi / 2, 0, 0, 0]]
TWISTED_DH = [[0, np.pi / 2, 0, 0], [2, 0.5, -0.25, 0.1], [0.3, 2, 1.5, 2.5], [np.pi / 2, 0.3, -0.2, 0.1]]
TABLES = ["robot", "offset"]
LIMITS = ((0.0, 6.0), (-6.0, 6.0), (-3.0, 6.0))
# Angles are compared where the problem is conditioned.  Near the stretched or folded arm an error dr in the wrist
# distance moves theta_3 by about dr r / (a_2 a_3 |sin theta_3|), so two correct fp64 evaluations that differ by an ulp
# in r differ by ~1e-11 rad at |sin theta_3| = 1e-4: the bar is 1e-12 rad from |sin theta_3| >= 1e-2 and 1e-10 from
# 1e-4.  The same holds for theta_1 of poses whose joint axis is nearly vertical (only poses no angles produce) and of
# positions close to the cylinder rho = |d| (q near 0).
SIN3 = 1e-4
PI = math.pi


def _robot():
    from inversekinematicsann_b200.robot.robot import SixDOFRobot
    return SixDOFRobot


def _dh(table):
    return {"robot": _robot().dh_matrix, "offset": OFFSET_DH, "twisted": TWISTED_DH}[table]


def _eng(table="robot"):
    from inversekinematicsann_b200.kinematics._shared import get_engine
    return get_engine(dh_matrix=_dh(table))


def _fresh_eng(table="robot"):
    """An engine of its own, so that its staging slots are sized by the first host call."""
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    return IkEngine(_dh(table), R.links_lengths, R.effector_workspace_limits)


def _aik(table="robot"):
    from inversekinematicsann_b200.kinematics.inverse import AnalyticInverseKinematics
    R = _robot()
    return AnalyticInverseKinematics(_dh(table), R.links_lengths, R.effector_workspace_limits)


def _angles(n, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.rand(n, 4, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * PI


def _poses(eng, th):
    """fkine_batch(th)[0] on the device: (n, 4, 4)."""
    import torch
    out = torch.empty((th.shape[0], 4, 4, 4), dtype=th.dtype, device=th.device)
    eng.fk_transforms_device(th, out, "matrices")
    return out[:, 3].contiguous()


def _angle_diff(a, b):
    """|a - b| modulo 2 pi (NumPy or torch)."""
    import torch
    d = a - b
    if not torch.is_tensor(d):
        return np.abs(np.remainder(d + PI, 2 * PI) - PI)
    return (torch.remainder(d + PI, 2 * PI) - PI).abs()


def _run(eng, x, pitch, dtype="float64", status=True):
    import torch
    B = 2 if pitch is None else 4
    out = torch.empty((x.shape[0], B, 4), dtype=getattr(torch, dtype), device=x.device)
    st = torch.empty(x.shape[0], dtype=torch.int32, device=x.device) if status else None
    eng.analytic_ik_device(x, pitch, out, st)
    return out, st


# ---- against NumPy ------------------------------------------------------------------------------------------------

def _inputs(eng, kind, n, seed):
    """Poses of random angles and the same positions with random rotations (poses no angles produce), or points in
    and around the reach with random pitches."""
    import torch
    th = _angles(n, seed)
    T = _poses(eng, th)
    if kind == "pose":
        g = torch.Generator(device="cuda").manual_seed(seed + 1)
        q = torch.randn(n // 2, 4, device="cuda", generator=g, dtype=torch.float64)
        w, x, y, z = (q / torch.linalg.vector_norm(q, dim=1, keepdim=True)).unbind(1)
        R = torch.stack([torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], -1),
                         torch.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)], -1),
                         torch.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1)], -2)
        T[n // 2:, :3, :3] = R
        return T, None
    g = torch.Generator(device="cuda").manual_seed(seed + 2)
    pts = T[:, :3, 3] * (0.5 + torch.rand(n, 1, device="cuda", generator=g, dtype=torch.float64))
    pitch = (torch.rand(n, device="cuda", generator=g, dtype=torch.float64) * 2 - 1) * PI
    return pts.contiguous(), pitch


@pytest.mark.parametrize("table", TABLES)
@pytest.mark.parametrize("kind", ["pose", "position"])
def test_matches_numpy(table, kind):
    from test_analytic_args import analytic_ik
    eng = _eng(table)
    x, pitch = _inputs(eng, kind, 1 << 16, 3)
    out, st = _run(eng, x, pitch)
    got, got_st = out.cpu().numpy(), st.cpu().numpy()
    want, want_st = analytic_ik(x.cpu().numpy(), _dh(table), None if pitch is None else pitch.cpu().numpy())
    assert np.array_equal(got_st, want_st), f"status differs on {(got_st != want_st).sum()} rows"
    xh = x.cpu().numpy()
    if kind == "pose":  # theta_1 from the joint axis' horizontal part
        lever = np.hypot(xh[:, 0, 2], xh[:, 1, 2])
    else:  # theta_1 from q = sqrt(rho^2 - d^2)
        dh = np.asarray(_dh(table))
        lever = np.sqrt(np.abs(xh[:, 0] ** 2 + xh[:, 1] ** 2 - ((dh[1, 1] + dh[1, 2]) + dh[1, 3]) ** 2))
    sin3 = np.abs(np.sin(want[:, :, 2]))
    d = _angle_diff(got, want).max(axis=2)
    for lo, bar in ((1e-2, 1e-12), (SIN3, 1e-10)):
        ok = (sin3 >= lo) & (lever[:, None] >= 1e-2)
        assert d[ok].max() <= bar, f"{d[ok].max():.3e} rad from NumPy ({(d[ok] > bar).sum()} branches)"
    print(f"{table} {kind}: max {d[sin3 >= SIN3].max():.3e} rad where |sin theta3| >= 1e-4, "
          f"{d[(sin3 >= 1e-2) & (lever[:, None] >= 1e-2)].max():.3e} where conditioned")
    assert np.isfinite(got).all() and (np.abs(got) <= PI).all()


# ---- round trip through the GPU's forward kinematics --------------------------------------------------------------

@pytest.mark.parametrize("table", TABLES)
def test_pose_round_trip(table):
    import torch
    eng = _eng(table)
    n = 1 << 20
    th = _angles(n, 5)
    T = _poses(eng, th)
    out, st = _run(eng, T, None)
    back = _poses(eng, out.view(-1, 4)).view(n, 2, 4, 4)
    err = (back[:, :, :3] - T[:, None, :3]).abs().amax()
    assert float(err) <= 1e-13, f"FK of a branch is {float(err):.3e} from its pose"
    d = _angle_diff(out, th[:, None]).amax(dim=2).amin(dim=1)
    ok = th[:, 2].sin().abs() >= SIN3
    print(f"{table}: FK of the branches within {float(err):.3e}, theta recovered to {float(d[ok].max()):.3e} rad")
    assert float(d[ok].max()) <= 1e-9, f"theta recovered to {float(d[ok].max()):.3e} rad"
    assert int(st.count_nonzero()) <= n // 10000, "a pose of some angles is reported out of reach"
    del back
    torch.cuda.empty_cache()


@pytest.mark.parametrize("table", TABLES)
def test_position_round_trip(table):
    import torch
    eng = _eng(table)
    n = 1 << 20
    th = _angles(n, 7)
    T = _poses(eng, th)
    p = T[:, :3, 3].contiguous()
    phi = th[:, 1:].sum(dim=1)
    best = None
    for pitch in (phi.contiguous(), (PI - phi).contiguous()):
        out, st = _run(eng, p, pitch)
        back = _poses(eng, out.view(-1, 4)).view(n, 4, 4, 4)
        reached = ((st[:, None] >> torch.arange(4, device="cuda", dtype=torch.int32)) & 1) == 0
        perr = (back[:, :, :3, 3] - p[:, None]).abs().amax(dim=2)
        assert float(perr[reached].max()) <= 1e-13, f"a reached branch is {float(perr[reached].max()):.3e} m off"
        if table == "robot":  # d = 0: every branch has the same tool axis
            x4 = back[:, :, :3, 0]
            assert float((x4 - x4[:, :1]).abs().max()) <= 1e-13
        d = _angle_diff(out, th[:, None]).amax(dim=2).amin(dim=1)
        best = d if best is None else torch.minimum(best, d)
        del back
    q = th[:, 0].cos() * p[:, 0] + th[:, 0].sin() * p[:, 1]  # the in-plane reach of the original angles
    ok = (th[:, 2].sin().abs() >= SIN3) & (q.abs() >= 1e-2)
    print(f"{table}: theta recovered to {float(best[th[:, 2].sin().abs() >= SIN3].max()):.3e} rad where "
          f"|sin theta3| >= 1e-4, {float(best[ok].max()):.3e} with |q| >= 1e-2 too")
    assert float(best[ok].max()) <= 1e-9, f"theta recovered to {float(best[ok].max()):.3e} rad"
    torch.cuda.empty_cache()


# ---- degenerate rows ----------------------------------------------------------------------------------------------

def _host(eng, x, pitch=None, out_dtype=np.float64):
    return eng.analytic_ik(np.asarray(x, dtype=np.float64), pitch, out_dtype)


def test_stretched_and_folded_arms():
    """theta_3 = 0 and +-pi poses, and wrists beyond reach and inside the inner radius: t = 0 gives both elbow branches
    the same bits; a wrist out of reach sets the status and points the arm at it, stretched or folded."""
    from test_analytic_args import analytic_ik
    for table in TABLES:
        eng = _eng(table)
        th = np.array([[0.3, 0.4, 0.0, -0.2], [-1.0, 1.2, PI, 0.5], [2.0, -0.7, -PI, 0.1], [0.0, 0.0, 0.0, 0.0]])
        T, _ = eng.fk_transforms(th, "matrices")
        T = np.ascontiguousarray(T[:, 3])
        ang, st, _ = _host(eng, T)
        want, want_st = analytic_ik(T, _dh(table))
        assert np.array_equal(st, want_st)
        stretched = ang[:, 0, 2] == 0.0
        assert np.array_equal(ang[stretched, 0].view(np.int64), ang[stretched, 1].view(np.int64))
        assert (np.abs(np.abs(ang[[1, 2], 0, 2]) - PI) < 1e-6).all()
    eng = _eng("offset")  # a_2 = 2, a_3 = 1.5: the wrist's inner radius is 0.5
    dh = np.asarray(OFFSET_DH)
    a1, a4, eps1 = dh[2, 0], dh[2, 3], dh[1, 0]
    # pitch 0, front branch: the wrist is at in-plane (q - a1 - a4, z - eps1) from joint 2
    pts = np.array([[9.0, 0.0, 0.7], [a1 + a4 + 0.2, 0.45, eps1 + 0.1]])
    ang, st, _ = _host(eng, pts, 0.0)
    assert st[0] & 3 == 3 and (ang[0, :2, 2] == 0.0).all()            # beyond reach: stretched (t = 0)
    assert np.array_equal(ang[0, 0].view(np.int64), ang[0, 1].view(np.int64))
    assert st[1] & 3 == 3 and np.allclose(np.abs(ang[1, :2, 2]), PI)  # inside the inner radius: folded (t = pi)
    want, want_st = analytic_ik(pts, OFFSET_DH, 0.0)
    assert np.array_equal(st, want_st) and _angle_diff(ang, want).max() <= 1e-12
    # exactly at full reach (num = 0) reaches: on the robot's table the wrist of (6, 0, 2) at pitch 0 is 4 m away
    full, full_st, _ = _host(_eng("robot"), [[6.0, 0.0, 2.0]], 0.0)
    assert full_st[0] & 3 == 0 and (full[0, :2, 2] == 0.0).all()
    # stretched and folded arms point at the wrist: the wrist's direction from joint 2 is theta_2 (+ theta_3)
    for row, t in ((0, 0.0), (1, PI)):
        q = math.sqrt(pts[row, 0] ** 2 + pts[row, 1] ** 2 - 0.45 ** 2)
        beta = math.atan2(-(pts[row, 2] - eps1), q - a1 - a4)  # s = -1 for alpha_1 = -pi/2
        assert abs(_angle_diff(np.array(ang[row, 0, 1]), np.array(beta))) < 1e-12, (row, t)


def test_inside_the_lateral_offset():
    from test_analytic_args import analytic_ik
    eng = _eng("offset")  # d = 0.45
    pts = np.array([[0.1, 0.1, 1.0], [0.0, 0.0, 0.5], [0.3, -0.2, 2.0]])
    ang, st, _ = _host(eng, pts, np.array([0.0, -PI / 2, 1.0]))
    assert (st == 15).all() and np.isfinite(ang).all()
    want, want_st = analytic_ik(pts, OFFSET_DH, np.array([0.0, -PI / 2, 1.0]))
    assert np.array_equal(st, want_st) and np.abs(_angle_diff(ang, want)).max() <= 1e-12


def test_base_axis_signed_zeros():
    """Every signed zero of a point (or pose) on the base axis gives the same bits; with d = 0 a point there gets
    theta_1 = 0 on the front branches and -pi on the back ones."""
    import itertools
    eng = _eng("robot")
    rows = np.array([[x, y, z] for x, y in itertools.product((0.0, -0.0), repeat=2) for z in (2.0, 5.0, 7.5)])
    ang, st, _ = _host(eng, rows, -PI / 2)
    bits = ang.view(np.int64).reshape(4, 3, -1)
    assert (bits == bits[:1]).all() and (st.reshape(4, 3) == st.reshape(4, 3)[:1]).all()
    assert (ang[:, :2, 0] == 0.0).all() and (ang[:, 2:, 0] == -PI).all()
    # poses on the axis: theta = (t1, pi/2, 0, 0) puts the arm straight up; every zero entry flips sign
    T, _ = eng.fk_transforms(np.array([[0.4, PI / 2, 0.0, 0.0], [-2.0, PI / 2, 0.5, -0.5]]), "matrices")
    T = np.ascontiguousarray(T[:, 3])
    T[:, 0, 3] = T[:, 1, 3] = 0.0
    T[np.abs(T) < 1e-15] = 0.0
    base, bst, _ = _host(eng, T)
    zeros = np.argwhere(T[:, :3] == 0.0)
    for k in range(len(zeros) + 1):
        V = T.copy()
        for idx in zeros[:k]:
            V[tuple(idx)] = -0.0
        a, s, _ = _host(eng, V)
        assert np.array_equal(a.view(np.int64), base.view(np.int64)) and np.array_equal(s, bst)


def test_non_finite_rows():
    eng = _eng("robot")
    T, _ = eng.fk_transforms(np.array([[0.1, 0.2, 0.3, 0.4]] * 6), "matrices")
    T = np.ascontiguousarray(T[:, 3])
    T[0, 0, 0], T[1, 2, 3], T[2, 1, 2] = np.nan, np.inf, -np.inf
    T[3, 3, 0] = np.nan  # row 3 of a pose is not read
    ang, st, _ = _host(eng, T)
    assert np.isnan(ang[:3]).all() and (st[:3] == 3).all()
    assert np.isfinite(ang[3:]).all() and np.array_equal(ang[3], ang[4])
    pts = np.array([[np.nan, 1, 1], [1, np.inf, 1], [2, 1, 1], [2, 1, 1]])
    ang, st, _ = _host(eng, pts, np.array([0.0, 0.0, np.nan, 0.5]))
    assert np.isnan(ang[:3]).all() and (st[:3] == 15).all() and np.isfinite(ang[3]).all()


def test_table_outside_the_family_is_refused():
    from inversekinematicsann_b200.kinematics.inverse import AnalyticInverseKinematics
    eng = _eng("twisted")
    before = eng.launch_count
    with pytest.raises(RuntimeError, match="outside the closed form's family.*ikine_pose / refine_pose"):
        eng.analytic_ik(np.zeros((4, 4, 4)))
    import torch
    with pytest.raises(RuntimeError, match="outside the closed form's family"):
        _run(eng, torch.zeros((4, 3), dtype=torch.float64, device="cuda"),
             torch.zeros(1, dtype=torch.float64, device="cuda"))
    assert eng.launch_count == before
    R = _robot()
    ik = AnalyticInverseKinematics(TWISTED_DH, R.links_lengths, R.effector_workspace_limits)
    with pytest.raises(RuntimeError, match="outside the closed form's family"):
        ik.ikine([[1.0, 1.0, 1.0]], 0.0)


# ---- consistency across paths -------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["pose", "position"])
def test_float32_host_device_and_chunks(kind):
    """float32 outputs are the float64 ones rounded once; the host path (three chunks) equals the device path bit for
    bit and reports the lowest out-of-box row by its global index; float32 inputs are widened exactly."""
    import torch
    eng = _fresh_eng("offset")
    n = 5000  # slots of 8192 rows: host chunks of 2048
    x, pitch = _inputs(_eng("offset"), kind, n, 11)
    col = (lambda t: t[:, :3, 3]) if kind == "pose" else (lambda t: t)
    lim = torch.tensor([hi for _, hi in LIMITS], dtype=torch.float64, device="cuda")
    x = x.clone()
    col(x)[:] = torch.minimum(col(x), lim - 0.5).clamp_min(0.25)
    col(x)[4500, 0] = 7.0
    col(x)[4999, 2] = -4.0
    eng.stats_reset_torch()
    d64, s64 = _run(eng, x, pitch)
    d32, s32 = _run(eng, x, pitch, "float32")
    stats = eng.stats_fetch_torch()
    assert stats.first_out_of_limits == 4500 and stats.n_solved == 2 * n
    assert torch.equal(d32, d64.float()) and torch.equal(s32, s64)
    xh = x.cpu().numpy()
    ph = None if pitch is None else pitch.cpu().numpy()
    for dtype, dev in ((np.float64, d64), (np.float32, d32)):
        h, hs, hstats = eng.analytic_ik(xh, ph, dtype)
        assert np.array_equal(h.view(np.uint8), dev.cpu().numpy().view(np.uint8)) and np.array_equal(hs, s64.cpu().numpy())
        assert hstats.first_out_of_limits == 4500 and hstats.n_solved == n
    # float32 inputs: the fp64 arithmetic on the widened values
    h32, hs32, _ = eng.analytic_ik(xh.astype(np.float32), None if ph is None else ph.astype(np.float32))
    w64, ws64, _ = eng.analytic_ik(xh.astype(np.float32).astype(np.float64),
                                   None if ph is None else ph.astype(np.float32).astype(np.float64))
    assert np.array_equal(h32.view(np.int64), w64.view(np.int64)) and np.array_equal(hs32, ws64)
    eng.close()


def test_broadcast_pitch_and_unaligned_output():
    import torch
    eng = _eng("robot")
    x, _ = _inputs(eng, "position", 4096, 13)
    one = torch.tensor([-PI / 2], dtype=torch.float64, device="cuda")
    a, sa = _run(eng, x, one)
    b, sb = _run(eng, x, one.expand(4096).contiguous())
    assert torch.equal(a, b) and torch.equal(sa, sb)
    buf = torch.empty(4096 * 16 + 1, dtype=torch.float64, device="cuda")  # 8-byte aligned: element stores
    out = buf[1:].view(4096, 4, 4)
    eng.analytic_ik_device(x, one, out)
    assert torch.equal(out, a)
    h, hs, _ = eng.analytic_ik(x.cpu().numpy(), -PI / 2)
    assert np.array_equal(h, a.cpu().numpy()) and np.array_equal(hs, sa.cpu().numpy())


@pytest.mark.parametrize("kind", ["pose", "position"])
def test_side_stream_with_late_inputs(kind):
    """On a side stream whose inputs hold decoys until a ~30 ms sleep there has passed, the call sees the real rows."""
    import torch
    eng = _eng("robot")
    x, pitch = _inputs(eng, kind, 8192, 17)
    want, want_st = _run(eng, x, pitch)
    torch.cuda.synchronize()
    xs, ps = torch.zeros_like(x), None if pitch is None else torch.zeros_like(pitch)
    out = torch.full_like(want, 5.0)
    st = torch.full_like(want_st, 99)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(60_000_000)
        xs.copy_(x)
        if ps is not None:
            ps.copy_(pitch)
        eng.analytic_ik_device(xs, ps, out, st)
    s.synchronize()
    assert torch.equal(out, want) and torch.equal(st, want_st)


# ---- the solver class ---------------------------------------------------------------------------------------------

def _box_poses(eng, n, seed):
    """r07 workload (a): poses of random angles whose position is inside the workspace box."""
    import torch
    th = _angles(3 * n, seed)
    T = _poses(eng, th)
    p = T[:, :3, 3]
    ok = torch.ones(3 * n, dtype=torch.bool, device="cuda")
    for i, (lo, hi) in enumerate(LIMITS):
        ok &= (p[:, i] >= lo) & (p[:, i] <= hi)
    return th[ok][:n].contiguous(), T[ok][:n].contiguous()


def test_ikine_pose_converges_on_every_row():
    from inversekinematicsann_b200 import engine as E
    ik = _aik()
    th, T = _box_poses(_eng(), 1 << 20, 19)
    assert T.shape[0] == 1 << 20
    Th = T.cpu().numpy()
    out, its, err = ik.ikine_pose(Th, as_array=True, return_iterations=True, return_fk_error=True)
    assert (err <= E.POSE_TOL).all(), f"{(err > E.POSE_TOL).sum()} rows above tol"
    print(f"steps: mean {its.mean():.4f}, at 0: {(its == 0).mean():.6f}, max {its.max()}")
    closed, _, err0 = ik.ikine_pose(Th[:4096], refine=False, as_array=True, return_iterations=True,
                                    return_fk_error=True)
    ang, _ = ik.ikine_pose_branches(Th[:4096])
    assert np.array_equal(closed, ang[:, 0]) and np.isfinite(err0).all()
    neg = ik.ikine_pose(Th[:64], elbow=-1, refine=False, as_array=True)
    assert np.array_equal(neg, ang[:64, 1])


def test_solver_methods_and_limits():
    import torch
    ik = _aik()
    pts = [[2.0, 1.0, 1.0], [3.0, -1.0, 0.5]]
    br, st = ik.ikine_branches(pts, -PI / 2)
    for e, b in ((1, "front"), (-1, "front"), (1, "back"), (-1, "back")):
        got, s = ik.ikine(pts, -PI / 2, elbow=e, base=b, as_array=True, return_status=True)
        k = {"front": 0, "back": 2}[b] + (0 if e == 1 else 1)
        assert np.array_equal(got, br[:, k]) and np.array_equal(s, (st >> k) & 1)
    assert ik.ikine(pts, -PI / 2) == br[:, 0].tolist()
    dev = ik.ikine_device(torch.tensor(pts, dtype=torch.float64, device="cuda"), -PI / 2)
    assert np.array_equal(dev.cpu().numpy(), br)
    with pytest.raises(Exception, match=r"point \[7\.0, 1\.0, 1\.0\] is out of manipulator reach area"):
        ik.ikine([[2.0, 1.0, 1.0], [7.0, 1.0, 1.0]], 0.0)
    T, _ = _eng().fk_transforms(np.array([[0.2, 0.3, -0.4, 0.5], [0.0, 0.0, 0.0, 0.0]]), "matrices")
    T = np.ascontiguousarray(T[:, 3])
    T[1, :3, 3] = [1.0, 8.0, 1.0]
    with pytest.raises(Exception, match=r"point \[1\.0, 8\.0, 1\.0\] is out of manipulator reach area"):
        ik.ikine_pose(T)
    with pytest.raises(Exception, match="out of manipulator reach area"):
        ik.ikine_pose_branches(T)
    pb, _ = ik.ikine_pose_branches(T[:1])
    dev = ik.ikine_pose_device(torch.from_numpy(T[:1]).cuda())
    assert np.array_equal(dev.cpu().numpy(), pb)
