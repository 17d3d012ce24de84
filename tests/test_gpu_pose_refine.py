"""Damped-least-squares refinement of joint angles onto full effector poses (InverseKinematics.refine_pose /
refine_pose_device / ikine_pose, IkEngine.dls_pose_refine / dls_pose_refine_device, csrc/fk.cu
dls_pose_refine_kernel).

The kernel builds on the chain of fkine_batch and jacobian_batch, so a NumPy restatement of the operation order in
include/ikb200.h, iterated on the GPU's own fkine_batch and jacobian_batch, reproduces every step bit for bit.
Independent checks: the closed form of the quaternion error, the C oracle's FK for converged rows, and the position
refinement (dls_refine), whose step is the same mathematically for weights (1, 1, 1, 0, 0, 0)."""
import math
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TWISTED_DH = [[0, np.pi / 2, 0, 0], [2, 0.5, -0.25, 0.1], [0.3, 2, 1.5, 2.5], [np.pi / 2, 0.3, -0.2, 0.1]]
TABLES = ["robot", "twisted"]
ANGLE_MSG = "Forward Kinematics exception, robot joints angles limits are (-2pi, 2pi)"
TOL = 1e-9
DH_SEED = [0.0, np.pi / 2, 0.0, 0.0]
ONES = (1.0, 1.0, 1.0, 1.0, 1.0, 1.0)
POSITION_ONLY = (1.0, 1.0, 1.0, 0.0, 0.0, 0.0)
WEIGHTS = [ONES, POSITION_ONLY, (0.0, 0.0, 0.0, 1.0, 1.0, 1.0), (2.0, 0.5, 1.0, 0.3, 0.0, 1.7)]
LIMITS = ((0.0, 6.0), (-6.0, 6.0), (-3.0, 6.0))


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


def _ik(cls="fabrik"):
    from inversekinematicsann_b200.kinematics.inverse import AnnInverseKinematics, FabrikInverseKinematics
    R = _robot()
    if cls == "fabrik":
        return FabrikInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    ik = AnnInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ik.load_model(os.path.join(root, "models", "roboarm_b200_r01.h5"))
    return ik


def _defaults():
    from inversekinematicsann_b200 import engine
    return engine.POSE_DAMPING, engine.POSE_MAX_ITER


def _same_bits(a, b):
    """Equal bit for bit, except that any NaN equals any NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    nan = np.isnan(a)
    u = {8: np.uint64, 4: np.uint32}[a.dtype.itemsize]
    return bool(np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(u), b[~nan].view(u)))


def _angles(n, seed, lo=-np.pi, hi=np.pi):
    return np.random.default_rng(seed).uniform(lo, hi, size=(n, 4))


def _in_box(p):
    return np.all([(p[:, i] >= lo) & (p[:, i] <= hi) for i, (lo, hi) in enumerate(LIMITS)], axis=0)


def _reachable_poses(n, seed, table="robot"):
    """(angles, poses): fkine_batch of random angles whose effector is inside the workspace box."""
    fk = _fk(table)
    rng = np.random.default_rng(seed)
    th = []
    while sum(len(t) for t in th) < n:
        t = rng.uniform(-np.pi, np.pi, size=(2 * n + 64, 4))
        th.append(t[_in_box(fk.fkine_batch(t)[0][:, :3, 3])])
    th = np.ascontiguousarray(np.vstack(th)[:n])
    return th, np.ascontiguousarray(fk.fkine_batch(th)[0])


def _rotation(axis, theta):
    """Rodrigues' rotation matrices for (n, 3) unit axes and (n,) angles."""
    x, y, z = axis[:, 0], axis[:, 1], axis[:, 2]
    c, s = np.cos(theta), np.sin(theta)
    C = 1 - c
    return np.stack([np.stack([c + x * x * C, x * y * C - z * s, x * z * C + y * s], -1),
                     np.stack([y * x * C + z * s, c + y * y * C, y * z * C - x * s], -1),
                     np.stack([z * x * C - y * s, z * y * C + x * s, c + z * z * C], -1)], -2)


def _unit(n, rng):
    u = rng.standard_normal((n, 3))
    return u / np.linalg.norm(u, axis=1, keepdims=True)


def _random_rotation_poses(n, seed, table="robot"):
    """Reachable positions with uniformly random rotations: generally not a pose of the arm."""
    rng = np.random.default_rng(seed)
    _, poses = _reachable_poses(n, seed + 1000, table)
    poses[:, :3, :3] = _rotation(_unit(n, rng), rng.uniform(0.0, np.pi, n))
    return poses


# ---- the NumPy restatement (operation order of include/ikb200.h) -------------------------------------------------
def np_pose_error(Rd, pd, T, w):
    """-> (e (m, 6), weighted err (m,)) for target rotations Rd (m, 3, 3), positions pd (m, 3) and poses T (m, 4, 4)."""
    R, p = T[:, :3, :3], T[:, :3, 3]
    M = np.empty(Rd.shape)
    for i in range(3):
        for j in range(3):
            M[:, i, j] = (Rd[:, i, 0] * R[:, j, 0] + Rd[:, i, 1] * R[:, j, 1]) + Rd[:, i, 2] * R[:, j, 2]
    tr = (M[:, 0, 0] + M[:, 1, 1]) + M[:, 2, 2]
    dx, dy, dz = M[:, 2, 1] - M[:, 1, 2], M[:, 0, 2] - M[:, 2, 0], M[:, 1, 0] - M[:, 0, 1]
    sxy, sxz, syz = M[:, 0, 1] + M[:, 1, 0], M[:, 0, 2] + M[:, 2, 0], M[:, 1, 2] + M[:, 2, 1]
    c0 = (tr >= M[:, 0, 0]) & (tr >= M[:, 1, 1]) & (tr >= M[:, 2, 2])
    c1 = ~c0 & (M[:, 0, 0] >= M[:, 1, 1]) & (M[:, 0, 0] >= M[:, 2, 2])
    c2 = ~c0 & ~c1 & (M[:, 1, 1] >= M[:, 2, 2])
    eo = np.empty((M.shape[0], 3))
    with np.errstate(all="ignore"):
        h = np.sqrt(1.0 + tr)
        cand0 = np.stack([dx / h, dy / h, dz / h], -1)
        h = np.sqrt(((1.0 + M[:, 0, 0]) - M[:, 1, 1]) - M[:, 2, 2])
        cand1 = np.stack([h, sxy / h, sxz / h], -1)
        cand1 = np.where((dx < 0)[:, None], -cand1, cand1)
        h = np.sqrt(((1.0 + M[:, 1, 1]) - M[:, 0, 0]) - M[:, 2, 2])
        cand2 = np.stack([sxy / h, h, syz / h], -1)
        cand2 = np.where((dy < 0)[:, None], -cand2, cand2)
        h = np.sqrt(((1.0 + M[:, 2, 2]) - M[:, 0, 0]) - M[:, 1, 1])
        cand3 = np.stack([sxz / h, syz / h, h], -1)
        cand3 = np.where((dz < 0)[:, None], -cand3, cand3)
    eo = np.where(c0[:, None], cand0, np.where(c1[:, None], cand1, np.where(c2[:, None], cand2, cand3)))
    e = np.concatenate([pd - p, eo], axis=1)
    s = w[None, :] * (e * e)
    err = np.sqrt(((s[:, 0] + s[:, 1]) + s[:, 2]) + ((s[:, 3] + s[:, 4]) + s[:, 5]))
    return e, err


def np_pose_refine(fk, poses, seed, weights, damping, tol, max_iter):
    """-> (angles, iters, err) in fp64; T_4 and J of every iterate from the GPU's fkine_batch / jacobian_batch."""
    poses = np.asarray(poses, dtype=np.float64)
    n = poses.shape[0]
    w = np.asarray(weights, dtype=np.float64)
    th = np.array(np.broadcast_to(seed, (n, 4)), dtype=np.float64)
    iters = np.zeros(n, dtype=np.int32)
    err_out = np.full(n, np.nan)
    active = np.ones(n, dtype=bool)
    lam2 = damping * damping
    k = 0
    while active.any():
        idx = np.flatnonzero(active)
        t = th[idx]
        T = fk.fkine_batch(t)[0]
        J = fk.jacobian_batch(t, "geometric")
        e, err = np_pose_error(poses[idx, :3, :3], poses[idx, :3, 3], T, w)
        done = (err <= tol) | (k == max_iter)
        err_out[idx[done]] = err[done]
        iters[idx[done]] = k
        active[idx[done]] = False
        go = ~done
        if not go.any():
            break
        J, e, t = J[go], e[go], t[go]
        g = w[None, :, None] * J
        A = np.zeros((J.shape[0], 4, 4))
        b = np.zeros((J.shape[0], 4))
        for kk in range(4):
            c = [g[:, i, kk] * e[:, i] + g[:, 3 + i, kk] * e[:, 3 + i] for i in range(3)]
            b[:, kk] = (c[0] + c[1]) + (c[2] + 0.0)
            for m in range(kk, 4):
                P = [g[:, i, kk] * J[:, i, m] + g[:, 3 + i, kk] * J[:, 3 + i, m] for i in range(3)]
                A[:, kk, m] = (P[0] + P[1]) + (P[2] + 0.0)
        for kk in range(4):
            A[:, kk, kk] = A[:, kk, kk] + lam2
        l10, l20, l30 = A[:, 0, 1] / A[:, 0, 0], A[:, 0, 2] / A[:, 0, 0], A[:, 0, 3] / A[:, 0, 0]
        d1 = A[:, 1, 1] - l10 * A[:, 0, 1]
        t21 = A[:, 1, 2] - l20 * A[:, 0, 1]
        t31 = A[:, 1, 3] - l30 * A[:, 0, 1]
        l21, l31 = t21 / d1, t31 / d1
        d2 = (A[:, 2, 2] - l20 * A[:, 0, 2]) - l21 * t21
        t32 = (A[:, 2, 3] - l30 * A[:, 0, 2]) - l31 * t21
        l32 = t32 / d2
        d3 = ((A[:, 3, 3] - l30 * A[:, 0, 3]) - l31 * t31) - l32 * t32
        z1 = b[:, 1] - l10 * b[:, 0]
        z2 = (b[:, 2] - l20 * b[:, 0]) - l21 * z1
        z3 = ((b[:, 3] - l30 * b[:, 0]) - l31 * z1) - l32 * z2
        y3 = z3 / d3
        y2 = z2 / d2 - l32 * y3
        y1 = (z1 / d1 - l21 * y2) - l31 * y3
        y0 = ((b[:, 0] / A[:, 0, 0] - l10 * y1) - l20 * y2) - l30 * y3
        t = t + np.stack([y0, y1, y2, y3], axis=1)
        for r, c in zip(*np.nonzero(np.abs(t) > math.pi)):
            t[r, c] = math.remainder(t[r, c], 2 * math.pi)
        th[idx[go]] = t
        k += 1
    return th, iters, err_out


def _mixed_targets(n, table, seed):
    """Half poses of random angles, half random rotations at reachable positions."""
    _, a = _reachable_poses(n // 2, seed, table)
    return np.ascontiguousarray(np.concatenate([a, _random_rotation_poses(n - n // 2, seed + 1, table)]))


# ---- 1. step bits --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_iter", [0, 1, 2, 3])
@pytest.mark.parametrize("table", TABLES)
def test_step_bits_against_the_numpy_restatement(table, max_iter):
    """tol = 0: every row takes max_iter steps; seeds across [-2pi, 2pi] exercise the wrap."""
    eng, fk = _eng(table), _fk(table)
    n = 2000
    th, poses = _reachable_poses(n // 2, 1, table)
    poses = np.ascontiguousarray(np.concatenate([poses, _random_rotation_poses(n - n // 2, 2, table)]))
    seed = np.vstack([_angles(n // 2, 3), _angles(n - n // 2, 4, -6.2, 6.2)])
    seed[:n // 8] = th[:n // 8] + _angles(n // 8, 5, -0.02, 0.02)  # near their solutions: these stop early below
    damping = _defaults()[0]
    for w in WEIGHTS:
        out, st, iters, err = eng.dls_pose_refine(poses, seed, w, damping, 0.0, max_iter, return_iters=True,
                                                  return_error=True)
        want, want_it, want_err = np_pose_refine(fk, poses, seed, w, damping, 0.0, max_iter)
        assert _same_bits(out, want) and np.array_equal(iters, want_it) and _same_bits(err, want_err), w
        assert (iters == max_iter).all() and st.n_solved == n and st.sum_iterations == n * max_iter
        if max_iter == 0:
            assert _same_bits(out, seed)
        else:
            assert (np.abs(out) <= np.pi).all()
    # a second damping, with a tolerance that stops some rows early
    out, _, iters, err = eng.dls_pose_refine(poses, seed, ONES, 0.3, 0.05, max_iter, return_iters=True,
                                             return_error=True)
    want, want_it, want_err = np_pose_refine(fk, poses, seed, ONES, 0.3, 0.05, max_iter)
    assert _same_bits(out, want) and np.array_equal(iters, want_it) and _same_bits(err, want_err)
    if max_iter:
        assert 0 < int((iters < max_iter).sum()) < n


# ---- 2. the quaternion error ---------------------------------------------------------------------------------------
def test_quaternion_error_of_constructed_rotations():
    """R_d = Rot(u, theta) R for the arm's own R and p_d = p: err = 2 sin(theta/2) sqrt(w).  The bound is a few ulps of
    the result plus the rounding of R_d R^T (entries of order 1: a few 1e-16 absolute).  theta = pi is not converged."""
    eng, fk = _eng(), _fk()
    thetas = np.array([0.0, 1e-8, 1.0, np.pi - 1e-8, np.pi])
    rng = np.random.default_rng(5)
    axes = np.vstack([np.eye(3), -np.eye(3), _unit(6, rng)])
    th0 = _angles(axes.shape[0], 6)
    T = fk.fkine_batch(th0)[0]
    rows, seeds, want = [], [], []
    for theta in thetas:
        P = T.copy()
        P[:, :3, :3] = _rotation(axes, np.full(axes.shape[0], theta)) @ T[:, :3, :3]
        rows.append(P)
        seeds.append(th0)
        want.append(np.full(axes.shape[0], 2 * math.sin(theta / 2)))
    poses, seed, want = np.concatenate(rows), np.concatenate(seeds), np.concatenate(want)
    for w_o in (1.0, 2.5):
        _, st, it, err = eng.dls_pose_refine(poses, seed, (1, 1, 1, w_o, w_o, w_o), max_iter=0, tol=TOL,
                                             return_iters=True, return_error=True)
        exp = want * math.sqrt(w_o)
        bound = 8 * np.spacing(exp) + 2e-15 * math.sqrt(w_o)
        assert (np.abs(err - exp) <= bound).all(), np.abs(err - exp).max()
        conv = err <= TOL
        assert conv[:axes.shape[0]].all() and not conv[axes.shape[0]:].any()  # theta = 0 only
        assert st.n_iter_capped == int((~conv).sum()) and (it == 0).all()
    # the restatement agrees bit for bit here too
    _, _, _, err = eng.dls_pose_refine(poses, seed, ONES, max_iter=0, return_iters=True, return_error=True)
    assert _same_bits(err, np_pose_refine(fk, poses, seed, ONES, 0.1, TOL, 0)[2])


# ---- 3. round trip -------------------------------------------------------------------------------------------------
# Bars from the measurement (profiles/r07_pose_bench.json: the sweep's 2^20 poses of random angles at the default
# damping, within the default 128 steps): 0.904 of the FABRIK-seeded rows, 0.907 of the network-seeded ones and 0.945
# from the DH seed row converged.  Almost all of the others start with theta_1 about pi from the pose's own (FABRIK and
# the network put the arm on the target's side of the base; half of these poses reach back over it) and end at a
# local minimum with the orientation about pi off.  The bars are about 6.5 standard deviations below these for 20 000 rows.
FABRIK_ROUND_TRIP_BAR = 0.89
ANN_ROUND_TRIP_BAR = 0.89
DH_SEED_ROUND_TRIP_BAR = 0.935
POSITION_BOUND = 1e-9 + 1e-12     # ||p - p*|| of a converged row (err <= tol bounds the weighted position error)
ROTATION_BOUND = 2e-9             # max |R - R*| elementwise: |e_o| <= tol bounds the rotation angle by ~tol


def _check_converged_with_the_oracle(T, out, conv, sample=2000):
    from oracle import c_oracle
    dh = np.asarray(_robot().dh_matrix, dtype=np.float64)
    idx = np.flatnonzero(conv)[:sample]
    for i in idx:
        st, chain = c_oracle.fk_chain(out[i], dh=dh)
        assert st == 0
        assert np.linalg.norm(chain[3][:3, 3] - T[i, :3, 3]) <= POSITION_BOUND
        assert np.abs(chain[3][:3, :3] - T[i, :3, :3]).max() <= ROTATION_BOUND


def test_round_trip_fabrik_seeded_and_from_the_dh_seed():
    ik = _ik()
    _, T = _reachable_poses(20_000, 7)
    out, iters, err = ik.ikine_pose(T, as_array=True, return_iterations=True, return_fk_error=True)
    assert out.dtype == np.float64 and out.shape == (T.shape[0], 4)
    conv = err <= TOL
    assert conv.mean() >= FABRIK_ROUND_TRIP_BAR, conv.mean()
    _check_converged_with_the_oracle(T, out, conv)
    st = ik.last_stats
    assert st.n_solved == T.shape[0] and st.n_iter_capped == int((~conv).sum())
    assert st.sum_iterations == int(iters.sum())
    out, iters, err = ik.refine_pose(T, DH_SEED, as_array=True, return_iterations=True, return_fk_error=True)
    conv = err <= TOL
    assert conv.mean() >= DH_SEED_ROUND_TRIP_BAR, conv.mean()
    _check_converged_with_the_oracle(T, out, conv)


# ---- 4. the position refinement ------------------------------------------------------------------------------------
def test_position_weights_agree_with_dls_refine():
    """With weights (1, 1, 1, 0, 0, 0), (J^T J + L I)^-1 J^T e = J^T (J J^T + L I)^-1 e: the first steps agree to
    rounding, and both converge onto the same targets.  J^T J is 4 x 4 of rank 3, so J^T J + L I has condition number
    up to ||J||_F^2 / L <= 144 / 4e-6 = 3.6e7 at the default damping (each column is at most 6 m long), and its
    solution may differ from the other form's by a few times that in units of 2^-53: the bound on the step's relative
    difference is 1e-7, at seeds whose position Jacobian is well conditioned."""
    eng = _eng()
    th, T = _reachable_poses(20_000, 8)
    xyz = np.ascontiguousarray(T[:, :3, 3])
    seed = _angles(th.shape[0], 9)
    _, w, _ = eng.jacobian(seed, None, manipulability=True)
    ok = w > 0.5
    assert ok.mean() > 0.3
    a, _ = eng.dls_pose_refine(T, seed, POSITION_ONLY, max_iter=1)
    b, _ = eng.dls_refine(xyz, seed, damping=_defaults()[0], max_iter=1)
    step_a = np.vectorize(math.remainder)(a - seed, 2 * math.pi)[ok]
    step_b = np.vectorize(math.remainder)(b - seed, 2 * math.pi)[ok]
    rel = np.abs(step_a - step_b).max(axis=1) / np.abs(step_b).max(axis=1)
    assert rel.max() <= 1e-7, rel.max()
    _, _, _, ea = eng.dls_pose_refine(T, seed, POSITION_ONLY, return_iters=True, return_error=True)
    _, _, _, eb = eng.dls_refine(xyz, seed, return_iters=True, return_error=True)
    ca, cb = ea <= TOL, eb <= TOL
    assert ca.mean() >= 0.999 and cb.mean() >= 0.999 and (ca == cb).mean() >= 0.999


# ---- 5. unreachable orientations -----------------------------------------------------------------------------------
def test_random_rotations_run_to_max_iter():
    eng = _eng()
    poses = _random_rotation_poses(20_000, 10)
    max_iter = _defaults()[1]
    out, st, iters, err = eng.dls_pose_refine(poses, DH_SEED, return_iters=True, return_error=True)
    capped = err > TOL
    assert capped.mean() >= 0.99
    assert (iters[capped] == max_iter).all() and st.n_iter_capped == int(capped.sum())
    assert np.isfinite(out).all() and (np.abs(out) <= np.pi).all()


# ---- 6. the machinery shared with the position refinement --------------------------------------------------------
@pytest.mark.parametrize("table", TABLES)
def test_float32_is_the_float64_run_rounded_once(table):
    eng = _eng(table)
    poses = _mixed_targets(20_000, table, 16)
    s32 = _angles(poses.shape[0], 17).astype(np.float32)
    for tol in (TOL, 1e-4):
        o32, _, i32, e32 = eng.dls_pose_refine(poses, s32, tol=tol, return_iters=True, return_error=True)
        o64, _, i64, e64 = eng.dls_pose_refine(poses, s32.astype(np.float64), tol=tol, return_iters=True,
                                               return_error=True)
        assert o32.dtype == np.float32 and e32.dtype == np.float32
        assert _same_bits(o32, o64.astype(np.float32)) and _same_bits(e32, e64.astype(np.float32))
        assert np.array_equal(i32, i64)
    p32 = poses.astype(np.float32)  # float32 poses are widened exactly
    a, _ = eng.dls_pose_refine(p32, s32)
    b, _ = eng.dls_pose_refine(p32.astype(np.float64), s32)
    assert _same_bits(a, b)


@pytest.mark.parametrize("table", TABLES)
def test_batch_independence_in_place_and_broadcast(table):
    import torch
    eng = _eng(table)
    big_n = 2 * torch.cuda.get_device_properties(0).multi_processor_count * 64 * 4 + 17  # several refill rounds
    poses = _mixed_targets(big_n, table, 21)
    seed = _angles(big_n, 23)
    ref, _, ref_it, ref_err = eng.dls_pose_refine(poses, seed, return_iters=True, return_error=True)
    rng = np.random.default_rng(24)
    for n in list(range(1, 130, 7)) + [big_n // 2 - 1, big_n // 2 + 1, big_n]:
        sel = rng.choice(big_n, size=n, replace=False)
        out, _, it, err = eng.dls_pose_refine(poses[sel], seed[sel], return_iters=True, return_error=True)
        assert _same_bits(out, ref[sel]) and np.array_equal(it, ref_it[sel]) and _same_bits(err, ref_err[sel]), n
    one = np.array([0.3, 1.0, -0.5, 0.2])
    a, _ = eng.dls_pose_refine(poses, one)
    b, _ = eng.dls_pose_refine(poses, np.tile(one, (big_n, 1)))
    assert _same_bits(a, b)
    s = seed.copy()
    got, _ = eng.dls_pose_refine(poses, s, out=s)
    assert got is s and _same_bits(s, ref)
    d_p, d_s = torch.from_numpy(poses).cuda(), torch.from_numpy(seed).cuda()
    eng.dls_pose_refine_device(d_p, d_s, d_s)
    torch.cuda.synchronize()
    assert _same_bits(d_s.cpu().numpy(), ref)


def _slot_rows(n):
    # capi.cu ensure_slots: the next power of two >= n, at least 1024, at most 4 Mi
    want = 1024
    while want < n and want < 1 << 22:
        want <<= 1
    return want


def test_host_chunks_equal_the_device_path_and_guards_across_them():
    """A fresh engine, so that its staging slots are sized by this call alone: S / 4 rows per chunk."""
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    n = 300_000
    S = _slot_rows(n)
    chunk = S // 4
    _, poses = _reachable_poses(n, 31)
    seed = _angles(n, 32)
    with IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits) as eng:
        before = eng.launch_count
        host, st, it, err = eng.dls_pose_refine(poses, seed, return_iters=True, return_error=True)
        assert eng.launch_count - before == -(-n // chunk) >= 3
        assert st.n_solved == n and st.first_out_of_limits == -1 and st.first_fk_angle_range == -1
        d_out = torch.empty((n, 4), dtype=torch.float64, device="cuda")
        d_it = torch.empty(n, dtype=torch.int32, device="cuda")
        d_err = torch.empty(n, dtype=torch.float64, device="cuda")
        before = eng.launch_count
        eng.dls_pose_refine_device(torch.from_numpy(poses).cuda(), torch.from_numpy(seed).cuda(), d_out, d_it, d_err)
        torch.cuda.synchronize()
        assert eng.launch_count - before == 1
        assert _same_bits(d_out.cpu().numpy(), host) and np.array_equal(d_it.cpu().numpy(), it)
        assert _same_bits(d_err.cpu().numpy(), err)
        # a broadcast seed, without the optional outputs
        one, st1 = eng.dls_pose_refine(poses, DH_SEED)
        d1 = torch.empty((n, 4), dtype=torch.float64, device="cuda")
        eng.dls_pose_refine_device(torch.from_numpy(poses).cuda(), torch.tensor(DH_SEED, dtype=torch.float64, device="cuda"), d1)
        torch.cuda.synchronize()
        assert _same_bits(d1.cpu().numpy(), one)
        # the lowest guard rows, by their global row numbers
        bad_p, bad_s = poses.copy(), seed.copy()
        bad_p[2 * chunk + 7, 0, 3] = 7.0            # out of the box, after the second chunk boundary
        bad_p[chunk - 2, 2, 3] = -3.5               # the lowest, just before the first one
        bad_s[chunk + 3, 2] = 6.5                   # out of the FK range, just after it
        bad_s[chunk + 100, 0] = -np.inf
        out, st, _, e2 = eng.dls_pose_refine(bad_p, bad_s, return_iters=True, return_error=True)
        assert st.first_out_of_limits == chunk - 2 and st.first_fk_angle_range == chunk + 3
        keep = np.ones(n, dtype=bool)
        keep[[2 * chunk + 7, chunk - 2, chunk + 3, chunk + 100]] = False
        assert _same_bits(out[keep], host[keep]) and _same_bits(e2[keep], err[keep])
        assert np.isfinite(out[[2 * chunk + 7, chunk - 2, chunk + 3]]).all()
        assert np.isnan(out[chunk + 100]).any()
        before = eng.launch_count
        out, st = eng.dls_pose_refine(np.empty((0, 4, 4)), np.empty((0, 4)))
        assert out.shape == (0, 4) and st.n_solved == 0 and eng.launch_count == before


def test_nan_rows_are_not_converged_and_max_iter_zero_returns_the_seeds():
    eng, fk = _eng(), _fk()
    _, poses = _reachable_poses(8, 61)
    seed = _angles(8, 62)
    poses[2, 1, 0] = np.nan
    seed[5, 3] = np.nan
    out, st, it, err = eng.dls_pose_refine(poses, seed, max_iter=5, return_iters=True, return_error=True)
    for r in (2, 5):
        assert np.isnan(err[r]) and it[r] == 5
    assert np.isnan(out[5]).any()
    ok = np.ones(8, dtype=bool)
    ok[[2, 5]] = False
    assert np.isfinite(out[ok]).all() and np.isfinite(err[ok]).all()
    assert st.n_iter_capped == 2 + int((err[ok] > TOL).sum()) and st.n_fk_error == 6
    assert st.first_out_of_limits == -1 and st.first_fk_angle_range == -1
    _, poses = _reachable_poses(1000, 71)
    for dtype in (np.float64, np.float32):
        s = _angles(1000, 72).astype(dtype)
        out, st, it, err = eng.dls_pose_refine(poses, s, max_iter=0, return_iters=True, return_error=True)
        assert _same_bits(out, s) and (it == 0).all() and st.sum_iterations == 0
        want = np_pose_refine(fk, poses, s.astype(np.float64), ONES, 0.1, TOL, 0)[2]
        assert _same_bits(err, want.astype(dtype))


def test_device_outputs_stay_inside_guard_bands():
    import torch
    eng = _eng()
    GUARD = 64
    pattern = {torch.float32: 0x7FC0BEEF, torch.float64: 0x7FF8DEADBEEF0001}
    _, all_poses = _reachable_poses(129, 2000)
    for td, npd in ((torch.float32, np.float32), (torch.float64, np.float64)):
        ubits = torch.int32 if td == torch.float32 else torch.int64
        item = np.dtype(npd).itemsize
        for n in range(1, 130):
            poses = torch.from_numpy(all_poses[:n].astype(npd)).cuda()
            seed = torch.from_numpy(_angles(n, 3000 + n).astype(npd)).cuda()
            ref = torch.empty((n, 4), dtype=td, device="cuda")
            ref_err = torch.empty(n, dtype=td, device="cuda")
            ref_it = torch.empty(n, dtype=torch.int32, device="cuda")
            eng.dls_pose_refine_device(poses, seed, ref, ref_it, ref_err)
            for off_bytes in (0, 4, 8, 12):
                if off_bytes % item:
                    continue
                off = GUARD + off_bytes // item
                ab = torch.full((4 * n + 2 * GUARD,), pattern[td], dtype=ubits, device="cuda").view(td)
                eb = torch.full((n + 2 * GUARD,), pattern[td], dtype=ubits, device="cuda").view(td)
                ib = torch.full((n + 2 * GUARD,), 0x5EED5EED, dtype=torch.int32, device="cuda")
                ib_off = GUARD + off_bytes // 4
                # the poses at an unaligned offset too
                pb = torch.zeros(16 * n + 4, dtype=td, device="cuda")
                p_off = off_bytes // item
                pb[p_off:p_off + 16 * n] = poses.reshape(-1)
                eng.dls_pose_refine_device(pb[p_off:p_off + 16 * n].view(n, 4, 4), seed,
                                           ab[off:off + 4 * n].view(n, 4), ib[ib_off:ib_off + n], eb[off:off + n])
                torch.cuda.synchronize()
                abits, ebits = ab.view(ubits), eb.view(ubits)
                for bits, inner in ((abits, 4 * n), (ebits, n)):
                    assert (bits[:off] == pattern[td]).all() and (bits[off + inner:] == pattern[td]).all(), (n, off)
                assert (ib[:ib_off] == 0x5EED5EED).all() and (ib[ib_off + n:] == 0x5EED5EED).all()
                assert torch.equal(ab[off:off + 4 * n].view(n, 4), ref) and torch.equal(eb[off:off + n], ref_err)
                assert torch.equal(ib[ib_off:ib_off + n], ref_it)


def test_side_stream_with_late_inputs_matches_a_plain_call():
    """Inputs that hold decoys until a ~30 ms sleep on the caller's side stream has passed (as test_gpu_streams.py
    does for the other entry points): the outputs and statistics equal a plain call's bit for bit."""
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    n = 4000
    _, poses = _reachable_poses(n, 81)
    real = [torch.from_numpy(poses).cuda(), torch.from_numpy(_angles(n, 82)).cuda()]
    decoy = [torch.roll(t, shifts=n // 3 + 1, dims=0).contiguous() for t in real]

    def launch(eng, p, s):
        it = torch.empty(n, dtype=torch.int32, device="cuda")
        err = torch.empty(n, dtype=s.dtype, device="cuda")
        eng.dls_pose_refine_device(p, s, s, iters=it, err=err)  # in place
        return s, it, err

    def counts(st):
        return (st.n_solved, st.sum_iterations, st.n_iter_capped, st.n_fk_error)

    with IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits) as eng:
        torch.cuda.synchronize()
        eng.stats_reset()
        want = [o.clone() for o in launch(eng, *[t.clone() for t in real])]
        torch.cuda.synchronize()
        st_want = eng.stats_fetch()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            eng.stats_reset_torch()
            bufs = [d.clone() for d in decoy]
            torch.cuda._sleep(50_000_000)
            for b, r in zip(bufs, real):
                b.copy_(r)
            got = [o.clone() for o in launch(eng, *bufs)]
            st_got = eng.stats_fetch_torch()
        side.synchronize()
        for w, g in zip(want, got):
            assert torch.equal(w.view(torch.int64 if w.dtype == torch.float64 else torch.int32),
                               g.view(torch.int64 if g.dtype == torch.float64 else torch.int32))
        assert counts(st_got) == counts(st_want)
        wrong = launch(eng, *[t.clone() for t in decoy])
        torch.cuda.synchronize()
        assert not torch.equal(wrong[0], want[0])


# ---- 7. the Python layer -------------------------------------------------------------------------------------------
def test_python_layer_shapes_and_messages():
    from inversekinematicsann_b200.robot.robot import OutOfRobotReachException
    ik = _ik()
    th, T = _reachable_poses(50, 91)
    seed = _angles(50, 92)
    # fkine_batch's T (a strided view) goes straight in
    T_view = ik.fkine.fkine_batch(th)[0]
    assert not T_view.flags.c_contiguous
    out = ik.refine_pose(T_view, seed.tolist())
    assert isinstance(out, list) and len(out) == 50 and all(isinstance(v, float) for v in out[0])
    assert ik.last_stats.n_solved == 50
    out, its, err = ik.refine_pose(T, seed.astype(np.float32), as_array=True, return_iterations=True,
                                   return_fk_error=True)
    assert out.dtype == np.float32 and its.dtype == np.int32 and err.dtype == np.float32 and out.shape == (50, 4)
    bad_T = T.copy()
    bad_T[9, :3, 3] = (1.0, 2.0, 7.0)
    bad_seed = seed.copy()
    bad_seed[3, 1] = -7.0
    with pytest.raises(OutOfRobotReachException) as exc:
        ik.refine_pose(bad_T, bad_seed)                  # limits first
    assert str(exc.value) == str(ik._limits_error([[1.0, 2.0, 7.0]], 0))
    assert "point [1.0, 2.0, 7.0] is out of manipulator reach area" in str(exc.value)
    with pytest.raises(OutOfRobotReachException) as exc:
        ik.refine_pose(T, bad_seed)
    assert str(exc.value) == ANGLE_MSG
    with pytest.raises(OutOfRobotReachException) as exc:
        ik.ikine_pose(bad_T)
    assert str(exc.value) == str(ik._limits_error([[1.0, 2.0, 7.0]], 0))
    out = ik.ikine_pose(T.tolist())
    assert isinstance(out, list) and len(out) == 50
    # refine_pose_device reports through the statistics instead, and refuses a strided pose tensor
    import torch
    eng = ik._engine()
    eng.stats_reset_torch()
    d = ik.refine_pose_device(torch.from_numpy(bad_T).cuda(), torch.from_numpy(bad_seed).cuda())
    st = eng.stats_fetch_torch()
    assert d.shape == (50, 4) and st.first_out_of_limits == 9 and st.first_fk_angle_range == 3
    eng.stats_reset_torch()
    chain = torch.from_numpy(ik.fkine.fkine_batch(th)[1]).cuda()
    with pytest.raises(ValueError, match="contiguous"):
        ik.refine_pose_device(chain[:, 3], torch.from_numpy(seed).cuda())


def test_ann_ikine_pose_and_refine_pose_device_after_ann_solve_device():
    import torch
    ann = _ik("ann")
    _, T = _reachable_poses(20_000, 101)
    out, its, err = ann.ikine_pose(T, as_array=True, return_iterations=True, return_fk_error=True)
    assert out.dtype == np.float64 and out.shape == (T.shape[0], 4) and its.shape == err.shape == (T.shape[0],)
    conv = err <= TOL
    assert conv.mean() >= ANN_ROUND_TRIP_BAR, conv.mean()
    _check_converged_with_the_oracle(T, out, conv)
    # the same chain by hand, with no host round trip between the network and the refinement
    eng = ann.ann._ensure_uploaded()
    d_T = torch.from_numpy(T).cuda()
    xyz = d_T[:, :3, 3].contiguous()
    pred = torch.empty((T.shape[0], 4), dtype=torch.float32, device="cuda")
    eng.ann_solve_device(xyz, pred, mode=ann.ann.mode)
    seed = pred.double()
    ann.refine_pose_device(d_T, seed, out=seed)
    assert _same_bits(seed.cpu().numpy(), out)
    from inversekinematicsann_b200.robot.robot import OutOfRobotReachException
    bad_T = T[:10].copy()
    bad_T[4, :3, 3] = (1.0, 2.0, 7.0)
    with pytest.raises(OutOfRobotReachException) as exc:
        ann.ikine_pose(bad_T)
    assert str(exc.value) == str(ann._limits_error([[1.0, 2.0, 7.0]], 0))
