"""Damped-least-squares refinement of joint angles onto position targets (InverseKinematics.refine / refine_device,
IkEngine.dls_refine / dls_refine_device, csrc/fk.cu dls_refine_kernel).

The kernel builds on the chain of fkine_batch and jacobian_batch, so a NumPy restatement of the operation order in
include/ikb200.h, iterated on the GPU's own joint_positions and jacobian_batch, reproduces every step bit for bit.
Independent checks: the C oracle's FK for converged rows and the geometric reach bound for targets out of reach."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TWISTED_DH = [[0, np.pi / 2, 0, 0], [2, 0.5, -0.25, 0.1], [0.3, 2, 1.5, 2.5], [np.pi / 2, 0.3, -0.2, 0.1]]
TABLES = ["robot", "twisted"]
ANGLE_MSG = "Forward Kinematics exception, robot joints angles limits are (-2pi, 2pi)"
SHOULDER = np.array([0.0, 0.0, 2.0])
TOL = 1e-9
DH_SEED = [0.0, np.pi / 2, 0.0, 0.0]


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


def _fabrik_ik():
    from inversekinematicsann_b200.kinematics.inverse import FabrikInverseKinematics
    R = _robot()
    return FabrikInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)


def _defaults():
    from inversekinematicsann_b200 import engine
    return engine.DLS_DAMPING, engine.DLS_MAX_ITER


def _same_bits(a, b):
    """Equal bit for bit, except that any NaN equals any NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    nan = np.isnan(a)
    u = {8: np.uint64, 4: np.uint32}[a.dtype.itemsize]
    return bool(np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(u), b[~nan].view(u)))


def _targets(n, seed, reach=True):
    """Targets in the workspace box: within 6 m of the shoulder (reach=True) or beyond 6.05 m (reach=False)."""
    rng = np.random.default_rng(seed)
    out = []
    while sum(len(o) for o in out) < n:
        p = rng.uniform((0.0, -6.0, -3.0), (6.0, 6.0, 6.0), size=(2 * n + 64, 3))
        d = np.linalg.norm(p - SHOULDER, axis=1)
        out.append(p[d < 5.999] if reach else p[d > 6.05])
    return np.ascontiguousarray(np.vstack(out)[:n])


def _angles(n, seed, lo=-np.pi, hi=np.pi):
    return np.random.default_rng(seed).uniform(lo, hi, size=(n, 4))


# ---- the NumPy restatement (operation order of include/ikb200.h) -------------------------------------------------
def np_refine(fk, xyz, seed, damping, tol, max_iter):
    """-> (angles, iters, err) in fp64, p_4 and Jv of every iterate from the GPU's joint_positions / jacobian_batch."""
    n = xyz.shape[0]
    th = np.array(np.broadcast_to(seed, (n, 4)), dtype=np.float64)
    iters = np.zeros(n, dtype=np.int32)
    err_out = np.full(n, np.nan)
    active = np.ones(n, dtype=bool)
    lam2 = damping * damping
    k = 0
    while active.any():
        idx = np.flatnonzero(active)
        t = th[idx]
        p = fk.joint_positions(t)[:, 3]
        J = fk.jacobian_batch(t, "position")
        e = xyz[idx] - p
        err = np.sqrt((e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2])
        done = (err <= tol) | (k == max_iter)
        err_out[idx[done]] = err[done]
        iters[idx[done]] = k
        active[idx[done]] = False
        go = ~done
        if not go.any():
            break
        J, e, t = J[go], e[go], t[go]
        A = np.empty((J.shape[0], 3, 3))
        for i in range(3):
            for j in range(3):
                A[:, i, j] = (J[:, i, 0] * J[:, j, 0] + J[:, i, 1] * J[:, j, 1]) + \
                             (J[:, i, 2] * J[:, j, 2] + J[:, i, 3] * J[:, j, 3])
        for i in range(3):
            A[:, i, i] = A[:, i, i] + lam2
        l10, l20 = A[:, 0, 1] / A[:, 0, 0], A[:, 0, 2] / A[:, 0, 0]
        d1 = A[:, 1, 1] - l10 * A[:, 0, 1]
        t12 = A[:, 1, 2] - l20 * A[:, 0, 1]
        l21 = t12 / d1
        d2 = (A[:, 2, 2] - l20 * A[:, 0, 2]) - l21 * t12
        z1 = e[:, 1] - l10 * e[:, 0]
        z2 = (e[:, 2] - l20 * e[:, 0]) - l21 * z1
        y2 = z2 / d2
        y1 = z1 / d1 - l21 * y2
        y0 = (e[:, 0] / A[:, 0, 0] - l10 * y1) - l20 * y2
        t = t + ((J[:, 0] * y0[:, None] + J[:, 1] * y1[:, None]) + J[:, 2] * y2[:, None])
        for r, c in zip(*np.nonzero(np.abs(t) > math.pi)):
            t[r, c] = math.remainder(t[r, c], 2 * math.pi)
        th[idx[go]] = t
        k += 1
    return th, iters, err_out


# ---- 1. step bits --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_iter", [0, 1, 2, 3])
@pytest.mark.parametrize("table", TABLES)
def test_step_bits_against_the_numpy_restatement(table, max_iter):
    """tol = 0: every row takes max_iter steps; seeds across [-2pi, 2pi] exercise the wrap."""
    eng, fk = _eng(table), _fk(table)
    n = 3000
    xyz = np.vstack([_targets(n // 2, 1), _targets(n - n // 2, 2, reach=False)])
    seed = np.vstack([_angles(n // 2, 3), _angles(n - n // 2, 4, -6.2, 6.2)])
    damping = _defaults()[0]
    out, st, iters, err = eng.dls_refine(xyz, seed, damping, 0.0, max_iter, return_iters=True, return_error=True)
    want, want_it, want_err = np_refine(fk, xyz, seed, damping, 0.0, max_iter)
    assert _same_bits(out, want) and np.array_equal(iters, want_it) and _same_bits(err, want_err)
    assert (iters == max_iter).all() and st.n_solved == n and st.sum_iterations == n * max_iter
    if max_iter == 0:
        assert _same_bits(out, seed)
    else:
        assert (np.abs(out) <= np.pi).all()
    # a second damping, with a tolerance that stops some rows early
    out, _, iters, err = eng.dls_refine(xyz, seed, 0.3, 0.05, max_iter, return_iters=True, return_error=True)
    want, want_it, want_err = np_refine(fk, xyz, seed, 0.3, 0.05, max_iter)
    assert _same_bits(out, want) and np.array_equal(iters, want_it) and _same_bits(err, want_err)


# ---- 2. convergence on reachable targets -------------------------------------------------------------------------
# Bars from the measurement (profiles/r06_dls_bench.json, damping sweep at the default damping, 2^20 rows per
# workload): every FABRIK- and ANN-seeded reachable row converged, within 23 and 41 steps.  The bar allows one row in
# 1e5.  The ANN branch: on these 1e5 targets the largest wrapped |theta_out - theta_seed| of a row measured 0.13 rad at
# the 99.9th percentile and 2.9 rad at most (the network lands within millimetres, a few 1e-4 rad, on almost all
# rows; the few it puts far from the target can be carried to another branch by the lightly damped first step).  The
# bars: 0.25 rad at the 99.9th percentile, 3 rad at most.
FABRIK_CONVERGED_BAR = 1 - 1e-5
ANN_CONVERGED_BAR = 1 - 1e-5
ANN_BRANCH_BOUND = 3.0
ANN_BRANCH_P999 = 0.25
# Seeds at a singular pose: the broadcast DH seed row converged on all but 1e-6 of 2^20 rows within 256 steps and on
# 99.9 % within 56; at the default max_iter the bar is 99.9 %.
SINGULAR_CONVERGED_BAR = 0.999


def _check_converged_with_the_oracle(xyz, out, err, conv):
    from oracle import c_oracle
    st, pos, _ = c_oracle.fk_positions(out[conv], dh=np.asarray(_robot().dh_matrix, dtype=np.float64))
    assert st == 0
    d = np.linalg.norm(pos - xyz[conv], axis=1)
    assert d.max() <= TOL + 1e-12, d.max()
    assert (err[conv] <= TOL).all()


def test_fabrik_seeded_convergence():
    ik = _fabrik_ik()
    xyz = _targets(100_000, 11)
    seed = ik.ikine(xyz, as_array=True)
    out, iters, err = ik.refine(xyz, seed, as_array=True, return_iterations=True, return_fk_error=True)
    conv = err <= TOL
    assert conv.mean() >= FABRIK_CONVERGED_BAR, conv.mean()
    _check_converged_with_the_oracle(xyz, out, err, conv)
    st = ik.last_stats
    assert st.n_solved == xyz.shape[0] and st.n_iter_capped == int((~conv).sum())
    assert st.sum_iterations == int(iters.sum()) and (iters[~conv] == _defaults()[1]).all()


def test_ann_seeded_convergence_stays_on_the_seed_branch():
    import os
    from inversekinematicsann_b200.kinematics.inverse import AnnInverseKinematics
    R = _robot()
    ann = AnnInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ann.load_model(os.path.join(root, "models", "roboarm_b200_r01.h5"))
    xyz = _targets(100_000, 12)
    seed = ann.ikine(xyz, as_array=True).astype(np.float64)
    out, iters, err = ann.refine(xyz, seed, as_array=True, return_iterations=True, return_fk_error=True)
    conv = err <= TOL
    assert conv.mean() >= ANN_CONVERGED_BAR, conv.mean()
    _check_converged_with_the_oracle(xyz, out, err, conv)
    moved = np.abs(np.vectorize(math.remainder)(out[conv] - seed[conv], 2 * math.pi))
    p999 = np.percentile(moved.max(axis=1), 99.9)
    assert moved.max() <= ANN_BRANCH_BOUND and p999 <= ANN_BRANCH_P999, (moved.max(), p999)
    # float32 seeds refine too, onto a float32 result
    out32 = ann.refine(xyz[:1000], seed[:1000].astype(np.float32), as_array=True)
    assert out32.dtype == np.float32


# ---- 3. out of reach -----------------------------------------------------------------------------------------------
def test_out_of_reach_runs_to_max_iter():
    ik = _fabrik_ik()
    xyz = _targets(20_000, 13, reach=False)
    seed = ik.ikine(xyz, as_array=True)
    max_iter = _defaults()[1]
    out, iters, err = ik.refine(xyz, seed, as_array=True, return_iterations=True, return_fk_error=True)
    assert (err > TOL).all() and (iters == max_iter).all()
    assert np.isfinite(out).all() and (np.abs(out) <= np.pi).all()
    bound = np.linalg.norm(xyz - SHOULDER, axis=1) - 6.0
    assert (err >= bound - 1e-12).all()
    st = ik.last_stats
    assert st.n_iter_capped == xyz.shape[0] and st.sum_iterations == xyz.shape[0] * max_iter


# ---- 4. singular seeds ---------------------------------------------------------------------------------------------
def test_singular_seeds_converge():
    """The DH seed row (the arm straight up) and stretched arms make Jv rank-deficient; damping keeps the step
    finite and the targets are still reached."""
    eng = _eng()
    xyz = _targets(20_000, 14)
    rng = np.random.default_rng(15)
    stretched = np.zeros((xyz.shape[0], 4))
    stretched[:, :2] = rng.uniform(-np.pi, np.pi, size=(xyz.shape[0], 2))
    _, w, _ = eng.jacobian(np.vstack([DH_SEED, stretched[:100]]), None, manipulability=True)
    assert w.max() <= 1e-12
    for seed in (np.array(DH_SEED), stretched):
        out, st, iters, err = eng.dls_refine(xyz, seed, return_iters=True, return_error=True)
        conv = err <= TOL
        assert np.isfinite(out).all() and np.isfinite(err).all()
        assert conv.mean() >= SINGULAR_CONVERGED_BAR, (conv.mean(), np.percentile(iters, 99.9))
        assert st.n_iter_capped == int((~conv).sum())


# ---- 5. float32 ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", TABLES)
def test_float32_is_the_float64_run_rounded_once(table):
    eng = _eng(table)
    xyz = _targets(20_000, 16)
    s32 = _angles(xyz.shape[0], 17).astype(np.float32)
    for tol in (TOL, 1e-4):
        o32, _, i32, e32 = eng.dls_refine(xyz, s32, tol=tol, return_iters=True, return_error=True)
        o64, _, i64, e64 = eng.dls_refine(xyz, s32.astype(np.float64), tol=tol, return_iters=True,
                                          return_error=True)
        assert o32.dtype == np.float32 and e32.dtype == np.float32
        assert _same_bits(o32, o64.astype(np.float32)) and _same_bits(e32, e64.astype(np.float32))
        assert np.array_equal(i32, i64)
    # float32 targets are widened exactly
    x32 = xyz.astype(np.float32)
    a, _ = eng.dls_refine(x32, s32)
    b, _ = eng.dls_refine(x32.astype(np.float64), s32)
    assert _same_bits(a, b)


# ---- 6. batch independence -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", TABLES)
def test_batch_independence(table):
    import torch
    eng = _eng(table)
    big_n = 2 * torch.cuda.get_device_properties(0).multi_processor_count * 64 * 4 + 17  # several refill rounds
    xyz = np.vstack([_targets(big_n - big_n // 4, 21), _targets(big_n // 4, 22, reach=False)])
    seed = _angles(big_n, 23)
    ref, _, ref_it, ref_err = eng.dls_refine(xyz, seed, return_iters=True, return_error=True)
    rng = np.random.default_rng(24)
    sizes = list(range(1, 130)) + [big_n // 2 - 1, big_n // 2, big_n // 2 + 1, big_n]
    for n in sizes:
        sel = rng.choice(big_n, size=n, replace=False)
        out, _, it, err = eng.dls_refine(xyz[sel], seed[sel], return_iters=True, return_error=True)
        assert _same_bits(out, ref[sel]) and np.array_equal(it, ref_it[sel]) and _same_bits(err, ref_err[sel]), n
    # one broadcast seed is the same seed repeated n times
    one = np.array([0.3, 1.0, -0.5, 0.2])
    a, _ = eng.dls_refine(xyz, one)
    b, _ = eng.dls_refine(xyz, np.tile(one, (big_n, 1)))
    assert _same_bits(a, b)
    # in place equals out of place, on the host and on the device
    s = seed.copy()
    got, _ = eng.dls_refine(xyz, s, out=s)
    assert got is s and _same_bits(s, ref)
    d_xyz, d_s = torch.from_numpy(xyz).cuda(), torch.from_numpy(seed).cuda()
    eng.dls_refine_device(d_xyz, d_s, d_s)
    torch.cuda.synchronize()
    assert _same_bits(d_s.cpu().numpy(), ref)


# ---- 7. host and device --------------------------------------------------------------------------------------------
def _slot_rows(n):
    # capi.cu ensure_slots: the next power of two >= n, at least 1024, at most 4 Mi
    want = 1024
    while want < n and want < 1 << 22:
        want <<= 1
    return want


def test_host_chunks_equal_the_device_path():
    """A fresh engine, so that its staging slots are sized by this call alone.  Chunks: 3 S / 4 rows with the
    errors, S without (include/ikb200.h)."""
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    n = 6_500_000
    xyz = _targets(n, 31)
    seed = np.array(DH_SEED)
    S = _slot_rows(n)
    with IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits) as eng:
        for want_err in (True, False):
            chunks = -(-n // (3 * S // 4 if want_err else S))
            before = eng.launch_count
            res = eng.dls_refine(xyz, seed, return_iters=True, return_error=want_err)
            assert eng.launch_count - before == chunks and chunks >= 2
            host, st, it = res[0], res[1], res[2]
            assert st.n_solved == n and st.first_out_of_limits == -1 and st.first_fk_angle_range == -1
            d_out = torch.empty((n, 4), dtype=torch.float64, device="cuda")
            d_it = torch.empty(n, dtype=torch.int32, device="cuda")
            d_err = torch.empty(n, dtype=torch.float64, device="cuda")
            before = eng.launch_count
            eng.dls_refine_device(torch.from_numpy(xyz).cuda(), torch.from_numpy(seed).cuda(), d_out, d_it, d_err)
            torch.cuda.synchronize()
            assert eng.launch_count - before == 1
            assert _same_bits(d_out.cpu().numpy(), host) and np.array_equal(d_it.cpu().numpy(), it)
            if want_err:
                assert _same_bits(d_err.cpu().numpy(), res[3])
        before = eng.launch_count
        out, st = eng.dls_refine(np.empty((0, 3)), np.empty((0, 4)))
        assert out.shape == (0, 4) and st.n_solved == 0
        eng.dls_refine_device(torch.empty((0, 3), dtype=torch.float64, device="cuda"),
                              torch.empty((0, 4), dtype=torch.float64, device="cuda"),
                              torch.empty((0, 4), dtype=torch.float64, device="cuda"))
        assert eng.launch_count == before


# ---- 8. guards -----------------------------------------------------------------------------------------------------
def test_guards_lowest_rows_across_host_chunks():
    from inversekinematicsann_b200.engine import IkEngine
    R = _robot()
    n = 1_000_000
    S = _slot_rows(n)
    chunk = 3 * S // 4
    assert n > chunk + 100
    xyz = _targets(n, 41)
    seed = _angles(n, 42)
    with IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits) as eng:
        clean, _, _, clean_err = eng.dls_refine(xyz, seed, return_iters=True, return_error=True)
        xyz[chunk + 7] = (7.0, 0.0, 0.0)           # out of the box, after the first chunk boundary
        xyz[chunk - 2] = (1.0, 1.0, -3.5)          # the lowest, just before it
        seed[chunk + 3, 2] = 6.5                   # out of the FK range, just after it
        seed[chunk + 100, 0] = -np.inf
        out, st, _, err = eng.dls_refine(xyz, seed, return_iters=True, return_error=True)
        assert st.first_out_of_limits == chunk - 2 and st.first_fk_angle_range == chunk + 3
        keep = np.ones(n, dtype=bool)
        keep[[chunk + 7, chunk - 2, chunk + 3, chunk + 100]] = False
        assert _same_bits(out[keep], clean[keep]) and _same_bits(err[keep], clean_err[keep])
        assert np.isfinite(out[[chunk + 7, chunk - 2, chunk + 3]]).all()   # still computed and written
        assert np.isnan(out[chunk + 100]).any()
        # float32 seeds are tested after widening: float32(2 pi) is outside, the float below it inside
        s32 = seed[:3].astype(np.float32)
        s32[1, 1] = np.float32(2 * np.pi)
        s32[0, 3] = np.nextafter(np.float32(2 * np.pi), np.float32(0))
        _, st = eng.dls_refine(xyz[:3], s32)
        assert st.first_fk_angle_range == 1


def test_python_layer_raises_the_reference_messages():
    from inversekinematicsann_b200.robot.robot import OutOfRobotReachException
    ik = _fabrik_ik()
    xyz = _targets(50, 51)
    seed = _angles(50, 52)
    bad_xyz = xyz.tolist()
    bad_xyz[9] = [1, 2, 7]
    bad_seed = seed.copy()
    bad_seed[3, 1] = -7.0
    with pytest.raises(OutOfRobotReachException) as exc:
        ik.refine(bad_xyz, seed)
    assert str(exc.value) == str(ik._limits_error(bad_xyz, 9))
    with pytest.raises(OutOfRobotReachException) as exc:
        ik.refine(bad_xyz, bad_seed)                    # limits first
    assert str(exc.value) == str(ik._limits_error(bad_xyz, 9))
    with pytest.raises(OutOfRobotReachException) as exc:
        ik.refine(xyz, bad_seed)
    assert str(exc.value) == ANGLE_MSG
    out = ik.refine(xyz.tolist(), seed.tolist())
    assert isinstance(out, list) and len(out) == 50 and all(isinstance(v, float) for v in out[0])
    assert ik.last_stats.n_solved == 50
    # refine_device reports through the statistics instead
    import torch
    eng = ik._engine()
    eng.stats_reset_torch()
    d = ik.refine_device(torch.from_numpy(np.array(bad_xyz)).cuda(), torch.from_numpy(bad_seed).cuda())
    st = eng.stats_fetch_torch()
    assert d.shape == (50, 4) and st.first_out_of_limits == 9 and st.first_fk_angle_range == 3
    eng.stats_reset_torch()


def test_device_outputs_stay_inside_guard_bands():
    import torch
    eng = _eng()
    GUARD = 64
    pattern = {torch.float32: 0x7FC0BEEF, torch.float64: 0x7FF8DEADBEEF0001}
    for td, npd in ((torch.float32, np.float32), (torch.float64, np.float64)):
        ubits = torch.int32 if td == torch.float32 else torch.int64
        item = np.dtype(npd).itemsize
        for n in list(range(1, 130)):
            xyz = torch.from_numpy(_targets(n, 2000 + n)).cuda()
            seed = torch.from_numpy(_angles(n, 3000 + n).astype(npd)).cuda()
            ref = torch.empty((n, 4), dtype=td, device="cuda")
            ref_err = torch.empty(n, dtype=td, device="cuda")
            ref_it = torch.empty(n, dtype=torch.int32, device="cuda")
            eng.dls_refine_device(xyz, seed, ref, ref_it, ref_err)
            for off_bytes in (0, 4, 8, 12):
                if off_bytes % item:
                    continue
                off = GUARD + off_bytes // item
                ab = torch.full((4 * n + 2 * GUARD,), pattern[td], dtype=ubits, device="cuda").view(td)
                eb = torch.full((n + 2 * GUARD,), pattern[td], dtype=ubits, device="cuda").view(td)
                ib = torch.full((n + 2 * GUARD,), 0x5EED5EED, dtype=torch.int32, device="cuda")
                ib_off = GUARD + off_bytes // 4
                eng.dls_refine_device(xyz, seed, ab[off:off + 4 * n].view(n, 4), ib[ib_off:ib_off + n],
                                      eb[off:off + n])
                torch.cuda.synchronize()
                abits, ebits = ab.view(ubits), eb.view(ubits)
                for bits, inner in ((abits, 4 * n), (ebits, n)):
                    assert (bits[:off] == pattern[td]).all() and (bits[off + inner:] == pattern[td]).all(), (n, off)
                assert (ib[:ib_off] == 0x5EED5EED).all() and (ib[ib_off + n:] == 0x5EED5EED).all()
                assert torch.equal(ab[off:off + 4 * n].view(n, 4), ref) and torch.equal(eb[off:off + n], ref_err)
                assert torch.equal(ib[ib_off:ib_off + n], ref_it)


def test_nan_rows_are_not_converged():
    eng = _eng()
    xyz = _targets(8, 61)
    seed = _angles(8, 62)
    xyz[2, 1] = np.nan
    seed[5, 3] = np.nan
    max_iter = 5
    out, st, it, err = eng.dls_refine(xyz, seed, max_iter=max_iter, return_iters=True, return_error=True)
    for r in (2, 5):
        assert np.isnan(out[r]).any() and np.isnan(err[r]) and it[r] == max_iter
    ok = np.ones(8, dtype=bool)
    ok[[2, 5]] = False
    assert np.isfinite(out[ok]).all() and np.isfinite(err[ok]).all()
    assert st.n_iter_capped == 2 + int((err[ok] > TOL).sum()) and st.n_fk_error == 6
    assert st.first_out_of_limits == -1
    assert st.first_fk_angle_range == -1


# ---- 9. max_iter = 0 -----------------------------------------------------------------------------------------------
def test_max_iter_zero_returns_the_seeds_and_their_errors():
    eng, fk = _eng(), _fk()
    xyz = _targets(1000, 71)
    for dtype in (np.float64, np.float32):
        seed = _angles(1000, 72).astype(dtype)
        out, st, it, err = eng.dls_refine(xyz, seed, max_iter=0, return_iters=True, return_error=True)
        assert _same_bits(out, seed) and (it == 0).all() and st.sum_iterations == 0
        _, _, want_err = np_refine(fk, xyz, seed.astype(np.float64), 0.05, TOL, 0)
        assert _same_bits(err, want_err.astype(dtype))
