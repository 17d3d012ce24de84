"""K3's fp32 paths over the whole guard range [-2 pi, 2 pi], and the angle guard of forward.py:23-25 on every FK path.

The fp32 FK kernels (fk.cu: the asynchronous-copy ring, the pair kernel, the generic kernel; the solvers' fused error
epilogues) use their own sine/cosine, ikb_sincos / ikb_sincos2 of csrc/fk_device.cuh: a Cody-Waite reduction by pi/2
with |k| <= 4 and quadrant selection.  Here every quadrant, every quadrant boundary (and the floats around it), signed
zeros, subnormals, the guard's edge float32(+-2 pi) and NaN / inf go through all three K3 paths, which must agree with
each other and with an fp64 restatement of the same DH chain on every row.

The guard rejects |theta| > 2 pi with theta widened to fp64 (the reference compares Python floats).  float32(2 pi) =
6.2831854820... is above 2 pi, so it is rejected on every path and in either buffer dtype."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TWO_PI = 2 * np.pi
F32_2PI = np.float32(TWO_PI)                          # 6.2831854820251465 > 2 pi: outside the guard
F32_BELOW_2PI = np.nextafter(F32_2PI, np.float32(0))  # 6.2831850051879883: the largest float32 inside

# ikb_sincos is within 1.2e-7 of sin / cos (the bound stated in fk_device.cuh); the probe reads its results through
# exact arithmetic, so that bound applies as is.  Measured on one B200: 8.3e-8 (sine), 9.1e-8 (cosine).
TOL_SINCOS = 1.2e-7
# FK position / error of the 2 m-link arm in fp32 against fp64 of the same float32 angles: each of the 4 joint angles
# contributes its sin/cos error (1.2e-7) through at most 6 m of lever arm and the chain rounds coordinates of up to
# 8 m (half an ulp: 2.4e-7) a few times; 2e-6 m covers the sum.  Measured on one B200: 1.2e-6 m.
TOL_POS = 2e-6


# ||pos - target|| adds its own rounding on top: the sum of squares and the root (sqrt.approx on the ring and pair paths,
# <= 2 ulp) -- 3 ulps of the error itself, up to 2.9e-6 m for the 16 m errors here.  Measured on one B200: 2.5e-6 m.
def tol_err(want_err):
    return TOL_POS + 3 * np.spacing(np.abs(want_err).astype(np.float32)).astype(np.float64)



# ---- fp64 reference (CPU) ------------------------------------------------------------------------------------------
def fk64(angles, dh):
    """Joint-4 origin of the DH chain T = prod Rz(theta_i) Tz(eps_i) Tx(a_i) Rx(alpha_i) (forward.py:62-94) in fp64,
    for the float32 (or float64) angles as given.  Rows the guard rejects (any |theta| > 2 pi, theta widened to fp64)
    come back NaN, like NaN angles do."""
    th = np.asarray(angles).astype(np.float64)
    n = th.shape[0]
    dh = np.asarray(dh, dtype=np.float64)
    R = np.broadcast_to(np.eye(3), (n, 3, 3)).copy()
    p = np.zeros((n, 3))
    with np.errstate(invalid="ignore"):
        for i in range(4):
            eps, a, al = dh[1, i], dh[2, i], dh[3, i]
            c, s = np.cos(th[:, i]), np.sin(th[:, i])
            ca, sa = np.cos(al), np.sin(al)
            p = p + np.einsum("nij,nj->ni", R, np.stack([a * c, a * s, np.full(n, eps)], axis=1))
            z = np.zeros(n)
            M = np.stack([np.stack([c, -s * ca, s * sa], 1), np.stack([s, c * ca, -c * sa], 1),
                          np.stack([z, z + sa, z + ca], 1)], axis=1)
            R = R @ M
    rejected = guard_rejects(th)
    p[rejected] = np.nan
    return p, rejected


def guard_rejects(angles):
    """forward.py:23-25: an angle outside [-2 pi, 2 pi] (compared in fp64; NaN is not rejected)."""
    with np.errstate(invalid="ignore"):
        return (np.abs(np.asarray(angles).astype(np.float64)) > TWO_PI).any(axis=1)


def first_rejected(angles):
    bad = np.flatnonzero(guard_rejects(angles))
    return int(bad[0]) if bad.size else -1


def _ulps_around(x, k=2):
    x = np.float32(x)
    out, up, dn = [x], x, x
    for _ in range(k):
        up, dn = np.nextafter(up, np.float32(np.inf)), np.nextafter(dn, np.float32(-np.inf))
        out += [up, dn]
    return out


def special_angles():
    """float32 angles where a bounded-range sine / cosine goes wrong: every quadrant boundary k pi / 2 (k = -4..4) and
    two ulps either side, signed zeros, subnormals and tiny angles, the guard edge +-2 pi and its neighbours, NaN and
    +-inf."""
    vals = []
    for k in range(-4, 5):
        vals += _ulps_around(k * np.pi / 2)
    vals += _ulps_around(F32_2PI) + _ulps_around(-F32_2PI)
    vals += [0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-39, 1.1754942e-38, 1e-30, -1e-20, 1e-10, -3e-8, 1e-4]
    vals += [np.nan, np.inf, -np.inf]
    return np.array(vals, dtype=np.float32)


def special_rows(rng):
    """One row per (special angle, joint): the special angle at that joint, ordinary angles at the others."""
    sp = special_angles()
    rows = rng.uniform(-3.0, 3.0, size=(4 * sp.size, 4)).astype(np.float32)
    for j in range(4):
        rows[j * sp.size:(j + 1) * sp.size, j] = sp
    return rows


def dense_angles(rng, n):
    return rng.uniform(-TWO_PI, TWO_PI, size=(n, 4)).astype(np.float32)


# ---- CPU-only checks -----------------------------------------------------------------------------------------------
def test_fp64_reference_matches_c_oracle():
    from oracle import c_oracle
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    rng = np.random.default_rng(1)
    ang = rng.uniform(-TWO_PI, TWO_PI, size=(4000, 4))
    _, want, _ = c_oracle.fk_positions(ang, dh=np.array(R.dh_matrix, dtype=np.float64))
    got, rejected = fk64(ang, R.dh_matrix)
    assert not rejected.any()
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)


def test_float_guard_constant_is_the_fp64_rule():
    """The float guard constant in fk_device.cuh is the largest float32 <= 2 pi, so that |theta| > it decides exactly as
    |(double)theta| > 2 pi does -- checked on every float32 within 64 ulps of +-2 pi."""
    src = open(os.path.join(ROOT, "inversekinematicsann_b200", "csrc", "fk_device.cuh")).read()
    const = np.float32(float(re.search(r"#define IKB_TWO_PI_F32 ([0-9.]+)f", src).group(1)))
    assert const == F32_BELOW_2PI and float(const) <= TWO_PI < float(np.nextafter(const, np.float32(7)))
    around = np.concatenate([np.array(_ulps_around(F32_2PI, 64), dtype=np.float32),
                             np.array(_ulps_around(-F32_2PI, 64), dtype=np.float32)])
    assert np.array_equal(np.abs(around) > const, np.abs(around.astype(np.float64)) > TWO_PI)


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _torch():
    import torch
    return torch


@pytest.fixture(scope="module")
def eng():
    from inversekinematicsann_b200.kinematics._shared import get_engine
    return get_engine()


@pytest.fixture(scope="module")
def dh():
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    return np.array(R.dh_matrix, dtype=np.float64)


def _num_sms():
    return _torch().cuda.get_device_properties(0).multi_processor_count


def _run_three_paths(eng, ang, tgt):
    """||FK - target|| of the same rows through the ring (+ pair kernel tail), the pair kernel alone (targets 8 bytes
    off 16-byte alignment) and the generic kernel (positions wanted); statistics of each call."""
    torch = _torch()
    n = ang.shape[0]
    a = torch.from_numpy(ang).cuda()
    t = torch.from_numpy(tgt).cuda()
    t_off = torch.empty(3 * n + 2, device="cuda")[2:].view(n, 3)
    t_off.copy_(t)
    assert t.data_ptr() % 16 == 0 and t_off.data_ptr() % 16 == 8
    res = {}
    for name, targets, want_pos in (("ring", t, False), ("pair", t_off, False), ("generic", t, True)):
        err = torch.full((n,), 12345.0, device="cuda")
        pos = torch.full((n, 3), 12345.0, device="cuda") if want_pos else None
        eng.stats_reset_torch()
        eng.fk_device(a, targets=targets, pos=pos, err=err)
        st = eng.stats_fetch_torch()
        res[name] = (err.cpu().numpy(), pos.cpu().numpy() if want_pos else None, st)
    return res


@pytest.mark.gpu
def test_k3_fp32_paths_over_the_whole_guard_range(eng, dh):
    """Dense uniform angles on [-2 pi, 2 pi] plus the special rows at the start, in the middle and in the ragged tail of
    a batch large enough for the ring (n >= 4 * SMs * 8 warps * 64 rows): the three paths against each other and every
    row against fp64 FK of the same float32 angles."""
    rng = np.random.default_rng(20)
    n = 4 * _num_sms() * 8 * 64 + 37                     # full ring trips + 37 rows for the pair kernel (odd: scalar tail)
    ang = dense_angles(rng, n)
    sp = special_rows(rng)
    m = sp.shape[0]
    for lo in (0, n // 2, n - m):
        ang[lo:lo + m] = sp
    tgt = rng.uniform(-8, 8, size=(n, 3)).astype(np.float32)
    want_pos, rejected = fk64(ang, dh)
    want_err = np.linalg.norm(want_pos - tgt, axis=1)
    nan_rows = np.isnan(want_err)
    res = _run_three_paths(eng, ang, tgt)
    e_ring, e_pair, e_gen = res["ring"][0], res["pair"][0], res["generic"][0]
    pos = res["generic"][1]
    # ring and pair kernel: same sincos2, same chain, same sqrt.approx -> the same bits, NaN rows included
    assert np.array_equal(e_ring.view(np.int32), e_pair.view(np.int32))
    # generic kernel: scalar sincos (bit-identical to sincos2) and the IEEE root instead of sqrt.approx (<= 1 ulp):
    # within 2 ulps of the ring's value; the scalar odd last row is the same code on every path
    for e in (e_ring, e_gen):
        assert np.array_equal(np.isnan(e), nan_rows)
    ok = ~nan_rows
    ulp = np.spacing(np.abs(e_gen[ok]))
    assert (np.abs(e_ring[ok] - e_gen[ok]) <= 2 * ulp).all()
    assert np.array_equal(e_ring[-1:], e_gen[-1:], equal_nan=True)   # (NaN payloads differ: the guard's vs sqrt's)
    d_pos = np.abs(pos[ok].astype(np.float64) - want_pos[ok]).max()
    d_err = max(np.abs(e.astype(np.float64)[ok] - want_err[ok]).max() for e in (e_ring, e_gen))
    print(f"n={n}: max |pos - fp64| {d_pos:.2e} m, max |err - fp64| {d_err:.2e} m, NaN rows {nan_rows.sum()}")
    assert d_pos <= TOL_POS
    for e in (e_ring, e_gen):
        assert (np.abs(e.astype(np.float64)[ok] - want_err[ok]) <= tol_err(want_err[ok])).all()
    assert np.isnan(pos[rejected]).all()                 # the guard blanks all three coordinates
    # statistics: the lowest rejected row, and sum / count of the finite per-row errors
    first = first_rejected(ang)
    assert first >= 0
    for name, (e, _, st) in res.items():
        assert st.first_fk_angle_range == first, name
        assert st.n_fk_error == int(ok.sum()), name
        want_sum = float(np.sum(e[ok], dtype=np.float64))
        assert abs(st.sum_fk_error - want_sum) <= 1e-6 * want_sum, name


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3, 64, 65, 127])
def test_k3_small_batches_take_the_pair_kernel(eng, dh, n):
    """Batches too small for the ring: pair kernel (error only) against the generic kernel and fp64, special rows
    included, and the odd last row through the pair kernel's scalar tail."""
    rng = np.random.default_rng(n)
    sp = special_rows(rng)
    ang = sp[rng.choice(sp.shape[0], n, replace=False)]
    tgt = rng.uniform(-8, 8, size=(n, 3)).astype(np.float32)
    want_pos, _ = fk64(ang, dh)
    want_err = np.linalg.norm(want_pos - tgt, axis=1)
    res = _run_three_paths(eng, ang, tgt)
    for name, (e, _, st) in res.items():
        assert np.array_equal(np.isnan(e), np.isnan(want_err)), name
        ok = ~np.isnan(want_err)
        assert (np.abs(e[ok].astype(np.float64) - want_err[ok]) <= tol_err(want_err[ok])).all(), name
        assert st.first_fk_angle_range == first_rejected(ang), name
        assert st.n_fk_error == int(ok.sum()), name


@pytest.mark.gpu
def test_ikb_sincos_against_fp64_sin_cos():
    """ikb_sincos read out exactly: an arm whose only link is a_1 = 1 along x (eps = alpha = 0, joints 2..4 at 0) has
    its joint-4 origin at (cos theta_1, sin theta_1, 0) -- the closed form multiplies by 1 and adds exact zeros."""
    torch = _torch()
    from inversekinematicsann_b200.engine import IkEngine
    probe = IkEngine([[0, 0, 0, 0], [0, 0, 0, 0], [1, 0, 0, 0], [0, 0, 0, 0]], [1, 1, 1, 1],
                     [-10, 10, -10, 10, -10, 10])
    try:
        x = np.linspace(-F32_BELOW_2PI, F32_BELOW_2PI, (1 << 20) + 1, dtype=np.float32)
        sp = special_angles()
        x = np.concatenate([x, sp[np.isfinite(sp) & (np.abs(sp.astype(np.float64)) <= TWO_PI)]])
        ang = np.zeros((x.size, 4), dtype=np.float32)
        ang[:, 0] = x
        pos = torch.empty(x.size, 3, device="cuda")
        probe.fk_device(torch.from_numpy(ang).cuda(), pos=pos)
        p = pos.cpu().numpy().astype(np.float64)
        xd = x.astype(np.float64)
        ds, dc = np.abs(p[:, 1] - np.sin(xd)), np.abs(p[:, 0] - np.cos(xd))
        print(f"ikb_sincos vs fp64: max |dsin| {ds.max():.2e} (at {x[ds.argmax()]!r}), "
              f"max |dcos| {dc.max():.2e} (at {x[dc.argmax()]!r})")
        assert ds.max() <= TOL_SINCOS and dc.max() <= TOL_SINCOS
        assert (p[:, 2] == 0).all()
        # tiny and subnormal angles: sin x == x, cos x == 1 exactly
        tiny = np.abs(xd) < 1e-8
        assert tiny.sum() >= 8 and (p[tiny, 1] == xd[tiny]).all() and (p[tiny, 0] == 1.0).all()
    finally:
        probe.close()


# ---- the angle guard on every path ---------------------------------------------------------------------------------
def _guard_rows(dtype):
    """Rows around the guard edge in one column each; float32(+-2 pi) is outside, the float just below is inside, and
    (in fp64 buffers) the fp64 2 pi itself is inside."""
    edge = [F32_2PI, -F32_2PI, F32_BELOW_2PI, -F32_BELOW_2PI, np.nextafter(F32_2PI, np.float32(7))]
    vals = np.array(edge, dtype=dtype)
    if dtype == np.float64:
        vals = np.concatenate([vals, [TWO_PI, -TWO_PI, np.nextafter(TWO_PI, 7.0)]])
    rows = []
    for v in vals:
        for j in range(4):
            r = np.full(4, 0.25, dtype=dtype)
            r[j] = v
            rows.append(r)
    return np.array(rows, dtype=dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_angle_guard_edge_on_every_fk_path(eng, dtype):
    """Which rows each path rejects, one edge row at a time behind ordinary rows: fk (host), fk_device on the ring, pair
    and generic kernels, fk_transforms (host, device) and ForwardKinematics.fkine_positions / fkine_batch must all follow
    the fp64 rule.  (Before the float guard constant was fixed, float32(+-2 pi) passed every fp32 K3 path and was
    rejected by fk_transforms.)"""
    torch = _torch()
    from inversekinematicsann_b200.kinematics.forward import ForwardKinematics
    from inversekinematicsann_b200.robot.robot import OutOfRobotReachException, SixDOFRobot as R
    fkin = ForwardKinematics(R.dh_matrix)
    edge = _guard_rows(dtype)
    rng = np.random.default_rng(5)
    n_big = 4 * _num_sms() * 8 * 64 + 6
    for k, row in enumerate(edge):
        want_reject = bool(guard_rejects(row[None])[0])
        for n in ((7, n_big) if k < 8 else (7,)):   # the large batch (ring + pair tail) for float32(+-2 pi)
            ang = rng.uniform(-3, 3, size=(n, 4)).astype(dtype)
            at = n - 3 if n == 7 else n // 3 + k
            ang[at] = row
            want_first = at if want_reject else -1
            tgt = rng.uniform(-8, 8, size=(n, 3)).astype(dtype)
            tag = (dtype.__name__, k, float(row[k % 4]), n)
            _, err, st = eng.fk(ang, tgt, want_pos=False)
            assert st.first_fk_angle_range == want_first and bool(np.isnan(err[at])) == want_reject, tag
            _, st = eng.fk_transforms(ang, what="joints")
            assert st.first_fk_angle_range == want_first, tag
            a, t = torch.from_numpy(ang).cuda(), torch.from_numpy(tgt).cuda()
            t_off = torch.empty(3 * n + 2, dtype=t.dtype, device="cuda")[2:].view(n, 3)
            t_off.copy_(t)
            for targets, pos in ((t, None), (t_off, None), (t, torch.empty(n, 3, dtype=a.dtype, device="cuda"))):
                e = torch.empty(n, dtype=a.dtype, device="cuda")
                eng.stats_reset_torch()
                eng.fk_device(a, targets=targets, pos=pos, err=e)
                st = eng.stats_fetch_torch()
                assert st.first_fk_angle_range == want_first and bool(torch.isnan(e[at]).item()) == want_reject, tag
                if pos is not None:
                    assert bool(torch.isnan(pos[at]).all().item()) == want_reject, tag
            out = torch.empty(n, 4, 4, 4, dtype=a.dtype, device="cuda")
            eng.stats_reset_torch()
            eng.fk_transforms_device(a, out)
            assert eng.stats_fetch_torch().first_fk_angle_range == want_first, tag
            if n == 7:
                for call in (fkin.fkine_positions, fkin.fkine_batch):
                    if want_reject:
                        with pytest.raises(OutOfRobotReachException):
                            call(ang)
                    else:
                        call(ang)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp16x3_ts", "fp16x3", "fp32"])
def test_angle_guard_edge_in_the_fused_ann_epilogue(mode):
    """The ANN solver's fused ||FK - target|| (fp16x3_ts: in the kernel's output stage; the other modes: K3 on the
    kernel's output).  A zero output scale makes every row's angles exactly float32(mean_y), so the guard edge can be
    put into the solver's own output: float32(+-2 pi) must give NaN, the float just below must not."""
    torch = _torch()
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    from oracle import np_oracle
    W, b = np_oracle.synthetic_mlp(seed=4, dims=[3, 64, 64, 4])
    eng = IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    try:
        rng = np.random.default_rng(6)
        xyz = rng.uniform([0, -6, -3], [6, 6, 6], size=(129, 3)).astype(np.float32)
        for j in range(4):
            for v in (F32_2PI, -F32_2PI, F32_BELOW_2PI, -F32_BELOW_2PI):
                mean_y = np.full(4, 0.25)
                mean_y[j] = float(v)
                eng.mlp_load(W, b, np_oracle.SHIPPED_MEAN_X, np_oracle.SHIPPED_SCALE_X, mean_y, np.zeros(4))
                want_reject = abs(float(v)) > TWO_PI
                ang, st, err = eng.ann_solve(xyz, mode=mode, return_fk_error=True)
                assert (ang == mean_y.astype(np.float32)).all()
                assert np.isnan(err).all() == want_reject and np.isnan(err).any() == want_reject, (j, v)
                assert st.n_fk_error == (0 if want_reject else xyz.shape[0])
                out = torch.empty(129, 4, device="cuda")
                e = torch.empty(129, device="cuda")
                eng.ann_solve_device(torch.from_numpy(xyz).cuda(), out, mode=mode, fk_err=e)
                assert np.array_equal(e.cpu().numpy(), err, equal_nan=True)
    finally:
        eng.close()
