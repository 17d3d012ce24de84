"""K1 (planar FABRIK + angle extraction) on the planes and axes where its angle extraction branches: the x = 0 face
of the workspace, targets with x < 0, the branch edges of the hand-written atan2 / acos tails and the z axis.

Every family goes through every entry point (`_solve`): float64 and float32 angle buffers, host and device calls,
batches of at most kFuseFkMaxRows = 1024 rows (fused FK-error epilogue) and larger ones, float32 inputs; a separate
test runs all of them once more with IKB_FABRIK_SPLIT=0.  The bars of each test are for the float64 buffer; a float32
buffer is held to the float64 buffer of the same rows within 1e-6 rad with identical iteration counts.

All rows are solved under workspace limits x in [-6, 6]: the limits only decide which rows are refused, and targets
with x < 0 are legal under such user limits."""
import os
import subprocess
import sys

import numpy as np
import pytest

import conftest as C

pytestmark = pytest.mark.gpu

TOL_F64_MODE = 1e-9     # rad, oracle parity of the float64 buffer (tests/test_gpu_fabrik.py)
TOL_F32_BUFFER = 1e-6   # rad, float32 buffer against the float64 buffer of the same rows (DESIGN 1)
TOL_THETA1 = 1e-14      # rad, theta_1 against np.arctan2 of the plane direction (DESIGN: atan2_unit is within 3e-15)
# theta_2..4 of a target with |x| < 1e-11 against the oracle at x = 1e-9 for the same (y, z): measured 2.7e-15 on a B200
# (x = +-0, the cube face, x = 1e-12 .. 5e-324 and the |x| < 1e-11 rows of the azimuth and branch-edge families).  The
# oracle's own spread is 0 between x = 1e-9 and 1e-11 and reaches 2.4e-5 towards x = 1e-6 (DESIGN 1); the parity bar
# applies.
TOL_CONTINUITY = TOL_F64_MODE
# targets within 1e-6 of the first joint S: both solvers amplify their rounding there (the reference's seed noise of
# 1e-16 against a target 1e-7 from S); measured 3.9e-8 on a B200
TOL_FOLDED = 1e-6
FUSE_MAX_ROWS = 1024    # capi.cu kFuseFkMaxRows
LIMITS = {'x': [-6, 6], 'y': [-6, 6], 'z': [-3, 6]}
ORACLE_LIMITS = np.array([-6.0, 6.0, -6.0, 6.0, -3.0, 6.0])
S = np.array([0.0, 0.0, 2.0])   # the arm's first joint


@pytest.fixture(scope="module")
def eng():
    from inversekinematicsann_b200.kinematics._shared import get_engine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    return get_engine(R.dh_matrix, R.links_lengths, LIMITS)


def _oracle(xyz):
    from oracle import c_oracle
    want = c_oracle.fabrik_ikine(xyz, limits=ORACLE_LIMITS)
    assert want["first_bad"] == -1
    return want


def _host(eng, xyz, dt):
    a, st, it, _ = eng.fabrik_solve(xyz, out_dtype=dt, return_iters=True, return_fk_error=True)
    return a, it, st


def _solve(eng, xyz):
    """Solve `xyz` through every entry point and check that they agree; returns the float64 angles, the float32 angles
    and the iteration counts."""
    import torch
    n = len(xyz)
    # more than kFuseFkMaxRows rows (K3 computes the error after the solve), repeated if the family is smaller
    big = np.tile(xyz, (-(-(FUSE_MAX_ROWS + 1) // n), 1))
    out = {}
    for dt, tdt in ((np.float64, torch.float64), (np.float32, torch.float32)):
        a, it, _ = _host(eng, big, dt)
        name = np.dtype(dt).name
        for r in range(n, len(big), n):   # the repeats of a small family are solved alike
            assert np.array_equal(a[r:r + n], a[:min(n, len(big) - r)], equal_nan=True), name
        a, it = a[:n], it[:n]
        fused = [_host(eng, xyz[i:i + FUSE_MAX_ROWS], dt) for i in range(0, n, FUSE_MAX_ROWS)]
        assert np.array_equal(np.concatenate([f[0] for f in fused]), a, equal_nan=True), f"{name}: fused epilogue"
        assert np.array_equal(np.concatenate([f[1] for f in fused]), it), f"{name}: fused epilogue iterations"
        x32 = xyz.astype(np.float32)   # float32 inputs reach the kernel as the same numbers as their float64 values
        assert np.array_equal(_host(eng, x32, dt)[0], _host(eng, x32.astype(np.float64), dt)[0], equal_nan=True), \
            f"{name}: float32 inputs"
        xd = torch.from_numpy(xyz).cuda()
        ad = torch.empty((n, 4), dtype=tdt, device="cuda")
        itd = torch.empty(n, dtype=torch.int32, device="cuda")
        eng.fabrik_solve_device(xd, ad, iters=itd, fk_err=torch.empty(n, dtype=tdt, device="cuda"))
        assert np.array_equal(ad.cpu().numpy(), a, equal_nan=True), f"{name}: device entry point"
        assert np.array_equal(itd.cpu().numpy(), it), f"{name}: device entry point iterations"
        out[name] = (a, it)
    a64, it64 = out["float64"]
    a32, it32 = out["float32"]
    assert np.array_equal(it32, it64)
    fin = np.isfinite(a64).all(axis=1)
    assert np.array_equal(fin, np.isfinite(a32).all(axis=1))
    d32 = np.abs(a32[fin].astype(np.float64) - a64[fin]).max(initial=0.0)
    print(f"  float32 buffer against float64 buffer: max {d32:.2e} rad over {fin.sum()} rows")
    assert d32 <= TOL_F32_BUFFER, f"float32 buffer {d32:.3e} rad from the float64 buffer"
    return a64, a32, it64


def _wrap(d):
    return (d + np.pi) % (2 * np.pi) - np.pi


def _parity(a, it, xyz, what, theta1_mod_2pi_at_pi=False, tol=TOL_F64_MODE):
    """Oracle parity on rows the reference solves without an exception: 1e-9 rad, identical iteration counts.  Rows with
    |x| < 1e-11 (where the reference follows seed noise) are held to the continuity bar instead."""
    noisy = np.abs(xyz[:, 0]) < 1e-11
    if noisy.any():
        _continuity(a[noisy], it[noisy], xyz[noisy], f"{what}, |x| < 1e-11")
    a, it, xyz = a[~noisy], it[~noisy], xyz[~noisy]
    want = _oracle(xyz)
    ok = want["status"] == 0
    assert np.array_equal(it[ok], want["iters"][ok]), f"{what}: iteration counts differ from the oracle"
    d = np.abs(a[ok] - want["angles"][ok])
    if theta1_mod_2pi_at_pi:  # the reference picks the sign of theta_1 = +-pi from seed noise
        at_pi = np.abs(np.abs(want["angles"][ok, 0]) - np.pi) <= TOL_F64_MODE
        d[at_pi, 0] = np.abs(_wrap(a[ok, 0][at_pi] - want["angles"][ok, 0][at_pi]))
    print(f"  {what}: oracle parity max {d.max(axis=0)} over {ok.sum()} rows ({(~ok).sum()} oracle exceptions)")
    for j in range(4):
        w = int(np.argmax(d[:, j]))
        assert d[w, j] <= tol, f"{what}: theta_{j + 1} {d[w, j]:.3e} rad from the oracle at {xyz[ok][w]}"


def _continuity(a, it, xyz, what):
    """Targets with |x| < 1e-11: the reference's elbow branch follows seed noise there (DESIGN 1), so theta_2..4 and the
    iteration count are held to the oracle at x = 1e-9 for the same (y, z)."""
    moved = xyz.copy()
    moved[:, 0] = 1e-9
    want = _oracle(moved)
    assert (want["status"] == 0).all()
    assert np.array_equal(it, want["iters"]), f"{what}: iteration counts differ from the oracle at x = 1e-9"
    d = np.abs(a[:, 1:] - want["angles"][:, 1:])
    print(f"  {what}: theta_2..4 against the oracle at x = 1e-9: max {d.max(axis=0)}")
    for j in range(3):
        m = d[:, j].max()
        assert m <= TOL_CONTINUITY, \
            (f"{what}: theta_{j + 2} {m:.3e} rad from the oracle at x = 1e-9 for the same (y, z) "
             f"({(d[:, j] > TOL_CONTINUITY).sum()} of {len(d)} rows above {TOL_CONTINUITY:g})")


# ---- the families ------------------------------------------------------------------------------------------------
def _yz(rng, n):
    """(y, z) across the workspace, |y| >= 0.01 (the z axis has its own family)."""
    y = rng.uniform(0.01, 6.0, n) * rng.choice([-1.0, 1.0], n)
    return y, rng.uniform(-3.0, 6.0, n)


def _rows_x_zero(case):
    """x = +0 rows, then the same rows with x = -0.0."""
    if case == "random":
        y, z = _yz(np.random.RandomState(41), 20_000)
        xyz = np.stack([np.zeros_like(y), y, z], axis=1)
    else:  # the x = 0 face of a cube grid (made on the device, as a user makes it)
        from inversekinematicsann_b200.robot.position_generator import TrainingDataGenerator
        grid = TrainingDataGenerator.cube_device(0.25, 6, 12, 9, start=(0, -6, -3), dtype="float64").cpu().numpy()
        face = grid[grid[:, 0] == 0]
        assert len(face) == 48 * 36
        xyz = face[face[:, 1] != 0]   # the face's z-axis rows belong to the z-axis family
    neg = xyz.copy()
    neg[:, 0] = -0.0
    return np.concatenate([xyz, neg])


def _rows_tiny_x():
    """x = 10^-k for k = 3 .. 300 and two subnormals, each with the same 400 (y, z)."""
    y, z = _yz(np.random.RandomState(42), 400)
    xs = np.array([10.0 ** -k for k in range(3, 301)] + [1e-310, 5e-324])
    return np.stack([np.repeat(xs, len(y)), np.tile(y, len(xs)), np.tile(z, len(xs))], axis=1)


def _rows_negative_x():
    """A dense azimuth circle with the exact +-x and +-y axes and y = +-0 on the negative x axis, and a uniform sample
    of the half x < 0."""
    phi = np.linspace(-np.pi, np.pi, 3601)
    r, zz = np.meshgrid([0.5, 2.0, 3.7, 5.5], [-2.0, 0.5, 2.0, 4.5])
    r, zz = r.ravel(), zz.ravel()
    ring = np.stack([np.outer(r, np.cos(phi)), np.outer(r, np.sin(phi)), np.repeat(zz[:, None], len(phi), 1)], -1)
    axes = [np.stack([sx * r, sy * r, zz], 1) for sx, sy in ((1, 0), (-1, 0), (0, 1), (0, -1))]
    axes += [np.stack([-r, np.full_like(r, s), zz], 1) for s in (0.0, -0.0)]
    half = np.random.RandomState(43).rand(20_000, 3) * [6, 12, 9] + [-6, -6, -3]
    return np.concatenate([ring.reshape(-1, 3)] + axes + [half])


def _ulps(v, k):
    """v moved by k units in the last place (k may be negative)."""
    out = np.float64(v)
    for _ in range(abs(k)):
        out = np.nextafter(out, np.inf if k > 0 else -np.inf)
    return out


def _rows_tail_edges():
    """Azimuths where |uy| or |ux| of the plane direction is 1/2 (every 30 degrees, with the axes), each coordinate
    moved by up to 4 ulps; targets on the reach sphere |T - S| = 6 and up to 4 ulps of the radius either side (cosines at
    or next to +-1); folded targets next to S."""
    rows = []
    for deg in range(0, 360, 30):
        for rad in (1.0, 3.0, 5.5):
            x0, y0 = rad * np.cos(np.deg2rad(deg)), rad * np.sin(np.deg2rad(deg))
            for zc in (-2.0, 1.0, 2.0, 3.5, 5.0):
                rows += [(_ulps(x0, kx), _ulps(y0, ky), zc) for kx in range(-4, 5) for ky in range(-4, 5)]
    rng = np.random.RandomState(44)
    d = rng.randn(2 * 3000, 3)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    sphere = [S + d[:3000] * _ulps(6.0, k) for k in range(-4, 5)]
    folded = [S + d[3000:] * rho for rho in (1e-7, 1e-4, 1e-2, 0.1, 0.5, 2.0, 4.0)]
    xyz = np.concatenate([np.array(rows)] + sphere + folded)
    inside = (np.abs(xyz[:, :2]) <= 6).all(axis=1) & (xyz[:, 2] >= -3) & (xyz[:, 2] <= 6)
    return xyz[inside]


AXIS_OFFSETS = [(0.0, 0.0), (-0.0, 0.0), (0.0, -0.0), (-0.0, -0.0),   # the z axis with every signed zero
                (5e-324, 0.0), (0.0, -5e-324),                          # x^2 + y^2 underflows to 0: on the axis too
                (1e-15, -3e-16), (-1e-12, 0.0), (0.0, 1e-11), (-7.0710678118654757e-11, 7.0710678118654757e-11),
                (1e-10, 0.0), (0.0, -1e-10)]                             # x^2 + y^2 from 1e-30 to 1e-20


def _rows_axis():
    """The z axis and targets next to it, at z every 0.1 from -3 to 6 and 1e-9 and 1e-3 above and below the first
    joint S = (0, 0, 2) (S itself is a zero-length segment, checked on its own)."""
    z = np.concatenate([np.linspace(-3.0, 6.0, 91), [2.0 - 1e-9, 2.0 + 1e-9, 2.0 - 1e-3, 2.0 + 1e-3]])
    z = z[z != 2.0]
    return np.array([(ox, oy, zz) for ox, oy in AXIS_OFFSETS for zz in z]), len(z)


# ---- the tests ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["random", "cube_face"])
def test_x_zero_plane_is_continuous_with_x_positive(eng, case):
    """The x = 0 face of the workspace: theta_1 is +-pi/2 to the last bit, theta_2..4 and the iteration counts are those
    of the oracle 1e-9 away, and x = -0.0 gives the same bits as x = +0."""
    xyz = _rows_x_zero(case)
    a64, _, it = _solve(eng, xyz)
    n = len(xyz) // 2
    assert np.array_equal(a64[:n], a64[n:]) and np.array_equal(it[:n], it[n:]), "x = -0.0 differs from x = +0"
    assert np.array_equal(a64[:, 0], np.arctan2(xyz[:, 1], xyz[:, 0]))
    _continuity(a64, it, xyz, f"x = +-0 ({case})")


def test_tiny_x_sweep(eng):
    """Oracle parity down to x = 1e-11; below that the reference follows seed noise and the continuity bar applies."""
    xyz = _rows_tiny_x()
    a64, _, it = _solve(eng, xyz)
    d1 = np.abs(a64[:, 0] - np.arctan2(xyz[:, 1], xyz[:, 0])).max()
    print(f"  theta_1 against np.arctan2: max {d1:.2e}")
    assert d1 <= TOL_THETA1
    _parity(a64, it, xyz, "x = 10^-k")


def test_negative_x_full_azimuth(eng):
    """The ux < 0 branch of atan2_unit and the flip of theta_1, all around the z axis."""
    xyz = _rows_negative_x()
    a64, _, it = _solve(eng, xyz)
    _parity(a64, it, xyz, "x < 0 and the azimuth circle", theta1_mod_2pi_at_pi=True)
    neg_axis = (xyz[:, 0] < 0) & (xyz[:, 1] == 0)
    assert np.array_equal(a64[neg_axis, 0], np.where(np.signbit(xyz[neg_axis, 1]), -np.pi, np.pi))


def test_tail_branch_edges(eng):
    """The branch edges of atan2_unit / acos_fast and of their fp32 forms (float32 buffer, held to the float64 buffer of
    the same call in _solve: both tails see the same fp64 cosines)."""
    xyz = _rows_tail_edges()
    a64, a32, it = _solve(eng, xyz)
    close = np.linalg.norm(xyz - S, axis=1) < 1e-6
    _parity(a64[~close], it[~close], xyz[~close], "branch edges")
    _parity(a64[close], it[close], xyz[close], "folded 1e-7 from S", tol=TOL_FOLDED)
    ok = np.isfinite(a64).all(axis=1)
    d1 = np.abs(_wrap(a64[ok, 0] - np.arctan2(xyz[ok, 1], xyz[ok, 0])))
    turned = np.abs(d1 - np.pi) <= 1e-9   # an effector beyond the z axis turns theta_1 by pi (folded targets next to S)
    assert (np.hypot(xyz[ok][turned, 0], xyz[ok][turned, 1]) < 2e-3).all()
    d1 = np.where(turned, np.abs(d1 - np.pi), d1)
    fin = np.isfinite(a64).all(axis=1)
    d32 = np.abs(a32[fin].astype(np.float64) - a64[fin]).max(axis=0)
    print(f"  theta_1 against np.arctan2: max {d1.max():.2e} ({turned.sum()} rows turned by pi); float32 tail against "
          f"the float64 tail: max {d32} rad")
    assert d1.max() <= TOL_THETA1


def test_z_axis_and_near_axis(eng):
    """Targets on the z axis (and those whose x^2 + y^2 underflows to 0) use the +x plane (DESIGN 1): theta_1 in {0, -pi},
    every angle finite, the same bits for every signed zero.  Targets next to the axis have theta_1 the azimuth of their
    plane (turned by pi when the effector ends beyond the axis).  S = (0, 0, 2) itself is a zero-length segment: NaN
    angles and its row reported, ZeroDivisionError from ikine, as upstream.
    theta_2..4 are not held to a reference here: FABRIK is ill-conditioned on the axis.  The oracle changes its iteration
    count on 834 of these 1128 rows when they move 1e-9 along +x, and the kernel's rounding against the oracle's (exactly
    planar there, its seed atan2(0, 0) = 0 has no noise) moves theta_2..4 by up to 0.14 rad and 114 iteration counts
    (measured on a B200)."""
    xyz, nz = _rows_axis()
    a64, _, _ = _solve(eng, xyz)
    assert np.isfinite(a64).all()
    on_axis = xyz[:, 0] * xyz[:, 0] + xyz[:, 1] * xyz[:, 1] == 0
    assert on_axis.sum() == 6 * nz
    assert np.isin(a64[on_axis, 0], [0.0, -np.pi]).all()
    zeros = a64[:4 * nz].reshape(4, nz, 4)
    assert all(np.array_equal(zeros[0], zeros[i]) for i in range(1, 4)), "a signed zero changes the result"
    near = ~on_axis
    d1 = np.abs(_wrap(a64[near, 0] - np.arctan2(xyz[near, 1], xyz[near, 0])))
    d1 = np.minimum(d1, np.abs(d1 - np.pi))
    print(f"  theta_1 of the rows next to the axis: max {d1.max():.2e}")
    assert d1.max() <= TOL_THETA1
    pts = np.array([[1.0, 2.0, 3.0], [0.0, 0.0, 2.0], [0.0, 0.0, 2.5]])
    a, _, st = _host(eng, pts, np.float64)
    assert st.first_zero_division == 1 and np.isnan(a[1]).all() and np.isfinite(a[[0, 2]]).all()
    from inversekinematicsann_b200.kinematics.inverse import FabrikInverseKinematics
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    with pytest.raises(ZeroDivisionError):
        FabrikInverseKinematics(R.dh_matrix, R.links_lengths, LIMITS).ikine(pts)


def test_planes_split_switch_is_value_identical(eng, tmp_path):
    """Every family above once more without the lockstep path for out-of-reach targets (IKB_FABRIK_SPLIT=0, read once
    per process): the same bits in both buffers and the same iteration counts."""
    axis, _ = _rows_axis()
    xyz = np.concatenate([_rows_x_zero("random"), _rows_x_zero("cube_face"), _rows_tiny_x(), _rows_negative_x(),
                          _rows_tail_edges(), axis])
    a64, a32, it = _solve(eng, xyz)
    np.save(tmp_path / "xyz.npy", xyz)
    code = ("import sys, numpy as np; sys.path.insert(0, sys.argv[1]);"
            "from inversekinematicsann_b200.kinematics._shared import get_engine;"
            "from inversekinematicsann_b200.robot.robot import SixDOFRobot as R;"
            "e = get_engine(R.dh_matrix, R.links_lengths, {'x': [-6, 6], 'y': [-6, 6], 'z': [-3, 6]});"
            "xyz = np.load(sys.argv[2]);"
            "a, _, it = e.fabrik_solve(xyz, out_dtype=np.float64, return_iters=True);"
            "a32, _ = e.fabrik_solve(xyz, out_dtype=np.float32);"
            "np.savez(sys.argv[3], a=a, it=it, a32=a32)")
    env = dict(os.environ, IKB_FABRIK_SPLIT="0")
    subprocess.run([sys.executable, "-c", code, C.ROOT, str(tmp_path / "xyz.npy"), str(tmp_path / "nosplit.npz")],
                   env=env, check=True, timeout=600)
    nosplit = np.load(tmp_path / "nosplit.npz")
    assert np.array_equal(it, nosplit["it"])
    assert np.array_equal(a64, nosplit["a"])
    assert np.array_equal(a32, nosplit["a32"])
    far = np.linalg.norm(xyz - S, axis=1) > 6.0011   # rows the split run gives to the lockstep path
    assert far.sum() > 10_000 and (it[far] == 100).all()
