"""The CPU oracle against (a) the golden vectors of the reference's own tests, (b) fixtures produced
by the unmodified reference (tools/make_golden.py), (c) the live reference when it is mounted."""
import numpy as np
import pytest

import conftest as C
from oracle import c_oracle, np_oracle, ref_import


def test_reference_inverse_unit_goldens():
    r = c_oracle.fabrik_ikine(C.REF_INVERSE_UNIT_POINTS)
    assert r["first_bad"] == -1
    np.testing.assert_almost_equal(r["angles"], C.REF_INVERSE_UNIT_FABRIK, decimal=6)
    # stronger than upstream's decimal=6: the restatement is bit-faithful
    np.testing.assert_allclose(r["angles"], C.REF_INVERSE_UNIT_FABRIK, rtol=0, atol=1e-14)


def test_reference_out_of_reach_golden():
    r = c_oracle.fabrik_ikine(C.REF_INVERSE_UNIT_OUT_OF_REACH)
    assert r["first_bad"] == 1  # z = -3.123 < -3 (inverse_unit.py:33)
    assert c_oracle.check_limits([[0, 0, 0], [6, 6, 6], [6, -6, -3]]) == -1  # inclusive bounds
    assert c_oracle.check_limits([[np.nan, 1, 1]]) == -1  # NaN passes (comparisons are False)
    assert c_oracle.check_limits([[1, 1, 1], [-1e-9, 0, 0]]) == 1


def test_reference_fabrik_unit_golden():
    st, chain = c_oracle.fk_chain(c_oracle.DH[0])
    init = chain[:, :3, 3]
    st, out, iters = c_oracle.fabrik_calculate(init, [1, 2, 3])
    assert st == 0
    np.testing.assert_array_almost_equal(out[3], C.REF_FABRIK_UNIT_EFFECTOR)  # upstream's assertion
    # upstream lists the intermediate joints too (fabrik_unit.py:25-27) but never asserts them, and the
    # live reference no longer produces them (they are not even coplanar with the z axis and the
    # target); only the start joint and the effector are pinned here.
    np.testing.assert_allclose(out[0], C.REF_FABRIK_UNIT_CHAIN[0], atol=1e-15)
    assert iters == 2


def test_reference_forward_unit_goldens():
    for ang, dest in zip(C.REF_FORWARD_UNIT_ANGLES, C.REF_FORWARD_UNIT_POINTS):
        st, chain = c_oracle.fk_chain(ang)
        assert st == 0
        np.testing.assert_array_almost_equal(dest, chain[3, :3, 3], decimal=4)
    st, _ = c_oracle.fk_chain([7.0, 0, 0, 0])  # > 2pi -> OutOfRobotReachException (forward.py:23)
    assert st == c_oracle.STATUS_FK_ANGLE_RANGE


def test_reference_point_unit_goldens():
    assert abs(c_oracle.distance([0, 0, 0], [-2.22, 3.123, 0.002]) - C.REF_POINT_UNIT_DISTANCE) < 5e-7
    st, mid = c_oracle.point_between([0, 0, 0], [-2.22, 3.123, 0.002])
    np.testing.assert_almost_equal(mid, np.array([-2.22, 3.123, 0.002]) / 2)
    st, _ = c_oracle.point_between([1, 1, 1], [1, 1, 1], 2.0)
    assert st == c_oracle.STATUS_ZERO_DIVISION  # point.py:40 ZeroDivisionError


@pytest.mark.parametrize("name", C.FABRIK_SETS)
def test_c_oracle_matches_reference_fixtures(golden_fabrik, name):
    xyz = golden_fabrik[f"{name}_xyz"]
    r = c_oracle.fabrik_ikine(xyz)
    assert r["first_bad"] == -1 and r["status"].max() == 0
    assert np.array_equal(r["iters"], golden_fabrik[f"{name}_iters"])
    np.testing.assert_allclose(r["angles"], golden_fabrik[f"{name}_angles"], rtol=0, atol=1e-12)


def test_c_oracle_fk_matches_reference_fixture(golden_fk):
    st, pos, err = c_oracle.fk_positions(golden_fk["angles"], targets=golden_fk["positions"])
    assert st == 0
    np.testing.assert_allclose(pos, golden_fk["positions"], rtol=0, atol=1e-13)
    assert err.max() < 1e-13
    st, chain = c_oracle.fk_chain(golden_fk["angles"][0])
    np.testing.assert_allclose(chain, golden_fk["chain0"], rtol=0, atol=1e-13)


def test_np_fabrik_cross_check(golden_fabrik):
    xyz = golden_fabrik["workspace_xyz"][:1500]
    ang, it = np_oracle.fabrik_ikine_np(xyz)
    assert np.array_equal(it, golden_fabrik["workspace_iters"][:1500])
    np.testing.assert_allclose(ang, golden_fabrik["workspace_angles"][:1500], rtol=0, atol=1e-9)


def test_degenerate_inputs_are_flagged():
    r = c_oracle.fabrik_ikine([[0, 0, 2.0]])  # target == start joint: ZeroDivisionError upstream
    assert r["status"][0] == c_oracle.STATUS_ZERO_DIVISION
    r = c_oracle.fabrik_ikine([[np.nan, 1, 1]])
    assert r["first_bad"] == -1 and np.isnan(r["angles"]).all() and r["iters"][0] == 1  # NaN > tol is False: one pass
    r = c_oracle.fabrik_ikine(np.zeros((0, 3)))
    assert r["first_bad"] == -1 and r["angles"].shape == (0, 4)


def test_generators_match_reference_fixtures(golden_generators):
    g = golden_generators
    np.random.seed(1234)
    np.testing.assert_array_equal(np_oracle.cube_random(648.0 / 1000, 6, 12, 9, (0, -6, -3)), g["cube_random"])
    np.random.seed(1234)
    lim = {"x": [0, 6], "y": [-6, 6], "z": [-3, 6]}
    np.testing.assert_array_equal(np_oracle.random_distribution_normal(500, lim, 0.35), g["normal035"])
    np.testing.assert_array_equal(np_oracle.circle(2, 50, (2, 0, 2)), g["circle"])
    np.testing.assert_array_equal(np_oracle.spring(50, 2, 3, 6), g["spring"])
    np.testing.assert_array_equal(np_oracle.cube(0.5, 2, 3, 1.5, (1, -1, 0)), g["cube"])


def test_mlp_oracle_fp32_vs_fp64():
    W, b = np_oracle.synthetic_mlp(seed=3)
    rng = np.random.default_rng(0)
    xyz = rng.uniform([0, -6, -3], [6, 6, 6], size=(256, 3))
    y32 = np_oracle.mlp_predict(xyz, W, b)
    y64 = np_oracle.mlp_predict(xyz, W, b, dtype=np.float64)
    assert y32.dtype == np.float32 and y32.shape == (256, 4)
    assert np.abs(y32 - y64).max() < 2e-5  # fp32 rounding noise through 13 layers
    assert np.std(y64, axis=0).min() > 1e-3  # the synthetic net is not constant


@pytest.mark.reference
@pytest.mark.skipif(not ref_import.available(), reason="reference tree not mounted")
def test_c_oracle_vs_live_reference():
    ref = ref_import.load()
    rng = np.random.RandomState(2024)
    pts = rng.rand(600, 3) * [6, 12, 9] + [0, -6, -3]
    angles, iters = ref_import.fabrik_ikine_with_iterations(ref, pts.tolist())
    r = c_oracle.fabrik_ikine(pts)
    assert np.array_equal(r["iters"], iters)
    np.testing.assert_allclose(r["angles"], angles, rtol=0, atol=1e-12)
    # the reference's exception for an out-of-box point, and its message format
    dh, links, limits = ref_import.fresh_robot_constants(ref)
    ik = ref.inverse.FabrikInverseKinematics(dh, links, limits)
    with pytest.raises(ref.robot.OutOfRobotReachException):
        ik.ikine(C.REF_INVERSE_UNIT_OUT_OF_REACH)


@pytest.mark.reference
@pytest.mark.skipif(not ref_import.available(), reason="reference tree not mounted")
def test_shipped_scalers_match_constants():
    import os
    import warnings
    import joblib
    base = os.path.join(ref_import.REFERENCE_ROOT, "models", "roboarm_model_1674153800-982793")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sx, sy = joblib.load(base + "_scaler_x.bin"), joblib.load(base + "_scaler_y.bin")
    np.testing.assert_array_equal(sx.mean_, np_oracle.SHIPPED_MEAN_X)
    np.testing.assert_array_equal(sx.scale_, np_oracle.SHIPPED_SCALE_X)
    np.testing.assert_array_equal(sy.mean_, np_oracle.SHIPPED_MEAN_Y)
    np.testing.assert_array_equal(sy.scale_, np_oracle.SHIPPED_SCALE_Y)


def test_oracle_scaler_arithmetic_matches_sklearn():
    """The oracle's scaler arithmetic equals sklearn's StandardScaler on both sides, with the shipped scalers' values."""
    pytest.importorskip("sklearn")
    from sklearn.preprocessing import StandardScaler
    sx, sy = StandardScaler(), StandardScaler()
    sx.mean_, sx.scale_ = np_oracle.SHIPPED_MEAN_X.copy(), np_oracle.SHIPPED_SCALE_X.copy()
    sy.mean_, sy.scale_ = np_oracle.SHIPPED_MEAN_Y.copy(), np_oracle.SHIPPED_SCALE_Y.copy()
    sx.n_features_in_, sy.n_features_in_ = 3, 4
    x = np.random.default_rng(1).uniform(-3, 6, size=(50, 3))
    np.testing.assert_array_equal(sx.transform(x), (x - sx.mean_) / sx.scale_)
    y = np.random.default_rng(2).normal(size=(50, 4)).astype(np.float32)
    mine = y.copy(); mine *= sy.scale_.astype(np.float32); mine += sy.mean_.astype(np.float32)
    np.testing.assert_array_equal(sy.inverse_transform(y), mine)


def test_reference_elbow_branch_follows_seed_noise_at_x_zero():
    """DESIGN 1: the elbow test C.x * D.x < 0 of inverse.py:82 compares seed noise when the target's x is 0 (the FK seed
    leaves cos(pi/2) ~ 1e-16 in C.x and D.x), and the reference's elbow branch then differs from that of the target 1e-9
    away on about a quarter of the rows.  From x = 1e-11 up nothing moves.  (Measured on this sample: the 3pi/2 - acos
    branch on 27.5 % of the rows at x = 1e-9 and 4.0 % at x = 0; 26 % of the x = 0 rows off by more than 1e-2 rad.)"""
    rng = np.random.RandomState(51)
    n = 20_000
    y, z = rng.uniform(-6, 6, n), rng.uniform(-3, 6, n)

    def solve(x):
        r = c_oracle.fabrik_ikine(np.stack([np.full(n, x), y, z], 1))
        assert (r["status"] == 0).all()
        return r["angles"], r["iters"], r["angles"][:, 1] > np.pi / 2   # theta_2 = 3pi/2 - acos: the negative branch

    a6, it6, neg6 = solve(1e-6)
    for x in (1e-9, 1e-11):   # measured 1.7e-8 rad from x = 1e-6 at both
        a, it, neg = solve(x)
        assert np.abs(a[:, 1:] - a6[:, 1:]).max() < 1e-6 and np.array_equal(it, it6) and np.array_equal(neg, neg6)
    a, _, _ = solve(1e-14)
    assert (np.abs(a[:, 1:] - a6[:, 1:]).max(axis=1) > 1e-2).sum() > 50   # measured 217 rows
    _, _, neg9 = solve(1e-9)
    for x in (0.0, -0.0):
        a0, it0, neg0 = solve(x)
        assert np.array_equal(it0, it6)
        assert 0.02 < neg0.mean() < 0.06 and 0.2 < neg9.mean() < 0.35
        # the in-plane rule (the branch at x = 1e-9) agrees with the reference's x = 0 branch on about three quarters
        # of the rows; always taking the non-negative branch agreed on 96 %
        assert 0.65 < (neg0 == neg9).mean() < 0.85 and (~neg0).mean() > 0.94
        assert (np.abs(a0[:, 1:] - a6[:, 1:]).max(axis=1) > 1e-2).mean() > 0.2
