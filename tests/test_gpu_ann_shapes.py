"""The three ANN kernels (fp16x3_ts: csrc/mlp_tc2.cu, fp16x3: mlp_tc.cu, fp32: mlp.cu) at the widths and weight scales
their packers branch on, against the fp64 NumPy restatement of ann.py:70-76.

ikb_mlp_tc2_pack chooses at load time between biases carried by the MMA (when the padded width hp has a spare column,
feature hmax is held at 1 and the biases are weight row hmax) and biases added in the epilogue (hidden width a multiple
of 128), picks a power-of-two weight scale per MMA layer clamped to 2^[-8, 24], splits hp into 256-wide N halves (the
last one 128 wide when hp = 128 (mod 256)) and pads unequal hidden widths to the widest.  Each shape below takes one of
those branches; each weight variant pushes the scale or the biases to an edge."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = ["fp16x3_ts", "fp16x3", "fp32"]
TOL = 1e-5  # rad: the project's bar for every mode (BASELINE.json north_star)

SHAPES = {
    "128x2": [3, 128, 128, 4],            # hp == hmax: no spare column -> epilogue bias
    "256x3": [3, 256, 256, 256, 4],       # epilogue bias over two MMA layers
    "512x2": [3, 512, 512, 4],            # widest net, epilogue bias, two full N halves
    "511x2": [3, 511, 511, 4],            # the spare column is the last one (bias row 511)
    "1": [3, 1, 4],                       # one hidden unit, no MMA layer
    "1x2": [3, 1, 1, 4],                  # one MMA layer of a single feature
    "ragged": [3, 17, 500, 33, 4],        # unequal widths padded to the widest (512)
    "deep": [3] + [64] * 15 + [4],        # 16 Dense layers, the maximum
    "384x2": [3, 384, 384, 4],            # NHALF = 2 with a 128-wide last half
}

# rows: one, a tile minus / exactly / plus one, and two full tiles per CTA on a 148-SM B200 plus one row
ROW_COUNTS = [1, 127, 128, 129, 148 * 128 * 2 + 1]


def _variant(dims, variant, seed):
    """Synthetic Glorot weights with non-zero biases, and edge cases of the per-layer weight scale and the biases.
    The MMA layers are the hidden-to-hidden ones (layers 1 .. len(dims) - 3)."""
    from oracle import np_oracle
    W, b = np_oracle.synthetic_mlp(seed=seed, dims=dims, bias_range=0.5)
    mma = range(1, len(W) - 1)
    if variant == "w*2^-14":        # tiny weights: with the biases in the epilogue (128x2) the scale exponent the
        for l in mma:               # packer wants is 28, clamped to 24; with a bias row, wmax is the row's 20
            W[l] = W[l] * np.float32(2.0 ** -14)
    elif variant == "w*2^10":       # large weights (max 78 .. 157): scale exponent 4 or 5, tanh mostly saturated
        for l in mma:
            W[l] = W[l] * np.float32(2.0 ** 10)
    elif variant == "bias+-5":
        rng = np.random.default_rng(seed + 1)
        b = [rng.uniform(-5, 5, size=v.shape).astype(np.float32) for v in b]
    elif variant == "zero-layer":   # an all-zero MMA layer (wmax = 0): its features are tanh(bias)
        W[1] = np.zeros_like(W[1])
    return W, b


CASES = [(s, "base") for s in SHAPES] + [(s, v) for s in ("128x2", "511x2", "ragged")
                                         for v in ("w*2^-14", "w*2^10", "bias+-5", "zero-layer")]

# Weights x 2^10 make the net ill-conditioned: fp32 evaluation itself (the NumPy oracle in float32, as Keras computes)
# misses the 1e-5 bar against fp64 -- max 3.9e-5 / 3.5e-5 / 9.3e-4 rad for 128x2 / 511x2 / ragged.  There each kernel is
# held to ILL_FACTOR times the fp32 oracle's own (mean, p99, max) error instead.  Measured on one B200: at most 2.7x
# (mean), 2.5x (p99), 2.6x (max) and 3.2x (saturating rows), all fp16x3 on 511x2; fp16x3_ts and fp32 stay within 1.4x.
ILL_CONDITIONED = {"w*2^10"}
ILL_FACTOR = 4


@pytest.fixture(scope="module")
def eng():
    from inversekinematicsann_b200.engine import IkEngine
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    e = IkEngine(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    yield e
    e.close()


def _points(n, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform([0, -6, -3], [6, 6, 6], size=(n, 3)).astype(np.float32).astype(np.float64)


def _saturating_points():
    """Targets far outside the scaler's range (standardised inputs of 1e3 .. 1e29): every first-layer unit saturates."""
    signs = np.array([[sx, sy, sz] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)], dtype=np.float64)
    rows = [signs * m for m in (1e3, 1e6, 1e30)]
    rows.append(np.array([[1e30, 1.0, 2.0], [0.5, -1e30, 1.0], [1.0, 2.0, 1e30]]))
    return np.concatenate(rows).astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("shape,variant", CASES, ids=[f"{s}-{v}" for s, v in CASES])
def test_ann_modes_at_packing_edges(eng, shape, variant):
    import torch
    from oracle import np_oracle
    dims = SHAPES[shape]
    W, b = _variant(dims, variant, seed=len(dims) * 1000 + dims[1])
    eng.mlp_load(W, b, np_oracle.SHIPPED_MEAN_X, np_oracle.SHIPPED_SCALE_X, np_oracle.SHIPPED_MEAN_Y,
                 np_oracle.SHIPPED_SCALE_Y)
    n = ROW_COUNTS[-1]
    xyz = _points(n, seed=dims[1])                       # float32 values: the float32 and float64 feeds are the same
    want = np_oracle.mlp_predict(xyz, W, b, dtype=np.float64)
    sat = _saturating_points()
    want_sat = np_oracle.mlp_predict(sat, W, b, dtype=np.float64)
    bound = (TOL, TOL, TOL)
    bound_sat = TOL
    if variant in ILL_CONDITIONED:
        e32 = np.abs(np_oracle.mlp_predict(xyz, W, b).astype(np.float64) - want)
        r32 = e32.max(axis=1)
        bound = tuple(ILL_FACTOR * v for v in (float(e32.mean()), float(np.quantile(r32, 0.99)), float(r32.max())))
        s32 = float(np.abs(np_oracle.mlp_predict(sat, W, b).astype(np.float64) - want_sat).max())
        bound_sat = max(TOL, ILL_FACTOR * s32)
        print(f"[{shape} {variant}] fp32 oracle vs fp64: mean {bound[0] / ILL_FACTOR:.2e} p99 {bound[1] / ILL_FACTOR:.2e} "
              f"max {bound[2] / ILL_FACTOR:.2e}; saturating {s32:.2e}")
    got = {}
    for mode in MODES:
        a64, _ = eng.ann_solve(xyz, mode=mode)                       # host, float64 targets
        a32, _ = eng.ann_solve(xyz.astype(np.float32), mode=mode)    # host, float32 targets
        assert np.array_equal(a64, a32), mode
        out = torch.full((n, 4), float("nan"), device="cuda")
        eng.ann_solve_device(torch.from_numpy(xyz.astype(np.float32)).cuda(), out, mode=mode)
        assert np.array_equal(out.cpu().numpy(), a64), mode
        out64 = torch.full((n, 4), float("nan"), device="cuda")
        eng.ann_solve_device(torch.from_numpy(xyz).cuda(), out64, mode=mode)
        assert np.array_equal(out64.cpu().numpy(), a64), mode
        for m in ROW_COUNTS[:-1]:                          # a row's result does not depend on the batch around it
            assert np.array_equal(eng.ann_solve(xyz[:m], mode=mode)[0], a64[:m]), (mode, m)
        err = np.abs(a64.astype(np.float64) - want).max(axis=1)
        mean, p99, mx = float(np.abs(a64 - want).mean()), float(np.quantile(err, 0.99)), float(err.max())
        s_out, _ = eng.ann_solve(sat, mode=mode)
        s_err = float(np.abs(s_out.astype(np.float64) - want_sat).max())
        print(f"[{shape} {variant} {mode}] vs fp64: mean {mean:.2e} p99 {p99:.2e} max {mx:.2e}; saturating {s_err:.2e}")
        assert np.isfinite(a64).all() and np.isfinite(s_out).all(), mode
        got[mode] = (a64, mean, p99, mx, s_err)
    for mode, (_, mean, p99, mx, s_err) in got.items():
        assert mean <= bound[0] and p99 <= bound[1] and mx <= bound[2], (mode, mean, p99, mx, bound)
        assert s_err <= bound_sat, (mode, s_err, bound_sat)
    # the three kernels are independent implementations of one network: pairwise within twice the bound
    for i, m1 in enumerate(MODES):
        for m2 in MODES[i + 1:]:
            assert np.abs(got[m1][0] - got[m2][0]).max() <= 2 * bound[2], (m1, m2)
