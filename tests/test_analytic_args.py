"""Argument checks of the closed-form inverse kinematics that need no GPU (the rest is in test_gpu_analytic_ik.py), and
`analytic_ik`, the NumPy restatement of its arithmetic that the GPU tests compare with."""
import math

import numpy as np
import pytest


# ---- NumPy restatement of include/ikb200.h ikb_analytic_ik_* (the reference the GPU tests compare with) -----------

def _wrap(th):
    """Angles with |theta| > pi replaced by the IEEE remainder(theta, 2 pi) (exact), as csrc/analytic.cu does."""
    th = np.array(th, dtype=np.float64)
    big = np.abs(th) > np.pi
    if big.any():
        th[big] = np.frompyfunc(lambda v: math.remainder(v, 2 * np.pi), 1, 1)(th[big]).astype(np.float64)
    return th


def _triangle(u, v, phi, a2, a3, a4):
    """The two-link triangle to the wrist point -> (theta2 [+, -], theta3 [+, -], theta4 [+, -], not reached)."""
    uw = u - a4 * np.cos(phi)
    vw = v - a4 * np.sin(phi)
    r = np.sqrt(uw * uw + vw * vw)
    num = ((a2 + a3) - r) * ((a2 + a3) + r)
    den = (r - (a2 - a3)) * (r + (a2 - a3))
    t = 2.0 * np.arctan2(np.sqrt(np.where(num > 0, num, 0.0)), np.sqrt(np.where(den > 0, den, 0.0)))
    st, ct = np.sin(t), np.cos(t)
    base = np.arctan2(vw, uw)
    g = np.arctan2(a3 * st, a2 + a3 * ct)
    th3 = (t, 0.0 - t)
    th2 = (base - g, base - (0.0 - g))
    th4 = tuple(phi - th2[k] - th3[k] for k in range(2))
    return th2, th3, th4, (num < 0) | (den < 0)


def analytic_ik(x, dh, pitch=None):
    """Every closed-form branch for an arm with a turning base and three parallel joints (alpha_2..4 = 0,
    |cos alpha_1| <= 1e-12, a_2, a_3 > 0), restating ikb_analytic_ik_* in fp64.  dh: the 4 x 4 table (rows theta,
    epsilon, a, alpha).  x: (n, 4, 4) poses (pitch None; 2 branches [theta3 >= 0, theta3 <= 0]) or (n, 3) positions
    with the pitch of the tool axis, one value or n (4 branches [front +, front -, back +, back -]).  Returns
    (angles (n, B, 4) float64, status (n,) int32: bit b set when branch b does not reach)."""
    dh = np.asarray(dh, dtype=np.float64)
    eps, a, alpha = dh[1], dh[2], dh[3]
    s = 1.0 if np.sin(alpha[0]) > 0 else -1.0
    a1, a2, a3, a4 = a
    d = (eps[1] + eps[2]) + eps[3]
    x = np.asarray(x, dtype=np.float64) + 0.0  # -0 reads as +0
    with np.errstate(all="ignore"):
        if pitch is None:
            x = x.reshape(-1, 4, 4)
            n = x.shape[0]
            R, p = x[:, :3, :3], x[:, :3, 3]
            th1 = np.arctan2(s * R[:, 0, 2], -s * R[:, 1, 2])
            c1, s1 = np.cos(th1), np.sin(th1)
            phi = np.arctan2(s * R[:, 2, 0], c1 * R[:, 0, 0] + s1 * R[:, 1, 0])
            u = c1 * p[:, 0] + s1 * p[:, 1] - a1
            v = s * (p[:, 2] - eps[0])
            th2, th3, th4, bad = _triangle(u, v, phi, a2, a3, a4)
            ang = np.stack([np.stack([th1, th2[k], th3[k], th4[k]], 1) for k in range(2)], 1)
            status = np.where(bad, 3, 0)
            finite = np.isfinite(x[:, :3, :]).all(axis=(1, 2))
        else:
            x = x.reshape(-1, 3)
            n = x.shape[0]
            pt = np.broadcast_to(np.asarray(pitch, dtype=np.float64).reshape(-1) + 0.0, (n,))
            px, py, pz = x[:, 0], x[:, 1], x[:, 2]
            rho2 = px * px + py * py
            short = rho2 < d * d
            q = np.sqrt(np.where(short, 0.0, rho2 - d * d))
            base = np.arctan2(py, px)
            v = s * (pz - eps[0])
            ang, status = [], np.zeros(n, dtype=np.int64)
            for side, (qq, phi) in enumerate(((q, pt), (-q, np.pi - pt))):
                th1 = base - np.arctan2(-s * d + 0.0, qq)
                th2, th3, th4, bad = _triangle(qq - a1, v, phi, a2, a3, a4)
                for k in range(2):
                    ang.append(np.stack([th1, th2[k], th3[k], th4[k]], 1))
                status |= np.where(bad | short, 3 << (2 * side), 0)
            ang = np.stack(ang, 1)
            finite = np.isfinite(x).all(axis=1) & np.isfinite(pt)
    ang = _wrap(ang)
    B = ang.shape[1]
    ang[~finite] = np.nan
    status = np.where(finite, status, (1 << B) - 1).astype(np.int32)
    return ang, status


def _refusal(fn, *args):
    from inversekinematicsann_b200 import _native
    lib = _native.load()
    assert fn(*args) == _native.IKB_ERR_INVALID
    return lib.ikb_last_error(None).decode()


def test_c_abi_refusals_without_an_engine():
    """The arguments are checked before the engine, so each refusal is told apart by its text."""
    from inversekinematicsann_b200 import _native
    lib = _native.load()
    poses, pts, pitch, ang, st = np.zeros((3, 4, 4)), np.zeros((3, 3)), np.zeros(3), np.zeros((3, 4, 4)), \
        np.zeros(3, np.int32)
    x, p, pp, a, s = (v.ctypes.data for v in (poses, pts, pitch, ang, st))
    F32, F64 = _native.IKB_F32, _native.IKB_F64
    POSE, POS = _native.IKB_AIK_POSE, _native.IKB_AIK_POSITION_PITCH
    stats = _native.IkbStats()
    for fn, name, last in ((lib.ikb_analytic_ik_host, "ikb_analytic_ik_host", stats),
                           (lib.ikb_analytic_ik_device, "ikb_analytic_ik_device", None)):
        def call(kind=POSE, xp=x, xd=F64, n=3, pt=None, npt=0, ap=a, ad=F64, sp=s):
            return (None, kind, xp, xd, n, pt, npt, ap, ad, sp, last)

        def pos(**kw):
            return call(**{"kind": POS, "xp": p, "pt": pp, "npt": 3, **kw})
        cases = [
            (call(), "NULL engine"),
            (call(sp=None), "NULL engine"),
            (call(n=0, xp=None, ap=None), "NULL engine"),
            (call(npt=7), "NULL engine"),                      # the pose kind ignores n_pitch
            (pos(), "NULL engine"),
            (pos(npt=1), "NULL engine"),
            (pos(n=0, xp=None, ap=None, pt=None, npt=1), "NULL engine"),
            (pos(xd=F32, ad=F32, pt=pp + 4), "NULL engine"),
            (call(xp=None), "NULL input"),
            (pos(xp=None), "NULL input"),
            (call(ap=None), "NULL angles_out"),
            (call(kind=2), "unknown kind"),
            (call(kind=-1), "unknown kind"),
            (call(xd=2), "unknown dtype"),
            (call(ad=-1), "unknown dtype"),
            (call(n=-1), "negative n"),
            (pos(pt=None), "NULL pitch"),
            (call(pt=pp, npt=3), "pitch given for the pose kind"),
            (pos(npt=2), "n_pitch must be 1 or n"),
            (pos(npt=0), "n_pitch must be 1 or n"),
            (call(xp=x + 4), "aligned"),
            (call(xp=x + 2, xd=F32), "aligned"),
            (call(xp=x + 4, xd=F32), "NULL engine"),
            (pos(pt=pp + 4), "aligned"),
            (call(ap=a + 4), "aligned"),
            (call(ap=a + 4, ad=F32), "NULL engine"),
            (call(sp=s + 2), "aligned"),
        ]
        for args, why in cases:
            msg = _refusal(fn, *args)
            assert msg.startswith(name + ": ") and why in msg, (args, msg)


def _engine_without_device():
    import ctypes

    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.engine import IkEngine
    eng = IkEngine.__new__(IkEngine)
    eng._lib = _native.load()
    eng._handle = ctypes.c_void_p()
    eng.device = 0
    return eng


def test_engine_argument_checks():
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.engine import IkEngine
    check = IkEngine._analytic_args
    x, kind, pitch, b = check(np.zeros((5, 4, 4)), None)
    assert kind == _native.IKB_AIK_POSE and pitch is None and b == 2 and x.shape == (5, 4, 4)
    chain = np.arange(5 * 4 * 16, dtype=np.float64).reshape(5, 4, 4, 4)
    x, _, _, _ = check(chain[:, 3], None)  # what fkine_batch returns: a strided view, made contiguous
    assert x.flags.c_contiguous and np.array_equal(x, chain[:, 3])
    x, kind, pitch, b = check(np.zeros((5, 3), np.float32), 0.25)
    assert kind == _native.IKB_AIK_POSITION_PITCH and b == 4 and pitch.dtype == np.float32 and pitch.shape == (1,)
    x, _, pitch, _ = check([[1, 2, 3]] * 5, np.arange(5))
    assert x.dtype == np.float64 and pitch.dtype == np.float64 and pitch.shape == (5,)
    for bad, p, why in ((np.zeros((5, 4, 4)), 0.5, "no pitch"), (np.zeros((5, 3)), None, "need a pitch"),
                        (np.zeros((5, 3)), np.zeros(2), "1 or 5"), (np.zeros((5, 4)), 0.5, "shape"),
                        (np.zeros((5, 3, 4)), None, "shape")):
        with pytest.raises(ValueError, match=why):
            check(bad, p)
    eng = _engine_without_device()
    with pytest.raises(TypeError, match="out_dtype"):
        eng.analytic_ik(np.zeros((2, 4, 4)), out_dtype=np.int32)
    for x, p in ((np.zeros((2, 4, 4)), None), (np.zeros((2, 3)), [0.1, 0.2])):
        with pytest.raises(ValueError, match="NULL engine"):
            eng.analytic_ik(x, p)


def test_device_argument_checks_before_any_device_use():
    import torch
    eng = _engine_without_device()
    with pytest.raises(TypeError, match="x must be a CUDA"):
        eng.analytic_ik_device(torch.zeros(4, 4, 4, dtype=torch.float64), None, torch.zeros(4, 2, 4))
    with pytest.raises(TypeError, match="x must be a CUDA"):
        eng.analytic_ik_device(np.zeros((4, 3)), torch.zeros(1), torch.zeros(4, 4, 4))


def test_python_layer_without_a_gpu():
    """Empty batches return their shapes without an engine; branch selection is checked before any device use."""
    from inversekinematicsann_b200.kinematics.inverse import AnalyticInverseKinematics, _branch
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    ik = AnalyticInverseKinematics(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
    assert ik.ikine([], 0.0) == []
    out, st = ik.ikine(np.zeros((0, 3)), -math.pi / 2, as_array=True, return_status=True)
    assert out.shape == (0, 4) and st.shape == (0,)
    ang, st = ik.ikine_branches([], 0.0)
    assert ang.shape == (0, 4, 4) and st.dtype == np.int32
    ang, st = ik.ikine_pose_branches(np.zeros((0, 4, 4)))
    assert ang.shape == (0, 2, 4) and st.shape == (0,)
    assert ik.ikine_pose([]) == []
    out, its, err = ik.ikine_pose(np.zeros((0, 4, 4)), as_array=True, return_iterations=True, return_fk_error=True)
    assert out.shape == (0, 4) and out.dtype == np.float64 and its.shape == (0,) and err.shape == (0,)
    assert [_branch(e, b) for b in ("front", "back") for e in (1, -1)] == [0, 1, 2, 3]
    for bad in ((0, "front"), (1, "up"), (2, "back")):
        with pytest.raises(ValueError):
            _branch(*bad)
    with pytest.raises(ValueError, match="elbow"):
        ik.ikine([[1.0, 0.0, 1.0]], 0.0, elbow=0)
    with pytest.raises(ValueError, match="elbow"):
        ik.ikine_pose(np.tile(np.eye(4), (1, 1, 1)), elbow=2)
    from dropin.kinematics import inverse as dropin_inverse
    assert dropin_inverse.AnalyticInverseKinematics is AnalyticInverseKinematics


def test_restatement_on_the_reference_table():
    """The NumPy restatement itself: every branch of poses of random angles reproduces the pose, the original angles
    are among the branches, and the position kind reaches with the pose's pitch."""
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    rng = np.random.default_rng(3)
    th = rng.uniform(-np.pi, np.pi, (2000, 4))
    T = _np_fk(th, R.dh_matrix)
    ang, st = analytic_ik(T, R.dh_matrix)
    for b in range(2):
        assert np.abs(_np_fk(ang[:, b], R.dh_matrix)[:, :3] - T[:, :3]).max() < 1e-13
    d = np.abs(np.remainder(ang - th[:, None] + np.pi, 2 * np.pi) - np.pi).max(axis=2).min(axis=1)
    assert d.max() < 1e-9
    phi = th[:, 1:].sum(axis=1)
    ds = []
    for pitch in (phi, np.pi - phi):  # the pose reaches toward its point at pitch phi, or back over the base
        ang, st = analytic_ik(T[:, :3, 3], R.dh_matrix, pitch)
        for b in range(4):
            ok = (st >> b) & 1 == 0
            assert np.abs(_np_fk(ang[ok, b], R.dh_matrix)[:, :3, 3] - T[ok, :3, 3]).max() < 1e-13
        assert (np.abs(ang) <= np.pi).all()
        ds.append(np.abs(np.remainder(ang - th[:, None] + np.pi, 2 * np.pi) - np.pi).max(axis=2).min(axis=1))
    assert np.minimum(*ds).max() < 1e-9


def _np_fk(th, dh):
    dh = np.asarray(dh, dtype=np.float64)
    eps, a, al = dh[1], dh[2], dh[3]
    T = np.tile(np.eye(4), (th.shape[0], 1, 1))
    for j in range(4):
        c, s = np.cos(th[:, j]), np.sin(th[:, j])
        M = np.zeros_like(T)
        M[:, 0] = np.stack([c, -s * np.cos(al[j]), s * np.sin(al[j]), a[j] * c], 1)
        M[:, 1] = np.stack([s, c * np.cos(al[j]), -c * np.sin(al[j]), a[j] * s], 1)
        M[:, 2, 1:] = [np.sin(al[j]), np.cos(al[j]), eps[j]]
        M[:, 3, 3] = 1.0
        T = T @ M
    return T
