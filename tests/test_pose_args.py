"""Argument checks of the damped-least-squares refinement onto poses that need no GPU (the rest is in
test_gpu_pose_refine.py)."""
import ctypes

import numpy as np
import pytest


def _refusal(fn, *args):
    from inversekinematicsann_b200 import _native
    lib = _native.load()
    assert fn(*args) == _native.IKB_ERR_INVALID
    return lib.ikb_last_error(None).decode()


def _weights(*w):
    return (ctypes.c_double * 6)(*w)


def test_c_abi_refusals_without_an_engine():
    """The arguments are checked before the engine, so each refusal is told apart by its text."""
    from inversekinematicsann_b200 import _native
    lib = _native.load()
    poses, seed, ang = np.zeros((3, 4, 4)), np.zeros((3, 4)), np.zeros((3, 4))
    its, err = np.zeros(3, np.int32), np.zeros(3)
    big = np.zeros((7, 4))
    x, s, a, i, e, b = (v.ctypes.data for v in (poses, seed, ang, its, err, big))
    F32, F64 = _native.IKB_F32, _native.IKB_F64
    ones = _weights(1, 1, 1, 1, 1, 1)
    st = _native.IkbStats()
    nan, inf = float("nan"), float("inf")
    for fn, name, last in ((lib.ikb_dls_pose_refine_host, "ikb_dls_pose_refine_host", ctypes.byref(st)),
                           (lib.ikb_dls_pose_refine_device, "ikb_dls_pose_refine_device", None)):
        def call(xp=x, xd=F64, n=3, sp=s, ns=3, ap=a, ad=F64, w=ones, damping=0.05, tol=1e-9, mi=32, ip=i, ep=e):
            return (None, xp, xd, n, sp, ns, ap, ad, w, damping, tol, mi, ip, ep, last)
        cases = [
            (call(), "NULL engine"),
            (call(ip=None, ep=None), "NULL engine"),
            (call(n=0, xp=None, sp=None, ap=None, ns=1), "NULL engine"),
            (call(w=_weights(1, 0, 0, 0, 0, 0)), "NULL engine"),
            (call(w=_weights(0, 0, 0, 0, 0, 2.5)), "NULL engine"),
            # the weights
            (call(w=None), "NULL weights"),
            (call(w=_weights(1, 1, -1, 1, 1, 1)), "weights must be >= 0 and finite"),
            (call(w=_weights(1, 1, 1, 1, -0.5, 1)), "weights must be >= 0 and finite"),
            (call(w=_weights(nan, 1, 1, 1, 1, 1)), "weights must be >= 0 and finite"),
            (call(w=_weights(1, 1, 1, inf, 1, 1)), "weights must be >= 0 and finite"),
            (call(w=_weights(0, 0, 0, 0, 0, 0)), "all six weights are zero"),
            (call(w=_weights(0, 0, 0, 0, -0.0, 0)), "all six weights are zero"),
            # everything the position refinement refuses
            (call(xp=None), "NULL targets"),
            (call(sp=None), "NULL seeds"),
            (call(ap=None), "NULL angles_out"),
            (call(n=-1), "negative n"),
            (call(ns=2), "n_seed must be 1 or n"),
            (call(ns=0), "n_seed must be 1 or n"),
            (call(xd=2), "unknown dtype"),
            (call(ad=-1), "unknown dtype"),
            (call(damping=0.0), "damping must be positive and finite"),
            (call(damping=-0.1), "damping must be positive and finite"),
            (call(damping=nan), "damping must be positive and finite"),
            (call(damping=inf), "damping must be positive and finite"),
            (call(tol=-1e-12), "tol must be >= 0 and not NaN"),
            (call(tol=nan), "tol must be >= 0 and not NaN"),
            (call(mi=-1), "max_iter must be >= 0"),
            # the pose buffer is aligned to its element size
            (call(xp=x + 4), "aligned"),
            (call(xp=x + 2, xd=F32), "aligned"),
            (call(xp=x + 4, xd=F32), "NULL engine"),
            (call(sp=s + 4), "aligned"),
            (call(ap=a + 4), "aligned"),
            (call(ep=e + 4), "aligned"),
            (call(ip=i + 2), "aligned"),
            (call(ap=s + 32), "overlap"),
            (call(sp=b + 32, ap=b), "overlap"),
            (call(sp=b, ns=1, ap=b, n=3), "overlap"),
            (call(sp=b, ns=1, ap=b + 32 * 2, n=3), "NULL engine"),
            (call(sp=s, ap=s), "NULL engine"),               # in place
        ]
        for args, why in cases:
            msg = _refusal(fn, *args)
            assert msg.startswith(name + ": ") and why in msg, (args, msg)


def test_engine_argument_checks():
    from inversekinematicsann_b200.engine import IkEngine
    check = IkEngine._pose_args
    poses = np.zeros((5, 4, 4))
    for seed, n_seed in ((np.zeros((5, 4)), 5), (np.zeros(4), 1), (np.zeros((1, 4)), 1)):
        p, s, ns, out = check(poses, seed, None)
        assert p.shape == (5, 4, 4) and ns == n_seed and s.shape == (n_seed, 4) and out.shape == (5, 4)
    # a strided view (what fkine_batch returns: chain[:, 3]) is made contiguous
    chain = np.arange(5 * 4 * 16, dtype=np.float64).reshape(5, 4, 4, 4)
    p, _, _, _ = check(chain[:, 3], np.zeros(4), None)
    assert p.flags.c_contiguous and np.array_equal(p, chain[:, 3])
    p, _, _, _ = check(np.zeros((2, 4, 4), np.float32), np.zeros(4), None)
    assert p.dtype == np.float32
    p, _, _, _ = check([np.eye(4).tolist()] * 2, np.zeros(4), None)
    assert p.dtype == np.float64 and p.shape == (2, 4, 4)
    for bad in (np.zeros((5, 3, 4)), np.zeros((5, 16)), np.zeros((4, 4))):
        with pytest.raises(ValueError):
            check(bad, np.zeros(4), None)
    with pytest.raises(ValueError):
        check(poses, np.zeros((2, 4)), None)
    with pytest.raises(TypeError):
        check(poses, np.zeros(4), np.empty((5, 4), np.float32))


def test_engine_refusals_reach_the_library_before_the_engine():
    from inversekinematicsann_b200 import _native, engine
    from inversekinematicsann_b200.engine import IkEngine
    eng = IkEngine.__new__(IkEngine)
    eng._lib = _native.load()
    eng._handle = ctypes.c_void_p()
    eng.device = 0
    poses, seed = np.zeros((3, 4, 4)), np.zeros((3, 4))
    for kw, why in (({"weights": [1, 1, 1, 1, 1, -1]}, "weights"), ({"weights": [0] * 6}, "all six"),
                    ({"damping": 0.0}, "damping"), ({"tol": -1.0}, "tol"), ({"max_iter": -2}, "max_iter"),
                    ({}, "NULL engine")):
        with pytest.raises(ValueError, match=why):
            eng.dls_pose_refine(poses, seed, **kw)
    with pytest.raises(ValueError, match="6 numbers"):
        eng.dls_pose_refine(poses, seed, weights=[1, 1, 1])
    with pytest.raises(TypeError, match="6 numbers"):
        eng.dls_pose_refine(poses, seed, weights=1.0)
    w, d, t, m = engine._pose_params(None, None, None, None)
    assert list(w) == list(engine.POSE_WEIGHTS) and (d, t, m) == (engine.POSE_DAMPING, engine.POSE_TOL,
                                                                 engine.POSE_MAX_ITER)


def test_device_argument_checks_before_any_device_use():
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    eng = IkEngine.__new__(IkEngine)
    eng.device = 0
    cpu_p, cpu4 = torch.zeros(4, 4, 4, dtype=torch.float64), torch.zeros(4, 4, dtype=torch.float64)
    with pytest.raises(TypeError, match="poses"):
        eng.dls_pose_refine_device(cpu_p, cpu4, cpu4)
    with pytest.raises(TypeError, match="poses"):
        eng.dls_pose_refine_device(np.zeros((4, 4, 4)), cpu4, cpu4)


def test_python_layer_without_a_gpu():
    """Empty batches return refine's shapes without an engine; the pose methods exist on both solver classes."""
    from inversekinematicsann_b200.kinematics.inverse import (AnnInverseKinematics, FabrikInverseKinematics,
                                                              poses_to_array)
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    for cls in (FabrikInverseKinematics, AnnInverseKinematics):
        ik = cls(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
        assert ik.refine_pose([], []) == []
        out, its, err = ik.refine_pose(np.zeros((0, 4, 4)), np.zeros((0, 4), np.float32), as_array=True,
                                       return_iterations=True, return_fk_error=True)
        assert out.shape == (0, 4) and out.dtype == np.float32 and its.dtype == np.int32 and err.dtype == np.float32
        assert ik.ikine_pose([]) == []
        out, its, err = ik.ikine_pose(np.zeros((0, 4, 4)), as_array=True, return_iterations=True,
                                      return_fk_error=True)
        assert out.shape == (0, 4) and out.dtype == np.float64 and its.shape == (0,) and err.shape == (0,)
    with pytest.raises(ValueError, match="shape"):
        poses_to_array(np.zeros((3, 4)))
