"""Argument checks of the damped-least-squares refinement that need no GPU (the rest is in test_gpu_dls_refine.py)."""
import ctypes

import numpy as np
import pytest


def _refusal(fn, *args):
    from inversekinematicsann_b200 import _native
    lib = _native.load()
    assert fn(*args) == _native.IKB_ERR_INVALID
    return lib.ikb_last_error(None).decode()


def test_c_abi_refusals_without_an_engine():
    """The arguments are checked before the engine, so each refusal is told apart by its text."""
    from inversekinematicsann_b200 import _native
    lib = _native.load()
    xyz, seed, ang = np.zeros((3, 3)), np.zeros((3, 4)), np.zeros((3, 4))
    its, err = np.zeros(3, np.int32), np.zeros(3)
    big = np.zeros((7, 4))
    x, s, a, i, e, b = (v.ctypes.data for v in (xyz, seed, ang, its, err, big))
    F32, F64 = _native.IKB_F32, _native.IKB_F64
    st = _native.IkbStats()
    for fn, name, last in ((lib.ikb_dls_refine_host, "ikb_dls_refine_host", ctypes.byref(st)),
                           (lib.ikb_dls_refine_device, "ikb_dls_refine_device", None)):
        def call(xp=x, xd=F64, n=3, sp=s, ns=3, ap=a, ad=F64, damping=0.05, tol=1e-9, mi=32, ip=i, ep=e):
            return (None, xp, xd, n, sp, ns, ap, ad, damping, tol, mi, ip, ep, last)
        cases = [
            (call(), "NULL engine"),
            (call(ip=None, ep=None), "NULL engine"),
            (call(n=0, xp=None, sp=None, ap=None, ns=1), "NULL engine"),
            (call(xp=None), "NULL targets"),
            (call(sp=None), "NULL seeds"),
            (call(ap=None), "NULL angles_out"),
            (call(n=-1), "negative n"),
            (call(ns=2), "n_seed must be 1 or n"),
            (call(ns=0), "n_seed must be 1 or n"),
            (call(ns=4), "n_seed must be 1 or n"),
            (call(xd=2), "unknown dtype"),
            (call(ad=-1), "unknown dtype"),
            (call(damping=0.0), "damping must be positive and finite"),
            (call(damping=-0.1), "damping must be positive and finite"),
            (call(damping=float("nan")), "damping must be positive and finite"),
            (call(damping=float("inf")), "damping must be positive and finite"),
            (call(tol=-1e-12), "tol must be >= 0 and not NaN"),
            (call(tol=float("nan")), "tol must be >= 0 and not NaN"),
            (call(mi=-1), "max_iter must be >= 0"),
            (call(xp=x + 4), "aligned"),
            (call(xp=x + 2, xd=F32), "aligned"),
            (call(sp=s + 4), "aligned"),
            (call(ap=a + 4), "aligned"),
            (call(ep=e + 4), "aligned"),
            (call(ip=i + 2), "aligned"),
            (call(ap=s + 32), "overlap"),                    # angles_out one row past the seeds
            (call(sp=b + 32, ap=b), "overlap"),
            (call(sp=b, ns=1, ap=b + 32 * 2, n=3), "NULL engine"),  # disjoint: only the engine is missing
            (call(sp=b, ns=1, ap=b, n=3), "overlap"),        # a broadcast seed cannot be written in place
            (call(sp=b, ap=b + 8 * 32, n=3), "NULL engine"),
            (call(sp=s, ap=s), "NULL engine"),               # in place
        ]
        for args, why in cases:
            msg = _refusal(fn, *args)
            assert msg.startswith(name + ": ") and why in msg, (args, msg)
        # float32 seeds: a partial overlap is measured in 16-byte rows
        s32 = np.zeros((3, 4), np.float32)
        p = s32.ctypes.data
        assert "overlap" in _refusal(fn, *call(sp=p, ap=p + 16, ad=F32, ep=None))
        assert "NULL engine" in _refusal(fn, *call(sp=p, ap=p, ad=F32, ep=None))


def test_engine_argument_checks():
    from inversekinematicsann_b200.engine import IkEngine
    check = IkEngine._dls_args
    xyz = np.zeros((5, 3))
    for seed, n_seed in ((np.zeros((5, 4)), 5), (np.zeros(4), 1), (np.zeros((1, 4)), 1), ([[0.0] * 4] * 5, 5)):
        x, s, ns, out = check(xyz, seed, None)
        assert ns == n_seed and s.shape == (n_seed, 4) and out.shape == (5, 4) and out.dtype == np.float64
    _, _, _, out = check(xyz.astype(np.float32), np.zeros((5, 4), np.float32), None)
    assert out.dtype == np.float32
    seed = np.zeros((5, 4))
    assert check(xyz, seed, seed)[3] is seed                     # in place
    given = np.empty((5, 4))
    assert check(xyz, np.zeros(4), given)[3] is given
    ro = np.empty((5, 4))
    ro.flags.writeable = False
    bad = [
        (ValueError, np.zeros((5, 4)), np.zeros((5, 4)), None),
        (ValueError, xyz, np.zeros((5, 3)), None),
        (ValueError, xyz, np.zeros((2, 4)), None),
        (ValueError, xyz, np.zeros((6, 4)), None),
        (ValueError, xyz, np.zeros(5), None),
        (ValueError, xyz, np.zeros(4), np.empty((4, 4))),
        (TypeError, xyz, np.zeros(4), np.empty((5, 4), np.float32)),
        (TypeError, xyz, np.zeros(4, np.float32), np.empty((5, 4))),
        (ValueError, xyz, np.zeros(4), np.empty((5, 8))[:, ::2]),
        (ValueError, xyz, np.zeros(4), ro),
        (TypeError, xyz, np.zeros(4), [[0.0] * 4] * 5),
    ]
    for exc, x, s, o in bad:
        with pytest.raises(exc):
            check(x, s, o)
    ro_seed = np.zeros((5, 4))
    ro_seed.flags.writeable = False
    with pytest.raises(ValueError):
        check(xyz, ro_seed, ro_seed)


def test_engine_refusals_reach_the_library_before_the_engine():
    """An engine object without a handle: shapes are refused in Python, values by the library, each by its text."""
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.engine import IkEngine
    eng = IkEngine.__new__(IkEngine)
    eng._lib = _native.load()
    eng._handle = ctypes.c_void_p()
    eng.device = 0
    xyz, seed = np.zeros((3, 3)), np.zeros((3, 4))
    for kw, why in (({"damping": 0.0}, "damping"), ({"damping": float("inf")}, "damping"), ({"tol": -1.0}, "tol"),
                    ({"max_iter": -2}, "max_iter"), ({}, "NULL engine")):
        with pytest.raises(ValueError, match=why):
            eng.dls_refine(xyz, seed, **kw)
    shared = np.zeros((4, 4))
    with pytest.raises(ValueError, match="overlap"):
        eng.dls_refine(xyz, shared[:3], out=shared[1:])
    with pytest.raises(ValueError, match="NULL engine"):  # the same memory as another view is in place
        eng.dls_refine(xyz, shared[:3], out=shared[:3])
    # the defaults
    from inversekinematicsann_b200 import engine
    assert engine._dls_params(None, None, None) == (engine.DLS_DAMPING, engine.DLS_TOL, engine.DLS_MAX_ITER)
    assert engine._dls_params(0.1, 0, 3) == (0.1, 0.0, 3)


def test_device_argument_checks_before_any_device_use():
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    eng = IkEngine.__new__(IkEngine)
    eng.device = 0
    cpu3, cpu4 = torch.zeros(4, 3, dtype=torch.float64), torch.zeros(4, 4, dtype=torch.float64)
    with pytest.raises(TypeError):
        eng.dls_refine_device(cpu3, cpu4, cpu4)
    with pytest.raises(TypeError):
        eng.dls_refine_device(np.zeros((4, 3)), cpu4, cpu4)


def test_python_layer_without_a_gpu():
    """Empty batches return ikine's shapes without an engine; refine exists on both solver classes."""
    from inversekinematicsann_b200.kinematics.inverse import AnnInverseKinematics, FabrikInverseKinematics
    from inversekinematicsann_b200.robot.robot import SixDOFRobot as R
    for cls in (FabrikInverseKinematics, AnnInverseKinematics):
        ik = cls(R.dh_matrix, R.links_lengths, R.effector_workspace_limits)
        assert ik.refine([], []) == []
        out, its, err = ik.refine(np.zeros((0, 3)), np.zeros((0, 4), np.float32), as_array=True,
                                  return_iterations=True, return_fk_error=True)
        assert out.shape == (0, 4) and out.dtype == np.float32 and its.dtype == np.int32 and err.dtype == np.float32
        assert ik.refine([], [], as_array=True).dtype == np.float64
