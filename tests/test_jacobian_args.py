"""Argument checks of the arm Jacobian that need no GPU (the rest is in test_gpu_jacobian.py)."""
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
    ang, jac, w = np.zeros((2, 4)), np.zeros((2, 6, 4)), np.zeros(2)
    a, j, m = ang.ctypes.data, jac.ctypes.data, w.ctypes.data
    G, F64 = _native.IKB_JAC_GEOMETRIC, _native.IKB_F64
    for fn, name in ((lib.ikb_jacobian_host, "ikb_jacobian_host"), (lib.ikb_jacobian_device, "ikb_jacobian_device")):
        cases = [
            ((None, a, F64, 2, G, j, m, None), "NULL engine"),
            ((None, a, F64, -1, G, j, m, None), "negative n"),
            ((None, a, 7, 2, G, j, m, None), "unknown dtype"),
            ((None, a, F64, 2, 2, j, m, None), "unknown `what`"),
            ((None, a, F64, 2, -1, None, m, None), "unknown `what`"),
            ((None, a, F64, 2, G, None, None, None), "both outputs are NULL"),
            ((None, a, F64, 0, G, None, None, None), "both outputs are NULL"),
            ((None, None, F64, 2, G, j, None, None), "NULL angles"),
            ((None, a + 4, F64, 2, G, j, None, None), "aligned"),
            ((None, a, F64, 2, G, None, m + 4, None), "aligned"),
        ]
        for args, why in cases:
            msg = _refusal(fn, *args)
            assert msg.startswith(name + ": ") and why in msg, (args, msg)


def test_host_argument_checks():
    from inversekinematicsann_b200 import _native
    from inversekinematicsann_b200.engine import IkEngine
    check = IkEngine._jacobian_args
    ang = np.zeros((5, 4))
    a, code, out = check(ang, "geometric", False, None)
    assert code == _native.IKB_JAC_GEOMETRIC and out.shape == (5, 6, 4) and out.dtype == np.float64
    a, code, out = check(ang.astype(np.float32), "position", True, None)
    assert code == _native.IKB_JAC_POSITION and out.shape == (5, 3, 4) and out.dtype == np.float32
    assert check(ang, None, True, None)[2] is None
    given = np.empty((5, 6, 4))
    assert check(ang, "geometric", False, given)[2] is given
    ro = np.empty((5, 6, 4))
    ro.flags.writeable = False
    bad = [
        (ValueError, ang, "matrices", False, None),
        (ValueError, ang, None, False, None),                              # nothing asked for
        (ValueError, ang, None, True, np.empty((5, 6, 4))),                # out without a Jacobian
        (ValueError, np.zeros((5, 3)), "geometric", False, None),
        (ValueError, ang, "geometric", False, np.empty((5, 3, 4))),
        (ValueError, ang, "position", False, np.empty((6, 3, 4))),
        (TypeError, ang, "geometric", False, np.empty((5, 6, 4), dtype=np.float32)),
        (ValueError, ang, "geometric", False, np.empty((5, 6, 8))[:, :, ::2]),
        (ValueError, ang, "geometric", False, ro),
        (TypeError, ang, "geometric", False, [[0.0] * 4] * 6),
    ]
    for exc, a_, what, manip, out_ in bad:
        with pytest.raises(exc):
            check(a_, what, manip, out_)


def test_device_argument_checks_before_any_device_use():
    """An engine object without a handle: every refusal below happens before the library is called."""
    import torch
    from inversekinematicsann_b200.engine import IkEngine
    eng = IkEngine.__new__(IkEngine)
    eng.device = 0
    cpu = torch.zeros(4, 4, dtype=torch.float64)
    with pytest.raises(ValueError):
        eng.jacobian_device(cpu, None, "matrices", None)
    with pytest.raises(TypeError):
        eng.jacobian_device(cpu, torch.empty(4, 6, 4, dtype=torch.float64), "geometric", None)
    with pytest.raises(TypeError):
        eng.jacobian_device(np.zeros((4, 4)), None, "geometric", None)
