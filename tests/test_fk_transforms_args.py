"""Argument checks of the batched DH transforms that need no GPU (the rest is in test_gpu_fk_transforms.py)."""
import numpy as np
import pytest


def test_out_buffer_checks_take_the_per_row_shape():
    from inversekinematicsann_b200.engine import IkEngine
    out = np.empty((5, 4, 4, 4))
    assert IkEngine._check_out(out, 5, (4, 4, 4), (np.float64,), "out") is out
    with pytest.raises(ValueError):
        IkEngine._check_out(np.empty((5, 4, 3)), 5, (4, 4, 4), (np.float64,), "out")
    with pytest.raises(TypeError):
        IkEngine._check_out(np.empty((5, 4, 3), dtype=np.float32), 5, (4, 3), (np.float64,), "out")
    ro = np.empty((5, 4, 3))
    ro.flags.writeable = False
    with pytest.raises(ValueError):
        IkEngine._check_out(ro, 5, (4, 3), (np.float64,), "out")


def test_c_abi_rejects_a_null_engine():
    from inversekinematicsann_b200 import _native
    lib = _native.load()
    buf = np.zeros(64)
    for fn in (lib.ikb_fk_transforms_host, lib.ikb_fk_transforms_device):
        assert fn(None, buf.ctypes.data, _native.IKB_F64, 1, _native.IKB_FK_MATRICES, buf.ctypes.data,
                  None) == _native.IKB_ERR_INVALID
