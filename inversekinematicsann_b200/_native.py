"""ctypes binding of csrc/libikb200.so (the C ABI declared in include/ikb200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``csrc/Makefile``.  If it is missing
this module raises -- there is deliberately no Python or NumPy fallback for the compute path.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IKB200_LIB") or os.path.join(_HERE, "csrc", "libikb200.so")  # override: A/B builds

IKB_OK = 0
IKB_ERR_INVALID, IKB_ERR_CUDA, IKB_ERR_NO_MODEL, IKB_ERR_UNSUPPORTED = -1, -2, -3, -4
IKB_F32, IKB_F64 = 0, 1
IKB_FABRIK_F64, IKB_FABRIK_F32 = 0, 1
IKB_MLP_FP32_SIMT, IKB_MLP_FP16X3_TC, IKB_MLP_FP16X3_TS = 0, 1, 2
IKB_CHAIN_MAX_POINTS = 256
IKB_FK_MATRICES, IKB_FK_JOINTS = 0, 1
IKB_JAC_GEOMETRIC, IKB_JAC_POSITION = 0, 1
IKB_AIK_POSE, IKB_AIK_POSITION_PITCH = 0, 1

# every symbol include/ikb200.h declares (tests check that the built library exports them all)
EXPORTED_SYMBOLS = [
    "ikb_engine_create", "ikb_engine_destroy", "ikb_last_error", "ikb_version", "ikb_device_count",
    "ikb_stats_reset", "ikb_stats_fetch",
    "ikb_check_limits_device", "ikb_check_limits_host",
    "ikb_fabrik_solve_device", "ikb_fabrik_solve_host", "ikb_fabrik_calculate_host",
    "ikb_fabrik_chain_device", "ikb_fabrik_chain_host",
    "ikb_fk_device", "ikb_fk_host", "ikb_fk_chain_host", "ikb_fk_transforms_device", "ikb_fk_transforms_host",
    "ikb_jacobian_device", "ikb_jacobian_host", "ikb_dls_refine_device", "ikb_dls_refine_host",
    "ikb_dls_pose_refine_device", "ikb_dls_pose_refine_host", "ikb_analytic_ik_device", "ikb_analytic_ik_host",
    "ikb_mlp_load", "ikb_ann_solve_device", "ikb_ann_solve_host",
    "ikb_generate_device", "ikb_microbench_fma", "ikb_launch_count",
    "ikb_host_alloc", "ikb_host_free", "ikb_host_register", "ikb_host_unregister",
    "ikb_copy_pipeline_host", "ikb_theoretical_fma_peak",
]


class NativeLibraryError(RuntimeError):
    """libikb200.so is missing or unusable (no CPU fallback exists)."""


class IkbConfig(ctypes.Structure):
    _fields_ = [("dh", ctypes.c_double * 16), ("links", ctypes.c_double * 4),
                ("limits", ctypes.c_double * 6), ("tol", ctypes.c_double),
                ("max_iter", ctypes.c_int32), ("device", ctypes.c_int32)]


class IkbStats(ctypes.Structure):
    _fields_ = [("n_solved", ctypes.c_int64), ("sum_iterations", ctypes.c_int64),
                ("n_iter_capped", ctypes.c_int64), ("first_out_of_limits", ctypes.c_int64),
                ("first_zero_division", ctypes.c_int64), ("first_domain_error", ctypes.c_int64),
                ("first_fk_angle_range", ctypes.c_int64), ("sum_fk_error", ctypes.c_double),
                ("n_fk_error", ctypes.c_int64)]


_LIB = None


def load():
    """Load libikb200.so once and declare the prototypes of include/ikb200.h."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C inversekinematicsann_b200/csrc`).  There is no CPU fallback.")
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as exc:
        raise NativeLibraryError(f"cannot load {LIB_PATH}: {exc}") from exc
    vp, i32, i64, dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
    engine = ctypes.c_void_p
    stats_p = ctypes.POINTER(IkbStats)
    dbl_p = ctypes.POINTER(dbl)
    protos = {
        "ikb_engine_create": (i32, [ctypes.POINTER(IkbConfig), ctypes.POINTER(engine)]),
        "ikb_engine_destroy": (None, [engine]),
        "ikb_last_error": (ctypes.c_char_p, [engine]),
        "ikb_version": (ctypes.c_char_p, []),
        "ikb_device_count": (i32, []),
        "ikb_stats_reset": (i32, [engine, vp]),
        "ikb_stats_fetch": (i32, [engine, vp, stats_p]),
        "ikb_check_limits_device": (i32, [engine, vp, i32, i64, vp]),
        "ikb_check_limits_host": (i32, [engine, vp, i32, i64, ctypes.POINTER(i64)]),
        "ikb_fabrik_solve_device": (i32, [engine, vp, i32, i64, vp, i32, vp, vp, i32, i32, vp]),
        "ikb_fabrik_solve_host": (i32, [engine, vp, i32, i64, vp, i32, vp, vp, i32, i32, stats_p]),
        "ikb_fabrik_calculate_host": (i32, [engine, vp, i64, vp, i64, vp, vp, stats_p]),
        "ikb_fabrik_chain_device": (i32, [engine, ctypes.c_int32, vp, dbl, ctypes.c_int32, vp, i64, vp, i64, vp, vp,
                                          vp]),
        "ikb_fabrik_chain_host": (i32, [engine, ctypes.c_int32, vp, dbl, ctypes.c_int32, vp, i64, vp, i64, vp, vp,
                                        stats_p]),
        "ikb_fk_device": (i32, [engine, vp, i32, i64, vp, vp, i32, vp, vp]),
        "ikb_fk_host": (i32, [engine, vp, i32, i64, vp, vp, i32, vp, stats_p]),
        "ikb_fk_chain_host": (i32, [engine, vp, vp, ctypes.POINTER(i32)]),
        "ikb_fk_transforms_device": (i32, [engine, vp, i32, i64, i32, vp, vp]),
        "ikb_fk_transforms_host": (i32, [engine, vp, i32, i64, i32, vp, stats_p]),
        "ikb_jacobian_device": (i32, [engine, vp, i32, i64, i32, vp, vp, vp]),
        "ikb_jacobian_host": (i32, [engine, vp, i32, i64, i32, vp, vp, stats_p]),
        "ikb_dls_refine_device": (i32, [engine, vp, i32, i64, vp, i64, vp, i32, dbl, dbl, ctypes.c_int32, vp, vp, vp]),
        "ikb_dls_refine_host": (i32, [engine, vp, i32, i64, vp, i64, vp, i32, dbl, dbl, ctypes.c_int32, vp, vp,
                                      stats_p]),
        "ikb_dls_pose_refine_device": (i32, [engine, vp, i32, i64, vp, i64, vp, i32, dbl_p, dbl, dbl, ctypes.c_int32,
                                             vp, vp, vp]),
        "ikb_dls_pose_refine_host": (i32, [engine, vp, i32, i64, vp, i64, vp, i32, dbl_p, dbl, dbl, ctypes.c_int32, vp,
                                           vp, stats_p]),
        "ikb_analytic_ik_device": (i32, [engine, i32, vp, i32, i64, vp, i64, vp, i32, vp, vp]),
        "ikb_analytic_ik_host": (i32, [engine, i32, vp, i32, i64, vp, i64, vp, i32, vp, stats_p]),
        "ikb_mlp_load": (i32, [engine, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32),
                               ctypes.POINTER(vp), ctypes.POINTER(vp), vp, vp, vp, vp]),
        "ikb_ann_solve_device": (i32, [engine, vp, i32, i64, vp, vp, i32, i32, vp]),
        "ikb_ann_solve_host": (i32, [engine, vp, i32, i64, vp, vp, i32, i32, stats_p]),
        "ikb_generate_device": (i32, [engine, i32, vp, i32, i64, i64, vp, i32, ctypes.c_uint64, vp]),
        "ikb_microbench_fma": (i32, [engine, i32, ctypes.POINTER(dbl)]),
        "ikb_launch_count": (i64, [engine]),
        "ikb_host_alloc": (i32, [engine, ctypes.c_size_t, ctypes.POINTER(vp)]),
        "ikb_host_free": (i32, [engine, vp]),
        "ikb_host_register": (i32, [engine, vp, ctypes.c_size_t, i32]),
        "ikb_host_unregister": (i32, [engine, vp]),
        "ikb_copy_pipeline_host": (i32, [engine, vp, i64, i64, vp, i64]),
        "ikb_theoretical_fma_peak": (i32, [engine, i32, ctypes.POINTER(dbl)]),
    }
    for name, (res, args) in protos.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise NativeLibraryError(f"{LIB_PATH} does not export {name}; rebuild it") from exc
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib
