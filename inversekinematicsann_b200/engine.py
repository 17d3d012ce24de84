"""IkEngine -- Python owner of one ``ikb_engine`` handle (one CUDA device).

Host code only marshals: list / ndarray / torch tensor -> contiguous buffer -> C ABI call.  All
arithmetic of the hot path happens in libikb200.so on the GPU.
"""
import ctypes
import math
from dataclasses import dataclass

import numpy as np

from . import _native
from ._native import NativeLibraryError  # noqa: F401  (re-exported)


@dataclass
class IkStats:
    """Mirror of ``ikb_stats`` (include/ikb200.h)."""
    n_solved: int = 0
    sum_iterations: int = 0
    n_iter_capped: int = 0
    first_out_of_limits: int = -1
    first_zero_division: int = -1
    first_domain_error: int = -1
    first_fk_angle_range: int = -1
    sum_fk_error: float = 0.0
    n_fk_error: int = 0

    @classmethod
    def from_c(cls, s):
        return cls(**{name: getattr(s, name) for name, _ in s._fields_})

    @property
    def mean_fk_error(self):
        return self.sum_fk_error / self.n_fk_error if self.n_fk_error else float("nan")


def _np_dtype_code(arr):
    if arr.dtype == np.float32:
        return _native.IKB_F32
    if arr.dtype == np.float64:
        return _native.IKB_F64
    raise TypeError(f"unsupported dtype {arr.dtype}; use float32 or float64")


def _is_torch_tensor(x):
    return type(x).__module__.startswith("torch") and hasattr(x, "data_ptr")


def _torch_dtype_code(t):
    import torch
    if t.dtype == torch.float32:
        return _native.IKB_F32
    if t.dtype == torch.float64:
        return _native.IKB_F64
    raise TypeError(f"unsupported dtype {t.dtype}; use float32 or float64")


def _torch_stream_ptr(device_index):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device_index).cuda_stream)


class IkEngine:
    """One engine per process and GPU.  Not thread-safe (as the reference is not, SURVEY 8b)."""

    def __init__(self, dh_matrix, joints_distances, workspace_limits, max_err=0.001,
                 max_iterations_num=100, device=0):
        dh = np.asarray(dh_matrix, dtype=np.float64)
        if dh.shape != (4, 4):
            raise ValueError(f"the DH table must be 4 rows x 4 joints (theta, epsilon, a, alpha), got {dh.shape}")
        links = np.asarray(joints_distances, dtype=np.float64)
        if links.shape != (4,):
            raise ValueError("Input vectors should have equal lengths!")  # fabrik.py:46-48
        lim = workspace_limits
        if isinstance(lim, dict):
            lim = [lim["x"][0], lim["x"][1], lim["y"][0], lim["y"][1], lim["z"][0], lim["z"][1]]
        lim = np.asarray(lim, dtype=np.float64).reshape(6)
        self._lib = _native.load()
        cfg = _native.IkbConfig()
        cfg.dh[:] = dh.reshape(-1).tolist()
        cfg.links[:] = links.tolist()
        cfg.limits[:] = lim.tolist()
        cfg.tol = float(max_err)
        cfg.max_iter = int(max_iterations_num)
        cfg.device = int(device)
        self.device = int(device)
        self._handle = ctypes.c_void_p()
        rc = self._lib.ikb_engine_create(ctypes.byref(cfg), ctypes.byref(self._handle))
        if rc != _native.IKB_OK:
            self._handle = ctypes.c_void_p()
            msg = self._lib.ikb_last_error(None).decode()
            raise RuntimeError(f"ikb_engine_create failed ({rc}): {msg}")
        self._mlp_keepalive = None

    # ---- lifetime -------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_handle", None) and self._handle.value:
            self._lib.ikb_engine_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc, what):
        if rc != _native.IKB_OK:
            msg = self._lib.ikb_last_error(self._handle).decode()
            if rc == _native.IKB_ERR_INVALID:
                raise ValueError(f"{what}: {msg}")
            raise RuntimeError(f"{what} failed ({rc}): {msg}")

    @property
    def launch_count(self):
        return int(self._lib.ikb_launch_count(self._handle))

    @staticmethod
    def version():
        return _native.load().ikb_version().decode()

    # ---- statistics -----------------------------------------------------------------------------
    def stats_reset(self, stream=None):
        self._check(self._lib.ikb_stats_reset(self._handle, stream), "ikb_stats_reset")

    def stats_fetch(self, stream=None):
        s = _native.IkbStats()
        self._check(self._lib.ikb_stats_fetch(self._handle, stream, ctypes.byref(s)), "ikb_stats_fetch")
        return IkStats.from_c(s)

    # ---- host-buffer entry points (NumPy) ---------------------------------------------------------
    @staticmethod
    def _rows(a, cols, what):
        a = np.ascontiguousarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        if a.ndim != 2 or a.shape[1] != cols:
            raise ValueError(f"{what} must have shape (n, {cols}), got {a.shape}")
        return a

    @staticmethod
    def _check_out(out, n, cols, dtypes, what):
        """A caller-supplied result buffer goes to the C ABI as a raw pointer: refuse anything the library would
        write past or into the wrong places (wrong shape, strided view, read-only, unexpected dtype)."""
        if not isinstance(out, np.ndarray):
            raise TypeError(f"{what} must be a numpy.ndarray, not {type(out).__name__}")
        want = (n, cols) if cols else (n,)
        if out.shape != want:
            raise ValueError(f"{what} must have shape {want}, got {out.shape}")
        if out.dtype not in dtypes:
            raise TypeError(f"{what} must have dtype {' or '.join(np.dtype(d).name for d in dtypes)}, got {out.dtype}")
        if not out.flags.c_contiguous:
            raise ValueError(f"{what} must be C-contiguous")
        if not out.flags.writeable:
            raise ValueError(f"{what} is read-only")
        return out

    def check_limits(self, xyz):
        """reference inverse.py:26-35 -> index of the first out-of-box row or -1."""
        xyz = self._rows(xyz, 3, "points")
        first = ctypes.c_int64(-1)
        self._check(self._lib.ikb_check_limits_host(self._handle, xyz.ctypes.data, _np_dtype_code(xyz),
                                                    xyz.shape[0], ctypes.byref(first)), "ikb_check_limits_host")
        return int(first.value)

    def fabrik_solve(self, xyz, out=None, out_dtype=np.float64, precision="f64", return_iters=False,
                     return_fk_error=False, fk_stats=False):
        """reference inverse.py:115-139 on an (n, 3) array.  Returns (angles[n,4], stats[, iters][, fk_error]);
        `return_fk_error` adds ||FK(angles) - target|| per row from the solver's own epilogue (no second pass),
        `fk_stats` only its sum / count in `stats`."""
        xyz = self._rows(xyz, 3, "points")
        n = xyz.shape[0]
        if out is None:
            out = np.empty((n, 4), dtype=out_dtype)
        self._check_out(out, n, 4, (np.float32, np.float64), "out")
        iters = np.empty(n, dtype=np.int32) if return_iters else None
        fk_err = np.empty(n, dtype=out.dtype) if return_fk_error else None
        s = _native.IkbStats()
        prec = _choice(_FABRIK_PRECISIONS, precision, "precision")
        self._check(self._lib.ikb_fabrik_solve_host(
            self._handle, xyz.ctypes.data, _np_dtype_code(xyz), n, out.ctypes.data, _np_dtype_code(out),
            iters.ctypes.data if return_iters else None, fk_err.ctypes.data if return_fk_error else None,
            int(bool(fk_stats)), prec, ctypes.byref(s)), "ikb_fabrik_solve_host")
        res = (out, IkStats.from_c(s))
        if return_iters:
            res += (iters,)
        if return_fk_error:
            res += (fk_err,)
        return res

    @staticmethod
    def _chain_links(links):
        links = np.ascontiguousarray(links, dtype=np.float64)
        if links.ndim != 1 or not 1 <= links.shape[0] <= _native.IKB_CHAIN_MAX_POINTS:
            raise ValueError(f"a chain needs 1..{_native.IKB_CHAIN_MAX_POINTS} link lengths, got shape {links.shape}")
        return links

    def fabrik_chain(self, links, tol, max_iter, init, goals):
        """reference fabrik.py:44-67 on J-point chains: J = len(links) link lengths, init (J,3) or (n,J,3), goals (n,3).
        Returns (chains[n,J,3], iters[n], stats); stats.first_zero_division >= 0 marks a zero-length segment."""
        links = self._chain_links(links)
        J = links.shape[0]
        init = np.ascontiguousarray(init, dtype=np.float64)
        goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(-1, 3)
        n = goals.shape[0]
        if init.shape == (J, 3):
            n_init = 1
        elif init.shape == (n, J, 3):
            n_init = n
        else:
            raise ValueError(f"initial chains must have shape ({J}, 3) or ({n}, {J}, 3), got {init.shape}")
        chain = np.empty((n, J, 3), dtype=np.float64)
        iters = np.empty(n, dtype=np.int32)
        s = _native.IkbStats()
        self._check(self._lib.ikb_fabrik_chain_host(self._handle, J, links.ctypes.data, float(tol), int(max_iter),
                                                    init.ctypes.data, n_init, goals.ctypes.data, n, chain.ctypes.data,
                                                    iters.ctypes.data, ctypes.byref(s)), "ikb_fabrik_chain_host")
        return chain, iters, IkStats.from_c(s)

    def fabrik_calculate(self, init, goals):
        """reference fabrik.py:44-67 for explicit 4-point chains with the engine's links, tolerance and iteration cap.
        init: (4,3) or (n,4,3); goals (n,3)."""
        init = np.ascontiguousarray(init, dtype=np.float64)
        goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(-1, 3)
        n = goals.shape[0]
        n_init = 1 if init.ndim == 2 else init.shape[0]
        init = init.reshape(n_init, 4, 3)
        chain = np.empty((n, 4, 3), dtype=np.float64)
        iters = np.empty(n, dtype=np.int32)
        s = _native.IkbStats()
        self._check(self._lib.ikb_fabrik_calculate_host(self._handle, init.ctypes.data, n_init, goals.ctypes.data,
                                                        n, chain.ctypes.data, iters.ctypes.data, ctypes.byref(s)),
                    "ikb_fabrik_calculate_host")
        return chain, iters, IkStats.from_c(s)

    def fk(self, angles, targets=None, want_pos=True, want_err=None):
        """reference forward.py:73-94 batched: (positions[n,3] | None, errors[n] | None, stats)."""
        angles = self._rows(angles, 4, "angles")
        n = angles.shape[0]
        if want_err is None:
            want_err = targets is not None
        tg = None
        if targets is not None:
            tg = self._rows(targets, 3, "targets")
            if tg.shape[0] != n:
                raise ValueError("angles and targets must have the same number of rows")
        pos = np.empty((n, 3), dtype=angles.dtype) if want_pos else None
        err = np.empty(n, dtype=angles.dtype) if want_err else None
        s = _native.IkbStats()
        self._check(self._lib.ikb_fk_host(
            self._handle, angles.ctypes.data, _np_dtype_code(angles), n,
            pos.ctypes.data if want_pos else None, tg.ctypes.data if tg is not None else None,
            _np_dtype_code(tg) if tg is not None else _native.IKB_F64,
            err.ctypes.data if want_err else None, ctypes.byref(s)), "ikb_fk_host")
        return pos, err, IkStats.from_c(s)

    def fk_chain(self, angles):
        """All four cumulative 4x4 DH matrices of one angle set -> (ndarray[4,4,4], status)."""
        ang = np.ascontiguousarray(angles, dtype=np.float64).reshape(4)
        chain = np.empty((4, 4, 4), dtype=np.float64)
        status = ctypes.c_int32(0)
        self._check(self._lib.ikb_fk_chain_host(self._handle, ang.ctypes.data, chain.ctypes.data,
                                                ctypes.byref(status)), "ikb_fk_chain_host")
        return chain, int(status.value)

    def mlp_load(self, weights, biases, mean_x, scale_x, mean_y, scale_y):
        """reference ann.py:78-85: upload Keras Dense kernels (in, out) + biases and both scalers."""
        ws = [np.ascontiguousarray(w, dtype=np.float32) for w in weights]
        bs = [np.ascontiguousarray(b, dtype=np.float32).reshape(-1) for b in biases]
        if len(ws) != len(bs) or not ws:
            raise ValueError("weights and biases must be non-empty lists of equal length")
        dims = [ws[0].shape[0]] + [w.shape[1] for w in ws]
        for l, (w, b) in enumerate(zip(ws, bs)):
            if w.ndim != 2 or w.shape[0] != dims[l] or b.shape[0] != w.shape[1]:
                raise ValueError(f"layer {l}: kernel {w.shape} / bias {b.shape} do not chain")
        n_layers = len(ws)
        dims_c = (ctypes.c_int32 * (n_layers + 1))(*dims)
        w_ptrs = (ctypes.c_void_p * n_layers)(*[w.ctypes.data for w in ws])
        b_ptrs = (ctypes.c_void_p * n_layers)(*[b.ctypes.data for b in bs])
        sc = [np.ascontiguousarray(v, dtype=np.float64).reshape(-1) for v in (mean_x, scale_x, mean_y, scale_y)]
        if [v.shape[0] for v in sc] != [3, 3, 4, 4]:
            raise ValueError("scalers must have 3 (x) and 4 (y) features")
        self._check(self._lib.ikb_mlp_load(self._handle, n_layers, dims_c, w_ptrs, b_ptrs,
                                           sc[0].ctypes.data, sc[1].ctypes.data, sc[2].ctypes.data,
                                           sc[3].ctypes.data), "ikb_mlp_load")
        self.mlp_dims = dims
        self.mlp_macs_per_row = int(sum(a * b for a, b in zip(dims[:-1], dims[1:])))

    def ann_solve(self, xyz, out=None, mode="fp32", return_fk_error=False, fk_stats=False):
        """reference ann.py:70-76 on an (n, 3) array -> (angles float32 [n,4], stats[, fk_error float32 [n]])."""
        mode_code = _choice(_MLP_MODES, mode, "mode")
        xyz = self._rows(xyz, 3, "points")
        n = xyz.shape[0]
        if out is None:
            out = np.empty((n, 4), dtype=np.float32)
        self._check_out(out, n, 4, (np.float32,), "out")  # Keras / sklearn return float32 (ann.py:70-76)
        fk_err = np.empty(n, dtype=np.float32) if return_fk_error else None
        s = _native.IkbStats()
        self._check(self._lib.ikb_ann_solve_host(self._handle, xyz.ctypes.data, _np_dtype_code(xyz), n,
                                                 out.ctypes.data, fk_err.ctypes.data if return_fk_error else None,
                                                 int(bool(fk_stats)), mode_code, ctypes.byref(s)),
                    "ikb_ann_solve_host")
        return (out, IkStats.from_c(s), fk_err) if return_fk_error else (out, IkStats.from_c(s))

    def microbench_fma(self, dtype="f64"):
        out = ctypes.c_double(0.0)
        code = _native.IKB_F64 if dtype == "f64" else _native.IKB_F32
        self._check(self._lib.ikb_microbench_fma(self._handle, code, ctypes.byref(out)), "ikb_microbench_fma")
        return float(out.value)

    def theoretical_fma_peak(self, dtype="f64"):
        """SMs x FMA lanes x 2 x max SM clock, in TFLOP/s (the number the live microbenchmark is checked against)."""
        out = ctypes.c_double(0.0)
        code = _native.IKB_F64 if dtype == "f64" else _native.IKB_F32
        self._check(self._lib.ikb_theoretical_fma_peak(self._handle, code, ctypes.byref(out)), "ikb_theoretical_fma_peak")
        return float(out.value)

    # ---- pinned host buffers ----------------------------------------------------------------------
    def pinned_buffer(self, nbytes):
        """Page-locked host memory from the library (cudaHostAlloc by this thread on this engine's device)."""
        return PinnedBuffer(self, nbytes)

    def pinned_empty(self, shape, dtype=np.float32):
        """An ndarray in page-locked memory: what `ikine(..., out=)` wants for large trajectories."""
        shape = tuple(int(v) for v in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        nbytes = max(1, int(np.prod(shape)) * np.dtype(dtype).itemsize)
        return self.pinned_buffer(nbytes).array(dtype, shape)

    def copy_pipeline(self, src, dst):
        """The host pipeline of the solve calls with the kernels removed (bench.py's copy ceiling): `src` rows go
        to the device, `dst` rows come back; both are (n, c) arrays of at most 32 bytes per row."""
        n = src.shape[0] if src is not None else dst.shape[0]
        for a in (src, dst):
            if a is not None and (a.shape[0] != n or not a.flags.c_contiguous):
                raise ValueError("src and dst must be C-contiguous with the same number of rows")
        self._check(self._lib.ikb_copy_pipeline_host(
            self._handle, src.ctypes.data if src is not None else None,
            src.strides[0] if src is not None else 0, n,
            dst.ctypes.data if dst is not None else None, dst.strides[0] if dst is not None else 0),
            "ikb_copy_pipeline_host")

    # ---- device-buffer entry points (torch CUDA tensors; async on torch's current stream) ---------
    def _dev_rows(self, t, cols, what):
        if not _is_torch_tensor(t) or not t.is_cuda:
            raise TypeError(f"{what} must be a CUDA torch tensor")
        if t.device.index != self.device:
            raise ValueError(f"{what} lives on cuda:{t.device.index}, the engine on cuda:{self.device}")
        if t.dim() != 2 or t.shape[1] != cols or not t.is_contiguous():
            raise ValueError(f"{what} must be a contiguous (n, {cols}) tensor")
        return t

    @staticmethod
    def _same_rows(a, b, what):
        if a.shape[0] != b.shape[0]:
            raise ValueError(f"{what} has {b.shape[0]} rows for {a.shape[0]} points")

    def _dev_vec(self, t, n, dtype, what):
        if not _is_torch_tensor(t) or not t.is_cuda or t.device.index != self.device:
            raise TypeError(f"{what} must be a CUDA torch tensor on cuda:{self.device}")
        if str(t.dtype) != dtype or t.numel() != n or not t.is_contiguous():
            raise ValueError(f"{what} must be a contiguous {dtype} tensor with {n} elements")
        return t

    def fabrik_solve_device(self, xyz, out, iters=None, precision="f64", fk_err=None, fk_stats=False):
        xyz = self._dev_rows(xyz, 3, "points")
        out = self._dev_rows(out, 4, "angles")
        self._same_rows(xyz, out, "angles")
        if iters is not None:
            self._dev_vec(iters, xyz.shape[0], "torch.int32", "iters")
        if fk_err is not None:
            self._dev_vec(fk_err, xyz.shape[0], str(out.dtype), "fk_err")
        prec = _choice(_FABRIK_PRECISIONS, precision, "precision")
        self._check(self._lib.ikb_fabrik_solve_device(
            self._handle, xyz.data_ptr(), _torch_dtype_code(xyz), xyz.shape[0], out.data_ptr(),
            _torch_dtype_code(out), iters.data_ptr() if iters is not None else None,
            fk_err.data_ptr() if fk_err is not None else None, int(bool(fk_stats)), prec,
            _torch_stream_ptr(self.device)), "ikb_fabrik_solve_device")

    def fabrik_chain_device(self, links, tol, max_iter, init, goals, out, iters=None):
        """fabrik_chain on float64 CUDA tensors of this engine's device, enqueued on torch's current stream (no
        synchronisation): init (J,3) or (n,J,3), goals (n,3), out (n,J,3), iters int32 (n,) or None.  Statistics
        accumulate in the engine's block (stats_fetch_torch)."""
        links = self._chain_links(links)
        J = links.shape[0]
        goals = self._dev_rows(goals, 3, "goals")
        n = goals.shape[0]
        for t, what in ((init, "init"), (goals, "goals"), (out, "out")):
            self._dev_vec(t, t.numel() if _is_torch_tensor(t) else -1, "torch.float64", what)
        if tuple(init.shape) == (J, 3):
            n_init = 1
        elif tuple(init.shape) == (n, J, 3):
            n_init = n
        else:
            raise ValueError(f"init must have shape ({J}, 3) or ({n}, {J}, 3), got {tuple(init.shape)}")
        if tuple(out.shape) != (n, J, 3):
            raise ValueError(f"out must have shape ({n}, {J}, 3), got {tuple(out.shape)}")
        if iters is not None:
            self._dev_vec(iters, n, "torch.int32", "iters")
        self._check(self._lib.ikb_fabrik_chain_device(
            self._handle, J, links.ctypes.data, float(tol), int(max_iter), init.data_ptr(), n_init, goals.data_ptr(), n,
            out.data_ptr(), iters.data_ptr() if iters is not None else None, _torch_stream_ptr(self.device)),
            "ikb_fabrik_chain_device")

    def ann_solve_device(self, xyz, out, mode="fp32", fk_err=None, fk_stats=False):
        mode_code = _choice(_MLP_MODES, mode, "mode")
        xyz = self._dev_rows(xyz, 3, "points")
        out = self._dev_rows(out, 4, "angles")
        self._same_rows(xyz, out, "angles")
        if str(out.dtype) != "torch.float32":
            raise TypeError(f"angles must be float32 (Keras / sklearn return float32), got {out.dtype}")
        if fk_err is not None:
            self._dev_vec(fk_err, xyz.shape[0], "torch.float32", "fk_err")
        self._check(self._lib.ikb_ann_solve_device(
            self._handle, xyz.data_ptr(), _torch_dtype_code(xyz), xyz.shape[0], out.data_ptr(),
            fk_err.data_ptr() if fk_err is not None else None, int(bool(fk_stats)),
            mode_code, _torch_stream_ptr(self.device)), "ikb_ann_solve_device")

    def fk_device(self, angles, targets=None, pos=None, err=None):
        angles = self._dev_rows(angles, 4, "angles")
        n = angles.shape[0]
        if targets is not None:
            self._same_rows(angles, self._dev_rows(targets, 3, "targets"), "targets")
        if pos is not None:
            self._same_rows(angles, self._dev_rows(pos, 3, "pos"), "pos")
            if pos.dtype != angles.dtype:
                raise TypeError("pos must have the angles' dtype")
        if err is not None:
            if targets is None:
                raise ValueError("err needs targets")
            self._dev_vec(err, n, str(angles.dtype), "err")
        self._check(self._lib.ikb_fk_device(
            self._handle, angles.data_ptr(), _torch_dtype_code(angles), angles.shape[0],
            pos.data_ptr() if pos is not None else None,
            targets.data_ptr() if targets is not None else None,
            _torch_dtype_code(targets) if targets is not None else _native.IKB_F64,
            err.data_ptr() if err is not None else None, _torch_stream_ptr(self.device)), "ikb_fk_device")

    def check_limits_device(self, xyz):
        xyz = self._dev_rows(xyz, 3, "points")
        self._check(self._lib.ikb_check_limits_device(self._handle, xyz.data_ptr(), _torch_dtype_code(xyz),
                                                      xyz.shape[0], _torch_stream_ptr(self.device)),
                    "ikb_check_limits_device")

    def stats_fetch_torch(self):
        return self.stats_fetch(_torch_stream_ptr(self.device))

    def stats_reset_torch(self):
        self.stats_reset(_torch_stream_ptr(self.device))


class PinnedBuffer:
    """nbytes of page-locked host memory owned by libikb200 (ikb_host_alloc / ikb_host_free).  Views handed out by
    `array()` / `view()` keep the buffer alive; it is freed when the last of them is gone."""

    def __init__(self, engine, nbytes):
        self._engine, self.nbytes = engine, int(nbytes)
        ptr = ctypes.c_void_p()
        engine._check(engine._lib.ikb_host_alloc(engine._handle, self.nbytes, ctypes.byref(ptr)), "ikb_host_alloc")
        self.ptr = ptr.value
        raw = (ctypes.c_ubyte * self.nbytes).from_address(self.ptr)
        raw._ikb_owner = self            # every NumPy view's base chain ends at `raw`
        self._bytes = np.frombuffer(raw, dtype=np.uint8)

    def array(self, dtype, shape, offset=0):
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        if offset < 0 or offset + count * dtype.itemsize > self.nbytes:
            raise ValueError("view exceeds the pinned buffer")
        return self._bytes[offset: offset + count * dtype.itemsize].view(dtype).reshape(shape)

    def view(self, offset=0, nbytes=None):
        nbytes = self.nbytes - offset if nbytes is None else nbytes
        return memoryview(self._bytes[offset: offset + nbytes])

    def close(self):
        if getattr(self, "ptr", None) and getattr(self._engine, "_handle", None) and self._engine._handle.value:
            self._engine._lib.ikb_host_free(self._engine._handle, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_MLP_MODES = {"fp32": _native.IKB_MLP_FP32_SIMT, "fp16x3": _native.IKB_MLP_FP16X3_TC,
              "fp16x3_ts": _native.IKB_MLP_FP16X3_TS}
_FABRIK_PRECISIONS = {"f64": _native.IKB_FABRIK_F64, "f32": _native.IKB_FABRIK_F32}


def _choice(table, key, what):
    try:
        return table[key]
    except (KeyError, TypeError):
        raise ValueError(f"{what} must be one of {sorted(table)}, got {key!r}") from None

# algorithmic work per unit (SURVEY 8d / DESIGN.md), used by bench.py's roofline arithmetic
FABRIK_FLOPS_PER_ITERATION = 114
FABRIK_FLOPS_EPILOGUE = 126


def fabrik_algorithmic_flops(sum_iterations, n):
    return FABRIK_FLOPS_PER_ITERATION * sum_iterations + FABRIK_FLOPS_EPILOGUE * n


def is_finite_number(x):
    return isinstance(x, (int, float)) and math.isfinite(x)
