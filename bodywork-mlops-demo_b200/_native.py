"""ctypes binding of libb2gram.so (include/b2gram.h) and a thin object wrapper.

There is deliberately no CPU implementation behind these calls: if the shared library is missing
or no B200 is visible, every compute entry point raises ``RuntimeError`` (the reference's error
style, stage_1_train_model.py:74,125,142).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Tuple

import numpy as np

from . import build as _build

F32, BF16, F64 = 0, 1, 2
MEM_DEVICE, MEM_HOST = 0, 1
KERNEL_AUTO, KERNEL_SIMT, KERNEL_TCGEN05, KERNEL_NARROW = 0, 1, 2, 3
PRECISION_SPLIT, PRECISION_BF16 = 0, 1
E_SINGULAR = -4
E_COMM = -5
EXCHANGE_NONE, EXCHANGE_NCCL, EXCHANGE_PEER = 0, 1, 2
ABI_VERSION = 2
MAX_D = 128

_c_i64 = C.c_int64
_vp = C.c_void_p

# name -> (restype, argtypes); mirrors include/b2gram.h one to one
_SIGNATURES = {
    "b2_abi_version": (C.c_int, []),
    "b2_last_error": (C.c_char_p, []),
    "b2_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "b2_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "b2_ctx_destroy": (C.c_int, [_vp]),
    "b2_ctx_sync": (C.c_int, [_vp]),
    "b2_ctx_info": (C.c_int, [_vp, C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "b2_ctx_set_kernel": (C.c_int, [_vp, C.c_int]),
    "b2_ctx_set_drain_rows": (C.c_int, [_vp, C.c_int]),
    "b2_ctx_set_precision": (C.c_int, [_vp, C.c_int]),
    "b2_ctx_set_sm_limit": (C.c_int, [_vp, C.c_int]),
    "b2_dev_alloc": (C.c_int, [_vp, C.c_size_t, C.POINTER(_vp)]),
    "b2_dev_free": (C.c_int, [_vp, _vp]),
    "b2_host_alloc": (C.c_int, [_vp, C.c_size_t, C.POINTER(_vp)]),
    "b2_host_free": (C.c_int, [_vp, _vp]),
    "b2_copy_h2d": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "b2_copy_d2h": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "b2_dev_memset": (C.c_int, [_vp, _vp, C.c_int, C.c_size_t]),
    "b2_gram_reset": (C.c_int, [_vp, C.c_int]),
    "b2_gram_accumulate": (C.c_int, [_vp, _vp, C.c_int, _vp, _c_i64, C.c_int, _c_i64, C.c_int, _vp, C.c_int]),
    "b2_gram_allreduce": (C.c_int, [_vp]),
    "b2_gram_export": (C.c_int, [_vp, _vp, C.POINTER(_c_i64)]),
    "b2_gram_import": (C.c_int, [_vp, _vp, C.c_int]),
    "b2_gram_kernels": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "b2_split_mask": (C.c_int, [_c_i64, _c_i64, C.c_uint32, _vp]),
    "b2_copy_d2d": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "b2_pack_columns": (C.c_int, [_vp, _vp, C.c_int, _c_i64, C.c_int, _vp]),
    "b2_upload_columns": (C.c_int, [_vp, _vp, _vp, C.c_int, _c_i64, C.c_int, _vp]),
    "b2_fit": (C.c_int, [_vp, _vp, C.c_int, _vp, _c_i64, C.c_int, _c_i64, C.c_int, _vp, C.c_int, C.c_double, C.c_int, _vp,
                         C.POINTER(C.c_double)]),
    "b2_solve": (C.c_int, [_vp, C.c_double, C.c_int, _vp, C.POINTER(C.c_double)]),
    "b2_solve_eigvals": (C.c_int, [_vp, C.c_double, C.c_int, _vp, C.POINTER(C.c_int), C.POINTER(_c_i64)]),
    "b2_solve_spectral": (C.c_int, [_vp, C.c_double, C.c_int, _vp, C.POINTER(C.c_double), _vp, C.POINTER(C.c_int)]),
    "b2_score": (C.c_int, [_vp, _vp, C.c_int, _c_i64, C.c_int, _c_i64, C.c_int, _vp, C.c_double, _vp, _vp,
                           C.c_int, _vp, _vp]),
    "b2_score_allreduce": (C.c_int, [_vp, _vp]),
    "b2_metrics": (C.c_int, [_vp, _vp, _vp, C.c_int, _c_i64, C.c_int, _vp]),
    "b2_synth_tranche": (C.c_int, [_vp, C.c_uint64, _c_i64, C.c_int, C.c_double, C.c_double, _vp, _vp,
                                   C.POINTER(_c_i64)]),
    "b2_synth": (C.c_int, [_vp, C.c_uint64, _c_i64, _c_i64, C.c_int, _c_i64, C.c_int, C.c_double, C.c_double,
                           C.c_double, _vp, _vp]),
    "b2_comm_unique_id": (C.c_int, [C.c_char_p]),
    "b2_comm_init": (C.c_int, [_vp, C.c_int, C.c_int, C.c_char_p]),
    "b2_comm_destroy": (C.c_int, [_vp]),
    "b2_comm_barrier": (C.c_int, [_vp]),
    "b2_comm_p2p_export": (C.c_int, [_vp, C.c_char_p]),
    "b2_comm_p2p_attach": (C.c_int, [_vp, C.c_int, C.c_int, C.c_char_p]),
    "b2_comm_p2p_detach": (C.c_int, [_vp]),
    "b2_comm_p2p_attach_local": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(_vp)]),
    "b2_comm_set_timeout_ms": (C.c_int, [_vp, _c_i64]),
    "b2_comm_info": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "b2_ctx_stats": (C.c_int, [_vp, C.POINTER(_c_i64)]),
    "b2_timer_start": (C.c_int, [_vp]),
    "b2_timer_stop": (C.c_int, [_vp, C.POINTER(C.c_double)]),
    "b2_last_kernel_ms": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "b2_launch_count": (C.c_int, [_vp, C.POINTER(_c_i64)]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)
_lib = None


def lib_path() -> str:
    return os.environ.get("B2_LIB_PATH") or _build.LIB_PATH   # B2_LIB_PATH: development override (kernel variants)


def load():
    """dlopen libb2gram.so (building it first if the sources are newer and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if os.environ.get("B2_LIB_PATH"):
        pass
    elif not os.path.exists(path) or (_build.is_stale() and os.environ.get("B2_NO_REBUILD") != "1"):
        try:
            _build.build()
        except Exception as exc:  # pragma: no cover - only without nvcc
            if not os.path.exists(path):
                raise RuntimeError(f"libb2gram.so is missing and could not be built: {exc}") from exc
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.b2_abi_version() != ABI_VERSION:
        raise RuntimeError("libb2gram.so ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    return load().b2_last_error().decode("utf-8", "replace")


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")


def device_count() -> int:
    n = C.c_int(0)
    rc = load().b2_device_count(C.byref(n))
    return int(n.value) if rc == 0 else 0


def pack_columns(columns) -> np.ndarray:
    """1-D host columns (all float64 or all float32, any stride) -> row-major float32 (n, d): ``b2_pack_columns``, the
    multi-threaded gather + conversion ``Context.upload_columns`` runs on the way to the device (host only, no GPU)."""
    cols = [np.asarray(c) for c in columns]
    if not cols or any(c.ndim != 1 or c.shape != cols[0].shape or c.dtype != cols[0].dtype for c in cols) \
            or cols[0].dtype not in (np.dtype(np.float64), np.dtype(np.float32)):
        raise RuntimeError("pack_columns: 1-D columns of one length and one dtype (float64 or float32) expected")
    n, d = int(cols[0].shape[0]), len(cols)
    out = np.empty((n, d), dtype=np.float32)
    ptrs = (C.c_void_p * d)(*[c.ctypes.data for c in cols])
    strides = (C.c_int64 * d)(*[c.strides[0] if n > 1 else c.itemsize for c in cols])
    _check(load().b2_pack_columns(C.cast(ptrs, C.c_void_p), C.cast(strides, C.c_void_p),
                                  F64 if cols[0].dtype == np.float64 else F32, n, d, out.ctypes.data), "b2_pack_columns")
    return out


def to_bf16_bits(a: np.ndarray) -> np.ndarray:
    """float32 -> bfloat16 bit patterns (uint16), round-to-nearest-even."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    rounded = u + (np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1)))
    return (rounded >> np.uint32(16)).astype(np.uint16)


def from_bf16_bits(b: np.ndarray) -> np.ndarray:
    return (b.astype(np.uint32) << np.uint32(16)).view(np.float32)


class DeviceArray:
    """A caller-owned HBM buffer: pointer + shape + element kind ('f32' | 'bf16' | 'u8' | 'f64')."""
    _ITEM = {"f32": 4, "bf16": 2, "u8": 1, "f64": 8}
    _NP = {"f32": np.float32, "bf16": np.uint16, "u8": np.uint8, "f64": np.float64}

    def __init__(self, ctx: "Context", shape: Tuple[int, ...], kind: str):
        self.ctx, self.shape, self.kind = ctx, tuple(int(s) for s in shape), kind
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self._ITEM[kind]
        p = _vp()
        _check(load().b2_dev_alloc(ctx._h, max(self.nbytes, 1), C.byref(p)), "b2_dev_alloc")
        self.ptr = p.value

    def copy_from(self, host: np.ndarray) -> "DeviceArray":
        host = np.ascontiguousarray(host, dtype=self._NP[self.kind])
        assert host.nbytes == self.nbytes, (host.nbytes, self.nbytes)
        _check(load().b2_copy_h2d(self.ctx._h, self.ptr, host.ctypes.data, self.nbytes), "b2_copy_h2d")
        return self

    def to_host(self) -> np.ndarray:
        out = np.empty(self.shape, dtype=self._NP[self.kind])
        _check(load().b2_copy_d2h(self.ctx._h, out.ctypes.data, self.ptr, self.nbytes), "b2_copy_d2h")
        return out

    def free(self) -> None:
        if self.ptr:
            load().b2_dev_free(self.ctx._h, self.ptr)
            self.ptr = None

    def __del__(self):  # best effort
        try:
            if self.ptr and self.ctx._h:
                self.free()
        except Exception:
            pass


class PinnedArray:
    """Pinned host memory exposed as a numpy array (for B2_MEM_HOST streaming)."""

    def __init__(self, ctx: "Context", shape, dtype):
        self.ctx = ctx
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
        p = _vp()
        _check(load().b2_host_alloc(ctx._h, max(nbytes, 1), C.byref(p)), "b2_host_alloc")
        self.ptr = p.value
        buf = (C.c_char * max(nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)

    def free(self) -> None:
        if self.ptr:
            self.array = None
            load().b2_host_free(self.ctx._h, self.ptr)
            self.ptr = None


def _x_kind(X) -> Tuple[int, int, int, int, int]:
    """(ptr, x_dtype, mem_kind, n, d) of a DeviceArray or a host ndarray (float32 / uint16-as-bf16)."""
    if isinstance(X, DeviceArray):
        if X.kind not in ("f32", "bf16"):
            raise RuntimeError("X must be f32 or bf16")
        n, d = X.shape
        return X.ptr, (F32 if X.kind == "f32" else BF16), MEM_DEVICE, n, d
    if not isinstance(X, np.ndarray) or X.ndim != 2 or not X.flags.c_contiguous:
        raise RuntimeError("host X must be a C-contiguous 2-D ndarray")
    if X.dtype == np.float32:
        return X.ctypes.data, F32, MEM_HOST, X.shape[0], X.shape[1]
    if X.dtype == np.uint16:
        return X.ctypes.data, BF16, MEM_HOST, X.shape[0], X.shape[1]
    raise RuntimeError(f"host X must be float32 (or uint16 bf16 bits), got {X.dtype}")


def _vec_ptr(v, kind: str, mem_kind: int, n: int, what: str) -> Optional[int]:
    if v is None:
        return None
    if isinstance(v, DeviceArray):
        if mem_kind != MEM_DEVICE or v.kind != kind or int(np.prod(v.shape)) != n:
            raise RuntimeError(f"{what}: device buffer of kind {kind} and length {n} expected")
        return v.ptr
    want = np.float32 if kind == "f32" else np.uint8
    if mem_kind != MEM_HOST or not isinstance(v, np.ndarray) or v.dtype != want or v.size != n \
            or not v.flags.c_contiguous:
        raise RuntimeError(f"{what}: contiguous host {want.__name__} array of length {n} expected")
    return v.ctypes.data


class Context:
    """One GPU: streams, the fp64 statistic S, scratch, (optionally) one NCCL communicator."""

    def __init__(self, device: int = 0):
        self._h = None
        h = _vp()
        _check(load().b2_ctx_create(int(device), C.byref(h)), "b2_ctx_create")
        self._h = h.value
        self.device = int(device)
        self.d = 0
        self.kernel = KERNEL_AUTO
        self.precision = PRECISION_SPLIT
        self.serial = 0      # bumped whenever the resident statistic S changes owner / content (estimators check it)

    # -- lifecycle -----------------------------------------------------------------------------
    def close(self) -> None:
        if self._h:
            load().b2_ctx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def sync(self) -> None:
        _check(load().b2_ctx_sync(self._h), "b2_ctx_sync")

    def info(self) -> dict:
        name = C.create_string_buffer(128)
        sm, hbm = C.c_int(0), C.c_size_t(0)
        _check(load().b2_ctx_info(self._h, name, 128, C.byref(sm), C.byref(hbm)), "b2_ctx_info")
        return {"name": name.value.decode(), "sm_count": sm.value, "hbm_bytes": hbm.value}

    def set_kernel(self, kernel: int) -> None:
        _check(load().b2_ctx_set_kernel(self._h, int(kernel)), "b2_ctx_set_kernel")
        self.kernel = int(kernel)

    def set_precision(self, precision: int) -> None:
        """PRECISION_SPLIT (default, bf16 hi+lo operands) or PRECISION_BF16 (single bf16 operand, 'bf16-accum')."""
        _check(load().b2_ctx_set_precision(self._h, int(precision)), "b2_ctx_set_precision")
        self.precision = int(precision)

    def set_sm_limit(self, n_sms: int) -> None:
        _check(load().b2_ctx_set_sm_limit(self._h, int(n_sms)), "b2_ctx_set_sm_limit")

    def set_drain_rows(self, rows: int) -> None:
        _check(load().b2_ctx_set_drain_rows(self._h, int(rows)), "b2_ctx_set_drain_rows")

    # -- buffers ----------------------------------------------------------------------------------
    def empty(self, shape, kind: str) -> DeviceArray:
        return DeviceArray(self, tuple(np.atleast_1d(shape)), kind)

    def to_device(self, host: np.ndarray, kind: Optional[str] = None) -> DeviceArray:
        if kind is None:
            kind = {np.dtype(np.float32): "f32", np.dtype(np.uint16): "bf16", np.dtype(np.uint8): "u8",
                    np.dtype(np.float64): "f64"}[host.dtype]
        return DeviceArray(self, host.shape, kind).copy_from(host)

    def upload_columns(self, columns) -> DeviceArray:
        """1-D host columns (all float64 or all float32, any stride -- what ``DataFrame[c].to_numpy()`` returns) -> a
        row-major float32 (n, d) DeviceArray: gathered, converted and copied by ``b2_upload_columns`` (host threads + a
        pinned ring), without the transposing copy / conversion passes of ``DataFrame.to_numpy``."""
        cols = [np.asarray(c) for c in columns]
        if not cols or any(c.ndim != 1 or c.shape != cols[0].shape or c.dtype != cols[0].dtype for c in cols) \
                or cols[0].dtype not in (np.dtype(np.float64), np.dtype(np.float32)):
            raise RuntimeError("upload_columns: 1-D columns of one length and one dtype (float64 or float32) expected")
        n, d = int(cols[0].shape[0]), len(cols)
        out = DeviceArray(self, (n, d), "f32")
        ptrs = (C.c_void_p * d)(*[c.ctypes.data for c in cols])
        strides = (C.c_int64 * d)(*[c.strides[0] if n > 1 else c.itemsize for c in cols])
        _check(load().b2_upload_columns(self._h, C.cast(ptrs, C.c_void_p), C.cast(strides, C.c_void_p),
                                        F64 if cols[0].dtype == np.float64 else F32, n, d, out.ptr), "b2_upload_columns")
        return out

    def copy_bandwidth_gbs(self, nbytes: int = 2 << 30, reps: int = 10) -> float:
        """This GPU's device-to-device copy bandwidth (read + write bytes per second, GB/s, best of ``reps``) -- the quantity
        MEASURED_PEAKS.json holds for the pool; boxes differ."""
        a, b = DeviceArray(self, (nbytes,), "u8"), DeviceArray(self, (nbytes,), "u8")
        try:
            _check(load().b2_dev_memset(self._h, a.ptr, 1, nbytes), "b2_dev_memset")
            best = 0.0
            for _ in range(reps + 2):
                self.sync(); self.timer_start()
                _check(load().b2_copy_d2d(self._h, b.ptr, a.ptr, nbytes), "b2_copy_d2d")
                ms = self.timer_stop()
                best = max(best, 2.0 * nbytes / (ms * 1e-3) / 1e9)
            return best
        finally:
            a.free(); b.free()

    def pinned(self, shape, dtype) -> PinnedArray:
        return PinnedArray(self, tuple(np.atleast_1d(shape)), dtype)

    # -- Gram ----------------------------------------------------------------------------------------
    def gram_reset(self, d: int) -> None:
        _check(load().b2_gram_reset(self._h, int(d)), "b2_gram_reset")
        self.d = int(d)
        self.serial += 1

    def gram_accumulate(self, X, y, row_mask=None, mask_keep: int = 1) -> None:
        ptr, xdt, mk, n, d = _x_kind(X)
        if self.d == 0:
            self.gram_reset(d)
        yp = _vec_ptr(y, "f32", mk, n, "y")
        mp = _vec_ptr(row_mask, "u8", mk, n, "row_mask")
        self.serial += 1
        _check(load().b2_gram_accumulate(self._h, ptr, xdt, yp, n, d, d, mk, mp, int(mask_keep)),
               "b2_gram_accumulate")

    def gram_allreduce(self) -> None:
        _check(load().b2_gram_allreduce(self._h), "b2_gram_allreduce")

    def gram_export(self) -> np.ndarray:
        S = np.empty((self.d + 2, self.d + 2), dtype=np.float64)
        n = _c_i64(0)
        _check(load().b2_gram_export(self._h, S.ctypes.data, C.byref(n)), "b2_gram_export")
        return S

    def gram_import(self, S: np.ndarray) -> None:
        S = np.ascontiguousarray(S, dtype=np.float64)
        d = S.shape[0] - 2
        _check(load().b2_gram_import(self._h, S.ctypes.data, d), "b2_gram_import")
        self.d = d
        self.serial += 1

    def gram_kernels(self) -> int:
        """OR of ``1 << KERNEL_*`` of the kernels that added to the resident statistic since the last reset / import /
        fit (b2_gram_kernels)."""
        k = C.c_int(0)
        _check(load().b2_gram_kernels(self._h, C.byref(k)), "b2_gram_kernels")
        return int(k.value)

    def fit(self, X, y, row_mask=None, mask_keep: int = 1, alpha: float = 0.0,
            fit_intercept: bool = True) -> Tuple[np.ndarray, float]:
        """The whole fit in one C call (b2_fit): reset + accumulate + all-reduce + solve.  Device-resident rows on the
        tensor-core path run as four launches (shift sample, Gram, finalize + peer scatter, gather + solve).  Raises ``np.linalg.LinAlgError`` on a rank-deficient Gram."""
        ptr, xdt, mk, n, d = _x_kind(X)
        yp = _vec_ptr(y, "f32", mk, n, "y")
        mp = _vec_ptr(row_mask, "u8", mk, n, "row_mask")
        coef = np.empty(d, dtype=np.float64)
        b0 = C.c_double(0.0)
        rc = load().b2_fit(self._h, ptr, xdt, yp, n, d, d, mk, mp, int(mask_keep), float(alpha),
                           int(bool(fit_intercept)), coef.ctypes.data, C.byref(b0))
        self.d = int(d)
        self.serial += 1
        if rc == E_SINGULAR:
            raise np.linalg.LinAlgError(last_error())
        _check(rc, "b2_fit")
        return coef, float(b0.value)

    # -- solve -----------------------------------------------------------------------------------------
    def solve(self, alpha: float = 0.0, fit_intercept: bool = True) -> Tuple[np.ndarray, float]:
        """Cholesky solve; raises ``np.linalg.LinAlgError`` when the Gram matrix is rank deficient."""
        coef = np.empty(self.d, dtype=np.float64)
        b0 = C.c_double(0.0)
        rc = load().b2_solve(self._h, float(alpha), int(bool(fit_intercept)), coef.ctypes.data, C.byref(b0))
        if rc == E_SINGULAR:
            raise np.linalg.LinAlgError(last_error())
        _check(rc, "b2_solve")
        return coef, float(b0.value)

    def solve_spectral(self, cond: float = 1e-6, fit_intercept: bool = True):
        coef = np.empty(self.d, dtype=np.float64)
        sing = np.empty(self.d, dtype=np.float64)
        b0, rank = C.c_double(0.0), C.c_int(0)
        _check(load().b2_solve_spectral(self._h, float(cond), int(bool(fit_intercept)), coef.ctypes.data,
                                        C.byref(b0), sing.ctypes.data, C.byref(rank)), "b2_solve_spectral")
        return coef, float(b0.value), sing, int(rank.value)

    def solve_eigvals(self, cond: float = 1e-6, fit_intercept: bool = True):
        """(singular_, rank_, rows): sqrt of the eigenvalues of the centred Gram, descending (no eigenvectors)."""
        sing = np.empty(self.d, dtype=np.float64)
        rank, rows = C.c_int(0), _c_i64(0)
        _check(load().b2_solve_eigvals(self._h, float(cond), int(bool(fit_intercept)), sing.ctypes.data,
                                       C.byref(rank), C.byref(rows)), "b2_solve_eigvals")
        return sing, int(rank.value), int(rows.value)

    # -- scoring ------------------------------------------------------------------------------------------
    def metrics(self, y_actual, y_predicted) -> np.ndarray:
        """The ten reductions of b2_score on two vectors (b2_metrics); float64 inputs stay float64."""
        if isinstance(y_actual, DeviceArray):
            if not isinstance(y_predicted, DeviceArray) or y_actual.kind != y_predicted.kind \
                    or y_actual.kind not in ("f32", "f64") or y_actual.nbytes != y_predicted.nbytes:
                raise RuntimeError("metrics: two device vectors of the same kind (f32 / f64) and length expected")
            n = int(np.prod(y_actual.shape))
            a_ptr, p_ptr, dt, mk = y_actual.ptr, y_predicted.ptr, (F32 if y_actual.kind == "f32" else F64), MEM_DEVICE
        else:
            dtype = np.float32 if (np.asarray(y_actual).dtype == np.float32 and
                                   np.asarray(y_predicted).dtype == np.float32) else np.float64
            a = np.ascontiguousarray(np.asarray(y_actual, dtype=dtype).ravel())
            p = np.ascontiguousarray(np.asarray(y_predicted, dtype=dtype).ravel())
            if a.size != p.size:
                raise ValueError(f"Found input variables with inconsistent numbers of samples: [{a.size}, {p.size}]")
            n, a_ptr, p_ptr, dt, mk = a.size, a.ctypes.data, p.ctypes.data, (F32 if dtype == np.float32 else F64), MEM_HOST
        stats = np.zeros(10, dtype=np.float64)
        _check(load().b2_metrics(self._h, a_ptr, p_ptr, dt, n, mk, stats.ctypes.data), "b2_metrics")
        return stats

    def score(self, X, coef: np.ndarray, intercept: float, y=None, row_mask=None, mask_keep: int = 1,
              want_yhat: bool = True, out=None):
        """Returns (yhat | None, stats | None); stats = the ten reductions of include/b2gram.h b2_score
        ([sum_ape, sse, sum_y, sum_yy, max_abs_res, rows, sum_p, sum_pp, sum_yp, max_ape]).
        ``out``: a preallocated prediction buffer (DeviceArray f32 for device rows, float32 ndarray for host rows)
        to write into instead of allocating one per call."""
        ptr, xdt, mk, n, d = _x_kind(X)
        coef = np.ascontiguousarray(coef, dtype=np.float64).ravel()
        if coef.size != d:
            raise RuntimeError(f"coef has {coef.size} entries, X has {d} columns")
        yp = _vec_ptr(y, "f32", mk, n, "y")
        mp = _vec_ptr(row_mask, "u8", mk, n, "row_mask")
        yhat = None
        yhat_ptr = None
        if out is not None:
            if mk == MEM_DEVICE:
                if not isinstance(out, DeviceArray) or out.kind != "f32" or int(np.prod(out.shape)) != n:
                    raise RuntimeError("out must be an f32 DeviceArray with one element per row")
                yhat, yhat_ptr = out, out.ptr
            else:
                if not (isinstance(out, np.ndarray) and out.dtype == np.float32 and out.size == n
                        and out.flags.c_contiguous):
                    raise RuntimeError("out must be a C-contiguous float32 ndarray with one element per row")
                yhat, yhat_ptr = out, out.ctypes.data
        elif want_yhat:
            yhat = self.empty((n,), "f32") if mk == MEM_DEVICE else np.empty(n, dtype=np.float32)
            yhat_ptr = yhat.ptr if mk == MEM_DEVICE else yhat.ctypes.data
        stats = np.zeros(10, dtype=np.float64) if y is not None else None
        _check(load().b2_score(self._h, ptr, xdt, n, d, d, mk, coef.ctypes.data, float(intercept), yp, mp,
                               int(mask_keep), yhat_ptr, stats.ctypes.data if stats is not None else None),
               "b2_score")
        return yhat, stats

    def score_allreduce(self, stats: np.ndarray) -> np.ndarray:
        stats = np.ascontiguousarray(stats, dtype=np.float64)
        _check(load().b2_score_allreduce(self._h, stats.ctypes.data), "b2_score_allreduce")
        return stats

    # -- synthetic rows --------------------------------------------------------------------------------------
    def synth(self, n: int, d: int, seed: int = 1234, row_offset: int = 0, kind: str = "f32", alpha: float = 1.0,
              beta: float = 0.5, sigma: float = 10.0) -> Tuple[DeviceArray, DeviceArray]:
        X = self.empty((n, d), kind)
        y = self.empty((n,), "f32")
        _check(load().b2_synth(self._h, int(seed), int(row_offset), int(n), int(d), int(d),
                               F32 if kind == "f32" else BF16, float(alpha), float(beta), float(sigma), X.ptr,
                               y.ptr), "b2_synth")
        return X, y

    def synth_tranche(self, n: int, day: int, seed: int = 1234, beta: float = 0.5, sigma: float = 10.0):
        """One reference tranche (stage_3's generate_dataset: alpha(day), y >= 0 filter) -> (X (n, 1), y (n,), n_kept);
        the buffers hold ``n`` rows, the first ``n_kept`` are valid."""
        X = self.empty((n, 1), "f32")
        y = self.empty((n,), "f32")
        kept = _c_i64(0)
        _check(load().b2_synth_tranche(self._h, int(seed), int(n), int(day), float(beta), float(sigma), X.ptr, y.ptr,
                                       C.byref(kept)), "b2_synth_tranche")
        return X, y, int(kept.value)

    def stats(self) -> dict:
        out = (_c_i64 * 3)()
        _check(load().b2_ctx_stats(self._h, out), "b2_ctx_stats")
        return {"fused_fits": int(out[0]), "peer_exchanges": int(out[1]), "launches": int(out[2])}

    # -- multi-GPU -----------------------------------------------------------------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        _check(load().b2_comm_unique_id(buf), "b2_comm_unique_id")
        return buf.raw

    def comm_init(self, n_ranks: int, rank: int, uid: bytes) -> None:
        _check(load().b2_comm_init(self._h, int(n_ranks), int(rank), C.create_string_buffer(uid, 128)),
               "b2_comm_init")

    def comm_p2p_export(self) -> bytes:
        """CUDA-IPC handle (64 bytes) of this rank's exchange buffer for the one-shot peer-memory all-reduce."""
        buf = C.create_string_buffer(64)
        _check(load().b2_comm_p2p_export(self._h, buf), "b2_comm_p2p_export")
        return buf.raw

    def comm_p2p_attach(self, n_ranks: int, rank: int, handles) -> None:
        """``handles``: the exported handles of all ranks, in rank order."""
        blob = b"".join(handles)
        if len(blob) != 64 * n_ranks:
            raise RuntimeError("need one 64-byte handle per rank")
        _check(load().b2_comm_p2p_attach(self._h, int(n_ranks), int(rank), C.create_string_buffer(blob, len(blob))),
               "b2_comm_p2p_attach")

    def comm_p2p_detach(self) -> None:
        _check(load().b2_comm_p2p_detach(self._h), "b2_comm_p2p_detach")

    @staticmethod
    def comm_p2p_attach_local(contexts) -> None:
        """Peer exchange between contexts of this process (rank = position in ``contexts``)."""
        arr = (_vp * len(contexts))(*[c._h for c in contexts])
        for rank, c in enumerate(contexts):
            _check(load().b2_comm_p2p_attach_local(c._h, len(contexts), rank, arr), "b2_comm_p2p_attach_local")

    def comm_set_timeout_ms(self, ms: int) -> None:
        _check(load().b2_comm_set_timeout_ms(self._h, int(ms)), "b2_comm_set_timeout_ms")

    def comm_info(self) -> dict:
        n, r, e = C.c_int(0), C.c_int(0), C.c_int(0)
        _check(load().b2_comm_info(self._h, C.byref(n), C.byref(r), C.byref(e)), "b2_comm_info")
        return {"n_ranks": n.value, "rank": r.value, "exchange": {0: "none", 1: "nccl", 2: "p2p"}[e.value]}

    def comm_barrier(self) -> None:
        _check(load().b2_comm_barrier(self._h), "b2_comm_barrier")

    # -- timing ---------------------------------------------------------------------------------------------------
    def timer_start(self) -> None:
        _check(load().b2_timer_start(self._h), "b2_timer_start")

    def timer_stop(self) -> float:
        ms = C.c_double(0.0)
        _check(load().b2_timer_stop(self._h, C.byref(ms)), "b2_timer_stop")
        return float(ms.value)

    def last_kernel_ms(self) -> Tuple[float, int]:
        ms, n = C.c_double(0.0), C.c_int(0)
        _check(load().b2_last_kernel_ms(self._h, C.byref(ms), C.byref(n)), "b2_last_kernel_ms")
        return float(ms.value), int(n.value)

    def launch_count(self) -> int:
        n = _c_i64(0)
        _check(load().b2_launch_count(self._h, C.byref(n)), "b2_launch_count")
        return int(n.value)
