"""ctypes binding of include/shifu_b200.h (the C-ABI a JNI shim binds the same way, INTEGRATION.md).

No compute lives here: every call forwards to libshifu_b200.so.  If the library has not been built the
import fails loudly - there is no Python / CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

# A step runs on up to five streams (main, side, two exchange streams, descriptor prefetch); with the default of 8 hardware
# queues CUDA maps several of them onto one queue and their kernels falsely serialise (an exchange kernel that waits for
# its peers then holds back an unrelated GEMM).  Read by the driver when the context is created, i.e. at the first CUDA call.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libshifu_b200.so")

SB_MAX_HIDDEN = 32
SB_NCCL_ID_BYTES = 128
ACT_SIGMOID, ACT_TANH, ACT_RELU, ACT_LEAKYRELU, ACT_NONE = 0, 1, 2, 3, -1
LOSS_MSE, LOSS_SIGMOID_CE = 0, 1
OPT_ADADELTA, OPT_ADAM, OPT_SGD, OPT_MOMENTUM = 0, 1, 2, 3
PREC_FP32, PREC_BF16, PREC_FP32_TC, PREC_BF16X2 = 0, 1, 2, 3
SB_OK, SB_ERR_INVALID, SB_ERR_CUDA, SB_ERR_NCCL, SB_ERR_IO, SB_ERR_STATE, SB_ERR_FORMAT = 0, -1, -2, -3, -4, -5, -6


class NetDesc(C.Structure):
    _fields_ = [
        ("n_features", C.c_int32), ("n_hidden", C.c_int32),
        ("hidden", C.c_int32 * SB_MAX_HIDDEN), ("acts", C.c_int32 * SB_MAX_HIDDEN),
        ("loss", C.c_int32), ("optimizer", C.c_int32),
        ("learning_rate", C.c_float), ("rho", C.c_float), ("epsilon", C.c_float),
        ("beta1", C.c_float), ("beta2", C.c_float), ("momentum", C.c_float),
        ("max_batch", C.c_int32), ("precision", C.c_int32),
    ]


def make_desc(n_features: int, hidden: Sequence[int], acts: Sequence[int], loss: int = LOSS_MSE,
              optimizer: int = OPT_ADADELTA, learning_rate: float = 0.001, rho: float = 0.95, epsilon: float = 1e-8,
              beta1: float = 0.9, beta2: float = 0.999, momentum: float = 0.9, max_batch: int = 128,
              precision: int = PREC_FP32) -> NetDesc:
    if len(hidden) != len(acts):
        raise ValueError("hidden and acts must have the same length")
    if len(hidden) > SB_MAX_HIDDEN:
        raise ValueError("at most %d hidden layers" % SB_MAX_HIDDEN)
    d = NetDesc()
    d.n_features, d.n_hidden = int(n_features), len(hidden)
    for i, (h, a) in enumerate(zip(hidden, acts)):
        d.hidden[i], d.acts[i] = int(h), int(a)
    d.loss, d.optimizer = int(loss), int(optimizer)
    d.learning_rate, d.rho, d.epsilon = learning_rate, rho, epsilon
    d.beta1, d.beta2, d.momentum = beta1, beta2, momentum
    d.max_batch, d.precision = int(max_batch), int(precision)
    return d


class CellFlag(C.Structure):
    _fields_ = [("row", C.c_int64), ("slot", C.c_int32), ("len", C.c_int32), ("offset", C.c_int64)]


COL_SKIP, COL_TARGET, COL_WEIGHT = -1, -2, -3


class ShifuB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("[%d] %s" % (code, msg))
        self.code = code


_lib = None

# name -> (restype, argtypes); the single source of truth for tests/test_capi_symbols.py
_P = C.POINTER
_f32p, _f64p, _vp, _cp = _P(C.c_float), _P(C.c_double), C.c_void_p, C.c_char_p
PROTOTYPES = {
    "sb_version": (C.c_char_p, []),
    "sb_last_error": (C.c_char_p, []),
    "sb_device_count": (C.c_int, []),
    "sb_host_alloc": (C.c_int, [_P(_vp), C.c_uint64]),
    "sb_host_free": (C.c_int, [_vp]),
    "sb_nccl_unique_id": (C.c_int, [_vp]),
    "sb_trainer_create": (C.c_int, [_P(NetDesc), C.c_int, _vp, C.c_int, C.c_int, _P(_vp)]),
    "sb_trainer_destroy": (C.c_int, [_vp]),
    "sb_trainer_ipc_handle": (C.c_int, [_vp, _vp]),
    "sb_trainer_set_peer_handles": (C.c_int, [_vp, _vp, C.c_int32]),
    "sb_trainer_clear_peer_handles": (C.c_int, [_vp]),
    "sb_trainer_exchange_base": (C.c_void_p, [_vp]),
    "sb_trainer_set_peer_pointers": (C.c_int, [_vp, _P(_vp), C.c_int32]),
    "sb_trainer_param_count": (C.c_int64, [_vp]),
    "sb_trainer_set_params": (C.c_int, [_vp, _f32p, C.c_int64]),
    "sb_trainer_get_params": (C.c_int, [_vp, _f32p, C.c_int64]),
    "sb_trainer_init_xavier": (C.c_int, [_vp, C.c_uint64]),
    "sb_trainer_get_grads": (C.c_int, [_vp, _f32p, C.c_int64]),
    "sb_trainer_step": (C.c_int, [_vp, _f32p, _f32p, _f32p, C.c_int32, _f32p]),
    "sb_trainer_set_sparse": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int32]),
    "sb_trainer_step_sparse": (C.c_int, [_vp, _f32p, _P(C.c_int32), _f32p, _f32p, C.c_int32, _f32p]),
    "sb_trainer_predict_sparse": (C.c_int, [_vp, _f32p, _P(C.c_int32), C.c_int64, _f32p]),
    "sb_trainer_eval_loss_sparse": (C.c_int, [_vp, _f32p, _P(C.c_int32), _f32p, _f32p, C.c_int64, _f32p]),
    "sb_trainer_step_async": (C.c_int, [_vp, _f32p, _f32p, _f32p, C.c_int32]),
    "sb_trainer_accumulate": (C.c_int, [_vp, _f32p, _f32p, _f32p, C.c_int32, _f32p]),
    "sb_trainer_apply_accumulated": (C.c_int, [_vp]),
    "sb_trainer_apply_accumulated_mean": (C.c_int, [_vp, C.c_int64]),
    "sb_trainer_loss_resident": (C.c_int, [_vp, C.c_int64, C.c_int32, _f32p]),
    "sb_trainer_broadcast_state": (C.c_int, [_vp, C.c_int32]),
    "sb_trainer_load_dataset": (C.c_int, [_vp, _f32p, _f32p, _f32p, C.c_int64]),
    "sb_trainer_load_dataset_sparse": (C.c_int, [_vp, _f32p, _P(C.c_int32), _f32p, _f32p, C.c_int64]),
    "sb_trainer_step_resident": (C.c_int, [_vp, C.c_int64, C.c_int32, _f32p]),
    "sb_trainer_step_resident_async": (C.c_int, [_vp, C.c_int64, C.c_int32]),
    "sb_trainer_run_resident": (C.c_int, [_vp, C.POINTER(C.c_int64), C.c_int32, C.c_int32]),
    "sb_trainer_accumulate_resident": (C.c_int, [_vp, C.c_int64, C.c_int32, _f32p]),
    "sb_trainer_last_loss": (C.c_int, [_vp, _f32p]),
    "sb_trainer_loss_history": (C.c_int, [_vp, C.c_int64, C.c_int32, _f32p]),
    "sb_trainer_sync": (C.c_int, [_vp]),
    "sb_trainer_stream": (C.c_void_p, [_vp]),
    "sb_trainer_kernels_per_step": (C.c_int, [_vp, C.c_int32]),
    "sb_trainer_profile_step": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_char_p, C.c_int32, _f32p, C.c_int32, _P(C.c_int32)]),
    "sb_trainer_eval_loss": (C.c_int, [_vp, _f32p, _f32p, _f32p, C.c_int64, _f32p]),
    "sb_trainer_predict": (C.c_int, [_vp, _f32p, C.c_int64, _f32p]),
    "sb_trainer_save_checkpoint": (C.c_int, [_vp, _cp]),
    "sb_trainer_load_checkpoint": (C.c_int, [_vp, _cp]),
    "sb_trainer_global_step": (C.c_int64, [_vp]),
    "sb_trainer_export_savedmodel": (C.c_int, [_vp, _cp]),
    "sb_model_load": (C.c_int, [_cp, _cp, _cp, _cp, C.c_int, C.c_int, _P(_vp)]),
    "sb_model_create": (C.c_int, [_P(NetDesc), _f32p, C.c_int64, C.c_int, _P(_vp)]),
    "sb_model_destroy": (C.c_int, [_vp]),
    "sb_model_n_features": (C.c_int32, [_vp]),
    "sb_model_n_layers": (C.c_int32, [_vp]),
    "sb_model_score": (C.c_int, [_vp, _f32p, C.c_int64, _f32p]),
    "sb_model_score_row_f64": (C.c_int, [_vp, _f64p, C.c_int32, _f64p]),
    "sb_model_score_device": (C.c_int, [_vp, _vp, C.c_int64, _vp]),
    "sb_model_sync": (C.c_int, [_vp]),
    "sb_model_stream": (C.c_void_p, [_vp]),
    "sb_text_parse": (C.c_int, [_cp, C.c_int64, C.c_char, _P(C.c_int32), C.c_int32, C.c_int32, _f32p, _f32p, _f32p, C.c_int64,
                                _P(C.c_int64), _P(CellFlag), C.c_int64, _P(C.c_int64), C.c_int]),
    "sb_text_parse_device": (C.c_int, [_cp, C.c_int64, C.c_char, _P(C.c_int32), C.c_int32, C.c_int32, _P(_f32p), _P(_f32p), _P(_f32p),
                                       _P(C.c_int64), _P(CellFlag), C.c_int64, _P(C.c_int64), C.c_int, _f32p]),
    "sb_device_alloc_f32": (C.c_int, [_P(_f32p), C.c_int64, C.c_int]),
    "sb_device_free": (C.c_int, [_vp]),
    "sb_device_patch_f32": (C.c_int, [_f32p, C.c_int64, C.c_float]),
    "sb_device_read_f32": (C.c_int, [_f32p, C.c_int64, _f32p]),
    "sb_device_gather_rows": (C.c_int, [_f32p, C.c_int32, _P(C.c_int64), C.c_int64, _f32p, C.c_int]),
    "sb_debug_text_parse_host": (C.c_int, [_cp, C.c_int64, C.c_char, _P(C.c_int32), C.c_int32, C.c_int32, _f32p, _f32p, _f32p,
                                           C.c_int64, _P(C.c_int64), _P(CellFlag), C.c_int64, _P(C.c_int64)]),
    "sb_savedmodel_write": (C.c_int, [_cp, _P(NetDesc), _f32p, C.c_int64]),
    "sb_savedmodel_read": (C.c_int, [_cp, _cp, _cp, _cp, _P(NetDesc), _P(C.c_int32), _f32p, C.c_int64, _P(C.c_int64)]),
    "sb_debug_gemm_split": (C.c_int, [_f32p, _f32p, _f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int]),
    "sb_debug_gemm_bf16": (C.c_int, [_f32p, _f32p, _f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int]),
    "sb_debug_gemm_bf16_ex": (C.c_int, [_f32p, _f32p, _f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int]),
    "sb_debug_step_trace": (C.c_int, [_vp, C.POINTER(C.c_uint64), C.c_int32, C.c_char_p, C.c_int32, C.POINTER(C.c_int32)]),
    "sb_debug_gemm_bench": (C.c_int, [_f32p, _f32p, _f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int, C.c_int32, _f32p]),
    "sb_debug_gemm_bf16_cfg": (C.c_int, [_f32p, _f32p, _f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.c_int32, C.c_int]),
}


def lib():
    """Load libshifu_b200.so (once).  Raises ImportError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libshifu_b200.so is missing (%s). Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `python shifu-tensorflow_b200/build.py`. There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def check(status: int) -> None:
    if status != SB_OK:
        raise ShifuB200Error(status, lib().sb_last_error().decode("utf-8", "replace"))


def _f32(a, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None and a.shape != shape:
        a = a.reshape(shape)
    return a


def _ptr(a):
    if a is None:
        return None
    if hasattr(a, "ptr") and not isinstance(a, np.ndarray):      # DeviceArray
        return a.ptr
    return a.ctypes.data_as(_f32p)


class DeviceArray:
    """fp32 array that lives in GPU memory (library-owned; what sb_text_parse_device returns).  Accepted by
    Trainer.load_dataset / eval_loss / predict in place of a numpy array."""

    def __init__(self, ptr, shape, device: int = 0, owner: bool = True):
        self.ptr, self.shape, self.device, self._own = ptr, tuple(shape), device, owner

    @classmethod
    def empty(cls, shape, device: int = 0) -> "DeviceArray":
        p = _f32p()
        n = int(np.prod(shape))
        check(lib().sb_device_alloc_f32(C.byref(p), max(n, 1), device))
        return cls(p, shape, device)

    def __len__(self):
        return self.shape[0]

    @property
    def size(self) -> int:
        return int(np.prod(self.shape))

    def numpy(self) -> np.ndarray:
        out = np.empty(self.shape, np.float32)
        if self.size:
            check(lib().sb_device_read_f32(self.ptr, self.size, _ptr(out)))
        return out

    def patch(self, flat_index: int, value: float):
        check(lib().sb_device_patch_f32(self.ptr, int(flat_index), float(value)))

    def take_rows(self, rows) -> "DeviceArray":
        """rows (host int64 indices) gathered on the device into a new DeviceArray"""
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        n_cols = int(np.prod(self.shape[1:])) if len(self.shape) > 1 else 1
        out = DeviceArray.empty((len(rows),) + self.shape[1:], self.device)
        check(lib().sb_device_gather_rows(self.ptr, n_cols, rows.ctypes.data_as(_P(C.c_int64)), len(rows), out.ptr, self.device))
        return out

    def free(self):
        if self._own and self.ptr:
            lib().sb_device_free(C.cast(self.ptr, _vp))
        self.ptr = None

    __del__ = free


class Trainer:
    """Owns one sb_trainer_t.  X is [rows, n_features] float32, y / w are [rows] (or [rows,1])."""

    def __init__(self, desc: NetDesc, device: int = 0, nccl_id: Optional[bytes] = None, rank: int = 0, world: int = 1):
        self._h = C.c_void_p()
        self.desc = desc
        idbuf = None
        if nccl_id is not None:
            if len(nccl_id) != SB_NCCL_ID_BYTES:
                raise ValueError("nccl_id must be %d bytes" % SB_NCCL_ID_BYTES)
            idbuf = C.create_string_buffer(bytes(nccl_id), SB_NCCL_ID_BYTES)
        check(lib().sb_trainer_create(C.byref(desc), device, C.cast(idbuf, _vp) if idbuf is not None else None,
                                      rank, world, C.byref(self._h)))
        self.n_params = int(lib().sb_trainer_param_count(self._h))
        self.n_features = int(desc.n_features)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().sb_trainer_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- peer-memory gradient exchange (CUDA IPC) ----
    def ipc_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        check(lib().sb_trainer_ipc_handle(self._h, C.cast(buf, _vp)))
        return buf.raw

    def set_peer_handles(self, handles: Sequence[bytes]):
        blob = b"".join(handles)
        buf = C.create_string_buffer(blob, len(blob))
        check(lib().sb_trainer_set_peer_handles(self._h, C.cast(buf, _vp), len(handles)))

    def clear_peer_handles(self):
        check(lib().sb_trainer_clear_peer_handles(self._h))

    @property
    def exchange_base(self) -> int:
        return int(lib().sb_trainer_exchange_base(self._h) or 0)

    def set_peer_pointers(self, bases: Sequence[int]):
        """in-process peers: every rank's exchange_base in rank order"""
        arr = (C.c_void_p * len(bases))(*[C.c_void_p(int(b)) for b in bases])
        check(lib().sb_trainer_set_peer_pointers(self._h, arr, len(bases)))

    # ---- parameters ----
    def set_params(self, flat):
        flat = _f32(flat).reshape(-1)
        check(lib().sb_trainer_set_params(self._h, _ptr(flat), flat.size))

    def get_params(self) -> np.ndarray:
        out = np.empty(self.n_params, np.float32)
        check(lib().sb_trainer_get_params(self._h, _ptr(out), out.size))
        return out

    def get_grads(self) -> np.ndarray:
        out = np.empty(self.n_params, np.float32)
        check(lib().sb_trainer_get_grads(self._h, _ptr(out), out.size))
        return out

    def init_xavier(self, seed: int):
        check(lib().sb_trainer_init_xavier(self._h, seed))

    # ---- steps ----
    def _xyw(self, X, y, w):
        if isinstance(X, DeviceArray):          # device-resident set: pointers pass through
            rows = X.shape[0]
            if len(X.shape) != 2 or X.shape[1] != self.n_features or y.size != rows or (w is not None and w.size != rows):
                raise ValueError("device arrays must be X [rows, %d], y [rows], w [rows]" % self.n_features)
            return X, y, w, rows
        X = _f32(X)
        rows = X.shape[0]
        if X.ndim != 2 or X.shape[1] != self.n_features:
            raise ValueError("X must be [rows, %d]" % self.n_features)
        y = _f32(y).reshape(-1)
        w = None if w is None else _f32(w).reshape(-1)
        if y.size != rows or (w is not None and w.size != rows):
            raise ValueError("y / w length must equal rows")
        return X, y, w, rows

    def step(self, X, y, w=None) -> float:
        X, y, w, rows = self._xyw(X, y, w)
        loss = C.c_float()
        check(lib().sb_trainer_step(self._h, _ptr(X), _ptr(y), _ptr(w), rows, C.byref(loss)))
        return float(loss.value)

    # ---- wide+deep: dense block + index matrix (oracle/wide_deep.py) ----
    def set_sparse(self, n_dense: int, n_onehot: int, n_cat: int):
        check(lib().sb_trainer_set_sparse(self._h, n_dense, n_onehot, n_cat))
        self._sparse = (n_dense, n_cat)

    def _xd_idx(self, Xd, idx):
        n_dense, n_cat = self._sparse
        Xd = _f32(Xd)
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        if Xd.ndim != 2 or Xd.shape[1] != n_dense or idx.shape != (Xd.shape[0], n_cat):
            raise ValueError("Xd must be [rows, %d], idx [rows, %d]" % (n_dense, n_cat))
        return Xd, idx

    def step_sparse(self, Xd, idx, y, w=None) -> float:
        Xd, idx = self._xd_idx(Xd, idx)
        y = _f32(y).reshape(-1)
        w = None if w is None else _f32(w).reshape(-1)
        loss = C.c_float()
        check(lib().sb_trainer_step_sparse(self._h, _ptr(Xd), idx.ctypes.data_as(_P(C.c_int32)), _ptr(y), _ptr(w), Xd.shape[0],
                                           C.byref(loss)))
        return float(loss.value)

    def predict_sparse(self, Xd, idx) -> np.ndarray:
        Xd, idx = self._xd_idx(Xd, idx)
        out = np.empty(Xd.shape[0], np.float32)
        check(lib().sb_trainer_predict_sparse(self._h, _ptr(Xd), idx.ctypes.data_as(_P(C.c_int32)), Xd.shape[0], _ptr(out)))
        return out

    def eval_loss_sparse(self, Xd, idx, y, w=None) -> float:
        Xd, idx = self._xd_idx(Xd, idx)
        y = _f32(y).reshape(-1)
        w = None if w is None else _f32(w).reshape(-1)
        loss = C.c_float()
        check(lib().sb_trainer_eval_loss_sparse(self._h, _ptr(Xd), idx.ctypes.data_as(_P(C.c_int32)), _ptr(y), _ptr(w), Xd.shape[0],
                                                C.byref(loss)))
        return float(loss.value)

    def step_async(self, X, y, w=None) -> None:
        """queue one step on HOST buffers without waiting (X/y/w should be pinned and not reused for two more steps)"""
        X, y, w, rows = self._xyw(X, y, w)
        check(lib().sb_trainer_step_async(self._h, _ptr(X), _ptr(y), _ptr(w), rows))

    def accumulate(self, X, y, w=None) -> float:
        X, y, w, rows = self._xyw(X, y, w)
        loss = C.c_float()
        check(lib().sb_trainer_accumulate(self._h, _ptr(X), _ptr(y), _ptr(w), rows, C.byref(loss)))
        return float(loss.value)

    def apply_accumulated(self, total_pushes: Optional[int] = None):
        """one update from the accumulated gradients; total_pushes = divisor over ALL ranks (default world * n_acc)"""
        if total_pushes is None:
            check(lib().sb_trainer_apply_accumulated(self._h))
        else:
            check(lib().sb_trainer_apply_accumulated_mean(self._h, int(total_pushes)))

    def loss_resident(self, row_offset: int, rows: int) -> float:
        loss = C.c_float()
        check(lib().sb_trainer_loss_resident(self._h, row_offset, rows, C.byref(loss)))
        return float(loss.value)

    def broadcast_state(self, root: int = 0):
        check(lib().sb_trainer_broadcast_state(self._h, root))

    def load_dataset(self, X, y, w=None):
        X, y, w, rows = self._xyw(X, y, w)
        check(lib().sb_trainer_load_dataset(self._h, _ptr(X), _ptr(y), _ptr(w), rows))
        self.dataset_rows = rows

    def load_dataset_sparse(self, Xd, idx, y, w=None):
        """wide+deep resident set (after set_sparse): Xd [rows, n_dense] and y / w [rows] as numpy or DeviceArray, idx
        [rows, n_cat] as a numpy integer array or a DeviceArray whose memory holds int32 values.  The resident calls
        (run_resident, step_resident, accumulate_resident, loss_resident, profile_step) then run sparse steps over it."""
        if getattr(self, "_sparse", None) is None:      # the library reports the missing set_sparse (SB_ERR_STATE)
            check(lib().sb_trainer_load_dataset_sparse(self._h, None, None, None, None, 0))
        n_dense, n_cat = self._sparse
        if isinstance(Xd, DeviceArray):
            rows = Xd.shape[0]
            if len(Xd.shape) != 2 or Xd.shape[1] != n_dense:
                raise ValueError("Xd must be [rows, %d]" % n_dense)
        else:
            Xd = _f32(Xd)
            rows = Xd.shape[0]
            if Xd.ndim != 2 or Xd.shape[1] != n_dense:
                raise ValueError("Xd must be [rows, %d]" % n_dense)
        if isinstance(idx, DeviceArray):
            if tuple(idx.shape) != (rows, n_cat):
                raise ValueError("idx must be [rows, %d]" % n_cat)
            idx_p = C.cast(idx.ptr, _P(C.c_int32))
        else:
            idx = np.ascontiguousarray(idx, dtype=np.int32)
            if idx.shape != (rows, n_cat):
                raise ValueError("idx must be [rows, %d]" % n_cat)
            idx_p = idx.ctypes.data_as(_P(C.c_int32))
        if not isinstance(y, DeviceArray):
            y = _f32(y).reshape(-1)
        if w is not None and not isinstance(w, DeviceArray):
            w = _f32(w).reshape(-1)
        if y.size != rows or (w is not None and w.size != rows):
            raise ValueError("y / w length must equal rows")
        check(lib().sb_trainer_load_dataset_sparse(self._h, _ptr(Xd), idx_p, _ptr(y), _ptr(w), rows))
        self.dataset_rows = rows

    def step_resident(self, row_offset: int, rows: int) -> float:
        loss = C.c_float()
        check(lib().sb_trainer_step_resident(self._h, row_offset, rows, C.byref(loss)))
        return float(loss.value)

    def step_resident_async(self, row_offset: int, rows: int):
        check(lib().sb_trainer_step_resident_async(self._h, row_offset, rows))

    def run_resident(self, row_offsets, rows: int):
        """n update steps over the resident set in one call (asynchronous; the reference's per-epoch batch loop)"""
        offs = np.ascontiguousarray(row_offsets, dtype=np.int64).reshape(-1)
        check(lib().sb_trainer_run_resident(self._h, offs.ctypes.data_as(C.POINTER(C.c_int64)), offs.size, rows))

    def accumulate_resident(self, row_offset: int, rows: int) -> float:
        loss = C.c_float()
        check(lib().sb_trainer_accumulate_resident(self._h, row_offset, rows, C.byref(loss)))
        return float(loss.value)

    def last_loss(self) -> float:
        loss = C.c_float()
        check(lib().sb_trainer_last_loss(self._h, C.byref(loss)))
        return float(loss.value)

    def loss_history(self, first_step: int, n: int) -> np.ndarray:
        """mini-batch losses of update steps first_step .. first_step+n-1 (1-based global_step); waits for the GPU"""
        out = np.empty(n, np.float32)
        check(lib().sb_trainer_loss_history(self._h, first_step, n, _ptr(out)))
        return out

    def sync(self):
        check(lib().sb_trainer_sync(self._h))

    @property
    def stream(self) -> int:
        return int(lib().sb_trainer_stream(self._h) or 0)

    def kernels_per_step(self, rows: int) -> int:
        n = lib().sb_trainer_kernels_per_step(self._h, rows)
        if n < 0:
            check(n)
        return n

    def profile_step(self, row_offset: int, rows: int):
        """-> [(kernel name, milliseconds)] for one real (un-graphed) step over resident rows"""
        names = C.create_string_buffer(4096)
        ms = (C.c_float * 256)()
        n = C.c_int32(0)
        check(lib().sb_trainer_profile_step(self._h, row_offset, rows, names, 4096, ms, 256, C.byref(n)))
        nm = names.value.decode().split("\n") if n.value else []
        return [(nm[i], float(ms[i])) for i in range(n.value)]

    def eval_loss(self, X, y, w=None) -> float:
        X, y, w, rows = self._xyw(X, y, w)
        loss = C.c_float()
        check(lib().sb_trainer_eval_loss(self._h, _ptr(X), _ptr(y), _ptr(w), rows, C.byref(loss)))
        return float(loss.value)

    def predict(self, X) -> np.ndarray:
        X = _f32(X)
        out = np.empty(X.shape[0], np.float32)
        check(lib().sb_trainer_predict(self._h, _ptr(X), X.shape[0], _ptr(out)))
        return out

    def debug_step_trace(self):
        """-> (names, stamps[k,16] uint64 ns) of the last step's GEMM launches (needs SB_STEP_TRACE=1 at creation)"""
        buf = np.zeros((32, 16), np.uint64)
        names = C.create_string_buffer(4096)
        k = C.c_int32()
        check(lib().sb_debug_step_trace(self._h, buf.ctypes.data_as(C.POINTER(C.c_uint64)), 32, names, 4096, C.byref(k)))
        return names.value.decode().split(","), buf[:k.value].copy()

    @property
    def global_step(self) -> int:
        return int(lib().sb_trainer_global_step(self._h))

    def save_checkpoint(self, path: str):
        check(lib().sb_trainer_save_checkpoint(self._h, path.encode()))

    def load_checkpoint(self, path: str):
        check(lib().sb_trainer_load_checkpoint(self._h, path.encode()))

    def export_savedmodel(self, export_dir: str):
        check(lib().sb_trainer_export_savedmodel(self._h, export_dir.encode()))


class Model:
    """Owns one sb_model_t (batched scorer)."""

    def __init__(self, handle):
        self._h = handle
        self.n_features = int(lib().sb_model_n_features(self._h))

    @classmethod
    def load(cls, saved_model_dir: str, input_name: str, output_name: str, tag: str = "serve", device: int = 0,
             precision: int = PREC_FP32) -> "Model":
        h = C.c_void_p()
        enc = lambda s: None if s is None else s.encode()
        check(lib().sb_model_load(enc(saved_model_dir), enc(input_name), enc(output_name), enc(tag), device, precision,
                                  C.byref(h)))
        return cls(h)

    @classmethod
    def create(cls, desc: NetDesc, flat_params, device: int = 0) -> "Model":
        h = C.c_void_p()
        flat = _f32(flat_params).reshape(-1)
        check(lib().sb_model_create(C.byref(desc), _ptr(flat), flat.size, device, C.byref(h)))
        return cls(h)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().sb_model_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def score(self, X) -> np.ndarray:
        X = _f32(X)
        if X.ndim != 2 or X.shape[1] != self.n_features:
            raise ValueError("X must be [rows, %d]" % self.n_features)
        out = np.empty(X.shape[0], np.float32)
        check(lib().sb_model_score(self._h, _ptr(X), X.shape[0], _ptr(out)))
        return out

    def score_row_f64(self, row) -> float:
        row = np.ascontiguousarray(row, dtype=np.float64).reshape(-1)
        out = C.c_double()
        check(lib().sb_model_score_row_f64(self._h, row.ctypes.data_as(_f64p), row.size, C.byref(out)))
        return float(out.value)

    def score_device(self, dX_ptr: int, rows: int, dOut_ptr: int):
        check(lib().sb_model_score_device(self._h, C.c_void_p(dX_ptr), rows, C.c_void_p(dOut_ptr)))

    def sync(self):
        check(lib().sb_model_sync(self._h))

    @property
    def stream(self) -> int:
        return int(lib().sb_model_stream(self._h) or 0)


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(SB_NCCL_ID_BYTES)
    check(lib().sb_nccl_unique_id(C.cast(buf, _vp)))
    return buf.raw


def device_count() -> int:
    return int(lib().sb_device_count())


def savedmodel_write(export_dir: str, desc: NetDesc, flat_params) -> None:
    flat = _f32(flat_params).reshape(-1)
    check(lib().sb_savedmodel_write(export_dir.encode(), C.byref(desc), _ptr(flat), flat.size))


def savedmodel_read(saved_model_dir: str, input_name: str, output_name: str, tag: str = "serve"):
    """-> (n_features, hidden list, acts list, out_act, flat params)"""
    d = NetDesc()
    out_act = C.c_int32(0)
    n = C.c_int64(0)
    args = (saved_model_dir.encode(), input_name.encode(), output_name.encode(), tag.encode())
    check(lib().sb_savedmodel_read(*args, C.byref(d), C.byref(out_act), None, 0, C.byref(n)))
    flat = np.empty(n.value, np.float32)
    check(lib().sb_savedmodel_read(*args, C.byref(d), C.byref(out_act), _ptr(flat), flat.size, C.byref(n)))
    return int(d.n_features), [int(d.hidden[i]) for i in range(d.n_hidden)], [int(d.acts[i]) for i in range(d.n_hidden)], \
        int(out_act.value), flat


def debug_gemm_bf16(A: np.ndarray, B: np.ndarray, split_k: int = 1, device: int = 0, a_mn: bool = False,
                    b_mn: bool = False, cg: int = 0, bn: int = 0) -> np.ndarray:
    """D[M,N] = sum_k A(m,k) B(n,k) through the tcgen05 kernel (operands rounded to bf16 on the device).
    A is [M,K] (K-major) or, with a_mn, [K,M] (MN-major); B is [N,K] or, with b_mn, [K,N]."""
    A, B = _f32(A), _f32(B)
    (K, M) = A.shape if a_mn else A.shape[::-1]
    (K2, N) = B.shape if b_mn else B.shape[::-1]
    assert K == K2
    D = np.zeros((M, N), np.float32)
    check(lib().sb_debug_gemm_bf16_cfg(_ptr(A), _ptr(B), _ptr(D), M, N, K, split_k, int(a_mn), int(b_mn), cg, bn, device))
    return D


def debug_gemm_split(A: np.ndarray, B: np.ndarray, np_parts: int, device: int = 0) -> np.ndarray:
    """D[M,N] = A[M,K] B[N,K]^T on the tcgen05 path with every fp32 value split into np_parts bf16 parts"""
    A, B = _f32(A), _f32(B)
    M, K = A.shape
    N, K2 = B.shape
    assert K == K2
    D = np.zeros((M, N), np.float32)
    check(lib().sb_debug_gemm_split(_ptr(A), _ptr(B), _ptr(D), M, N, K, np_parts, device))
    return D


def debug_gemm_bench(M: int, N: int, K: int, split_k: int = 1, a_mn: bool = False, b_mn: bool = False, cg: int = 0,
                     bn: int = 0, iters: int = 50, device: int = 0) -> float:
    """average device ms per launch of one tile configuration (random operands)"""
    rng = np.random.default_rng(0)
    A = rng.standard_normal((K, M) if a_mn else (M, K), dtype=np.float32)
    B = rng.standard_normal((K, N) if b_mn else (N, K), dtype=np.float32)
    D = np.zeros((M, N), np.float32)
    ms = C.c_float()
    check(lib().sb_debug_gemm_bench(_ptr(A), _ptr(B), _ptr(D), M, N, K, split_k, int(a_mn), int(b_mn), cg, bn, device,
                                    iters, C.byref(ms)))
    return float(ms.value)


def text_parse_device(text: bytes, col_map: Sequence[int], n_feat: int, delim: str = "|", device: int = 0, flag_cap: int = 65536):
    """sb_text_parse_device: -> (X DeviceArray [rows, n_feat], y DeviceArray [rows], w DeviceArray [rows], flags, text, kernel_ms)"""
    if not text.endswith(b"\n"):
        text = text + b"\n"
    cm = (C.c_int32 * len(col_map))(*[int(c) for c in col_map])
    dX, dy, dw = _f32p(), _f32p(), _f32p()
    flags = (CellFlag * flag_cap)()
    n_rows, n_flags, kms = C.c_int64(0), C.c_int64(0), C.c_float(0)
    check(lib().sb_text_parse_device(text, len(text), delim.encode()[:1], cm, len(col_map), n_feat, C.byref(dX), C.byref(dy), C.byref(dw),
                                     C.byref(n_rows), flags, flag_cap, C.byref(n_flags), device, C.byref(kms)))
    if n_flags.value > flag_cap:
        raise ShifuB200Error(SB_ERR_FORMAT, "%d cells need the slow path, more than flag_cap=%d" % (n_flags.value, flag_cap))
    fl = [(int(flags[i].row), int(flags[i].slot), int(flags[i].offset), int(flags[i].len)) for i in range(n_flags.value)]
    n = n_rows.value
    return DeviceArray(dX, (n, n_feat), device), DeviceArray(dy, (n,), device), DeviceArray(dw, (n,), device), fl, text, float(kms.value)


def text_parse(text: bytes, col_map: Sequence[int], n_feat: int, delim: str = "|", device: int = 0, host_debug: bool = False,
               flag_cap: int = 65536):
    """GPU ingest of delimiter-separated numeric text -> (X [rows, n_feat] f32, y [rows] f32, w [rows] f32, flags).
    flags = [(row, slot, offset, length)] for cells the exact fast path declined; the caller resolves them with float().
    host_debug=True runs the identical state machine on the host (unit tests only)."""
    if not text.endswith(b"\n"):
        text = text + b"\n"
    max_rows = text.count(b"\n")
    cm = (C.c_int32 * len(col_map))(*[int(c) for c in col_map])
    X = np.zeros((max_rows, n_feat), np.float32)
    y = np.zeros(max_rows, np.float32)
    w = np.ones(max_rows, np.float32)
    flags = (CellFlag * flag_cap)()
    n_rows, n_flags = C.c_int64(0), C.c_int64(0)
    args = [text, len(text), delim.encode()[:1], cm, len(col_map), n_feat, _ptr(X), _ptr(y), _ptr(w), max_rows, C.byref(n_rows),
            flags, flag_cap, C.byref(n_flags)]
    if host_debug:
        check(lib().sb_debug_text_parse_host(*args))
    else:
        check(lib().sb_text_parse(*args, device))
    if n_flags.value > flag_cap:
        raise ShifuB200Error(SB_ERR_FORMAT, "%d cells need the slow path, more than flag_cap=%d" % (n_flags.value, flag_cap))
    fl = [(int(flags[i].row), int(flags[i].slot), int(flags[i].offset), int(flags[i].len)) for i in range(n_flags.value)]
    n = n_rows.value
    return X[:n], y[:n], w[:n], fl, text
