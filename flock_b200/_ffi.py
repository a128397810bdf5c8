"""ctypes binding of libflockgpu.so (include/flockgpu.h) -- the same C ABI the Rust shim binds.

Loud, no fallback: importing flock_b200 raises when the shared object is missing; the object itself is mapped (and
every declared symbol resolved) on first use, so that pure-Python helpers (plans, nexgen) can be imported by the CPU
reference arm without mapping the product library.  Opening a context without a CUDA device raises FlockGpuError too.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "libflockgpu.so"


class FlockGpuError(RuntimeError):
    """A non-zero return code of the C ABI (maps to FlockError::Execution on the Rust side)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"[flockgpu {code}] {message}")
        self.code = code
        self.message = message


# error codes (include/flockgpu.h)
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NCCL, ERR_EXECUTION, ERR_NO_DEVICE = 0, -1, -2, -3, -4, -5, -6

# enum flockgpu_join_type, by the lower-case DataFusion 6 JoinType name
JOIN_TYPES = {"inner": 0, "left": 1, "right": 2, "full": 3, "semi": 4, "anti": 5}


class ArrowSchema(C.Structure):
    pass


ArrowSchema._fields_ = [
    ("format", C.c_char_p), ("name", C.c_char_p), ("metadata", C.c_void_p), ("flags", C.c_int64),
    ("n_children", C.c_int64), ("children", C.POINTER(C.POINTER(ArrowSchema))),
    ("dictionary", C.POINTER(ArrowSchema)), ("release", C.c_void_p), ("private_data", C.c_void_p),
]


class ArrowArray(C.Structure):
    pass


ArrowArray._fields_ = [
    ("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64), ("n_buffers", C.c_int64),
    ("n_children", C.c_int64), ("buffers", C.POINTER(C.c_void_p)), ("children", C.POINTER(C.POINTER(ArrowArray))),
    ("dictionary", C.POINTER(ArrowArray)), ("release", C.c_void_p), ("private_data", C.c_void_p),
]


class ExprToken(C.Structure):
    _fields_ = [("op", C.c_int32), ("dtype", C.c_int32), ("col", C.c_int32), ("str_len", C.c_int32),
                ("i64", C.c_int64), ("f64", C.c_double), ("str", C.c_char_p)]


class Expr(C.Structure):
    _fields_ = [("tokens", C.POINTER(ExprToken)), ("n_tokens", C.c_int32)]


class AggSpec(C.Structure):
    _fields_ = [("func", C.c_int32), ("col", C.c_int32), ("name", C.c_char_p)]


def _require_library() -> None:
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(flock_b200 has no CPU fallback)")


_require_library()      # importing the package without the shared object fails here, loudly


class _Library:
    """The shared object, mapped on FIRST USE: `bench.py --impl reference` imports flock_b200.plans / .nexgen (plan JSON
    and input generators, pure Python) and must not map the product library into the CPU arm's process."""

    def __init__(self):
        self._cdll = None

    def _load(self) -> C.CDLL:
        if self._cdll is None:
            _require_library()
            cdll = C.CDLL(str(LIB_PATH), mode=os.RTLD_GLOBAL if hasattr(os, "RTLD_GLOBAL") else C.DEFAULT_MODE)
            for name, (res, args) in PROTOTYPES.items():
                fn = getattr(cdll, name)          # AttributeError here = the .so does not export a declared symbol
                fn.restype = res
                fn.argtypes = args
            self._cdll = cdll
        return self._cdll

    @property
    def loaded(self) -> bool:
        return self._cdll is not None

    def __getattr__(self, name):
        return getattr(self._load(), name)


lib = _Library()

_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_I32P = C.POINTER(C.c_int32)

# name -> (restype, argtypes); every symbol declared in include/flockgpu.h
PROTOTYPES = {
    "flockgpu_open": (C.c_int, [C.c_int, _PP]),
    "flockgpu_close": (C.c_int, [_P]),
    "flockgpu_last_error": (C.c_char_p, []),
    "flockgpu_version": (C.c_char_p, []),
    "flockgpu_synchronize": (C.c_int, [_P]),
    "flockgpu_timer_start": (C.c_int, [_P, C.c_int]),
    "flockgpu_timer_stop": (C.c_int, [_P, C.c_int]),
    "flockgpu_timer_elapsed_ms": (C.c_int, [_P, C.c_int, C.POINTER(C.c_float)]),
    "flockgpu_kernel_launches": (C.c_int64, [_P]),
    "flockgpu_bytes_moved": (C.c_int64, [_P, C.c_int32]),
    "flockgpu_set_option": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "flockgpu_profile_begin": (C.c_int, [_P]),
    "flockgpu_profile_end": (C.c_int, [_P, C.c_char_p, C.c_int32]),
    "flockgpu_host_alloc": (C.c_int, [_P, C.c_int64, _PP]),
    "flockgpu_host_free": (C.c_int, [_P, _P]),
    "flockgpu_flush_l2": (C.c_int, [_P]),
    "flockgpu_table_import": (C.c_int, [_P, C.POINTER(ArrowSchema), C.POINTER(C.POINTER(ArrowArray)), C.c_int32, _I32P, C.c_int32, _PP]),
    "flockgpu_table_export": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.POINTER(ArrowSchema), C.POINTER(ArrowArray)]),
    "flockgpu_table_schema": (C.c_int, [_P, _P, C.POINTER(ArrowSchema)]),
    "flockgpu_table_import_ipc": (C.c_int, [_P, C.POINTER(ArrowSchema), C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_void_p),
                                           C.POINTER(C.c_int64), C.c_int32, _I32P, C.c_int32, _PP]),
    "flockgpu_table_export_ipc": (C.c_int, [_P, _P, C.c_int64, C.c_int64, _PP, C.POINTER(C.c_int64), _PP, C.POINTER(C.c_int64)]),
    "flockgpu_ipc_free": (None, [_P]),
    "flockgpu_table_import_ndjson": (C.c_int, [_P, C.POINTER(ArrowSchema), _P, C.c_int64, _PP]),
    "flockgpu_table_retain": (C.c_int, [_P]),
    "flockgpu_table_release": (C.c_int, [_P]),
    "flockgpu_table_num_rows": (C.c_int64, [_P]),
    "flockgpu_table_num_columns": (C.c_int32, [_P]),
    "flockgpu_table_nbytes": (C.c_int64, [_P]),
    "flockgpu_table_concat": (C.c_int, [_P, _PP, C.c_int32, _PP]),
    "flockgpu_window_open": (C.c_int, [_P, C.c_int32, C.c_int32, _PP]),
    "flockgpu_window_close": (C.c_int, [_P]),
    "flockgpu_window_push": (C.c_int, [_P, _P]),
    "flockgpu_window_ready": (C.c_int, [_P, _I32P]),
    "flockgpu_window_next": (C.c_int, [_P, _PP, C.POINTER(C.c_int64)]),
    "flockgpu_filter_project": (C.c_int, [_P, _P, C.POINTER(Expr), C.POINTER(Expr), C.POINTER(C.c_char_p), C.c_int32, _PP]),
    "flockgpu_hash_aggregate": (C.c_int, [_P, _P, C.c_int32, _I32P, C.c_int32, C.POINTER(AggSpec), C.c_int32, _PP]),
    "flockgpu_hash_join": (C.c_int, [_P, _P, _P, _I32P, _I32P, C.c_int32, _PP]),
    "flockgpu_hash_join_typed": (C.c_int, [_P, _P, _P, _I32P, _I32P, C.c_int32, C.c_int32, _PP]),
    "flockgpu_hash_partition": (C.c_int, [_P, _P, _I32P, C.c_int32, C.c_int32, _PP]),
    "flockgpu_sort": (C.c_int, [_P, _P, _I32P, _I32P, C.c_int32, _PP]),
    "flockgpu_row_number": (C.c_int, [_P, _P, _I32P, C.c_int32, C.c_char_p, _PP]),
    "flockgpu_limit": (C.c_int, [_P, _P, C.c_int64, _PP]),
    "flockgpu_comm_unique_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "flockgpu_comm_init": (C.c_int, [_P, C.POINTER(C.c_uint8), C.c_int32, C.c_int32]),
    "flockgpu_comm_rank": (C.c_int, [_P, _I32P, _I32P]),
    "flockgpu_all_to_all": (C.c_int, [_P, _PP, C.c_int32, _PP]),
    "flockgpu_hash_exchange": (C.c_int, [_P, _P, _I32P, C.c_int32, _PP]),
    "flock_context_unmarshal": (C.c_int, [_P, C.c_char_p, _PP]),
    "flock_context_free": (C.c_int, [_P]),
    "flock_context_num_plans": (C.c_int32, [_P]),
    "flock_context_feed_data_sources": (C.c_int, [_P, C.POINTER(C.POINTER(ArrowSchema)), C.POINTER(C.POINTER(C.POINTER(ArrowArray))), _I32P, C.c_int32]),
    "flock_context_feed_tables": (C.c_int, [_P, _PP, C.c_int32]),
    "flock_context_execute": (C.c_int, [_P, C.c_int32, _PP]),
    "flock_context_execute_partitioned": (C.c_int, [_P, C.c_int32, _PP, C.c_int32, _I32P]),
    "flock_context_clean_data_sources": (C.c_int, [_P]),
    "flock_context_is_shuffling": (C.c_int, [_P, _I32P]),
    "flock_context_plan_str": (C.c_char_p, [_P, C.c_int32]),
    "flockgpu_selftest_eval_predicate": (C.c_int, [C.POINTER(ArrowSchema), C.POINTER(ArrowArray), C.POINTER(Expr), _P, _I32P]),
    "flockgpu_selftest_eval_value": (C.c_int, [C.POINTER(ArrowSchema), C.POINTER(ArrowArray), C.POINTER(Expr), _P, _I32P, _I32P]),
    "flockgpu_selftest_pred_i32": (C.c_int, [C.c_int64, C.c_int32, C.c_int64, _I32P, C.c_int64, C.POINTER(C.c_uint8), _I32P]),
}


def check(rc: int) -> None:
    if rc != 0:
        raise FlockGpuError(rc, lib.flockgpu_last_error().decode("utf-8", "replace"))
