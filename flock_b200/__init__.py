"""flock_b200 -- host-side Python mirror of the B200-native executor behind Flock's ExecutionPlan path.

Everything here is a thin veneer over the C ABI in include/flockgpu.h (ctypes, Arrow C Data
Interface through pyarrow); the product is libflockgpu.so.  Names follow the reference:

    ExecutionContext            flock/src/runtime/context.rs (feed_data_sources / execute /
                                execute_partitioned / clean_data_sources / is_shuffling)
    Context.filter_project      FilterExec + CoalesceBatchesExec + ProjectionExec
    Context.hash_aggregate      HashAggregateExec {Partial, Final, FinalPartitioned}
    Context.hash_join           HashJoinExec {Partitioned, Inner | Left | Right | Full | Semi | Anti}
    Context.hash_partition      RepartitionExec: Hash(keys, n)
"""
from __future__ import annotations

import ctypes as C
import json
from typing import Iterable, Sequence

import pyarrow as pa

from . import _ffi
from ._ffi import FlockGpuError, lib, check

__all__ = ["Context", "Table", "HostRelation", "ExecutionContext", "Window", "FlockGpuError", "col", "lit", "E"]

# enum flockgpu_dtype
BOOL, INT32, INT64, UINT64, FLOAT64, TIMESTAMP, UTF8, UINT32 = range(8)
_DTYPE_BY_NAME = {"bool": BOOL, "int32": INT32, "int64": INT64, "uint64": UINT64, "float64": FLOAT64,
                  "timestamp": TIMESTAMP, "utf8": UTF8, "uint32": UINT32,
                  "Int32": INT32, "Int64": INT64, "UInt64": UINT64, "Float64": FLOAT64, "Utf8": UTF8, "UInt32": UINT32}
# enum flockgpu_op
OP_COLUMN, OP_LIT_I64, OP_LIT_F64, OP_LIT_UTF8, OP_CAST = 1, 2, 3, 4, 5
OP_ADD, OP_SUB, OP_MUL, OP_DIV, OP_MOD = 10, 11, 12, 13, 14
OP_EQ, OP_NE, OP_LT, OP_LE, OP_GT, OP_GE = 20, 21, 22, 23, 24, 25
OP_AND, OP_OR, OP_NOT = 30, 31, 32
# enum flockgpu_agg_mode / flockgpu_agg_func
AGG_PARTIAL, AGG_FINAL, AGG_FINAL_PARTITIONED, AGG_SINGLE = 0, 1, 2, 3
AGG_COUNT, AGG_SUM, AGG_MIN, AGG_MAX, AGG_AVG = 0, 1, 2, 3, 4
_AGG_BY_NAME = {"count": AGG_COUNT, "sum": AGG_SUM, "min": AGG_MIN, "max": AGG_MAX, "avg": AGG_AVG}
_MODE_BY_NAME = {"partial": AGG_PARTIAL, "final": AGG_FINAL, "final_partitioned": AGG_FINAL_PARTITIONED, "single": AGG_SINGLE}


# ------------------------------------------------------------------------------------------------
# expressions: a tiny builder producing the postfix token programs of the C ABI
# ------------------------------------------------------------------------------------------------
class E:
    """A physical expression as a postfix token list [(op, dtype, col, i64, f64, str)]."""

    def __init__(self, tokens: list[tuple]):
        self.tokens = tokens

    @staticmethod
    def wrap(v) -> "E":
        return v if isinstance(v, E) else lit(v)

    def _bin(self, op: int, other, swap: bool = False) -> "E":
        o = E.wrap(other)
        a, b = (o, self) if swap else (self, o)
        return E(a.tokens + b.tokens + [(op, 0, 0, 0, 0.0, None)])

    def cast(self, dtype: str | int) -> "E":
        dt = _DTYPE_BY_NAME[dtype] if isinstance(dtype, str) else dtype
        return E(self.tokens + [(OP_CAST, dt, 0, 0, 0.0, None)])

    def __add__(self, o): return self._bin(OP_ADD, o)
    def __radd__(self, o): return self._bin(OP_ADD, o, True)
    def __sub__(self, o): return self._bin(OP_SUB, o)
    def __rsub__(self, o): return self._bin(OP_SUB, o, True)
    def __mul__(self, o): return self._bin(OP_MUL, o)
    def __rmul__(self, o): return self._bin(OP_MUL, o, True)
    def __truediv__(self, o): return self._bin(OP_DIV, o)
    def __rtruediv__(self, o): return self._bin(OP_DIV, o, True)
    def __mod__(self, o): return self._bin(OP_MOD, o)
    def __rmod__(self, o): return self._bin(OP_MOD, o, True)
    def __eq__(self, o): return self._bin(OP_EQ, o)      # noqa: builds an expression, not a bool
    def __ne__(self, o): return self._bin(OP_NE, o)
    def __lt__(self, o): return self._bin(OP_LT, o)
    def __le__(self, o): return self._bin(OP_LE, o)
    def __gt__(self, o): return self._bin(OP_GT, o)
    def __ge__(self, o): return self._bin(OP_GE, o)
    def __and__(self, o): return self._bin(OP_AND, o)
    def __or__(self, o): return self._bin(OP_OR, o)
    def __invert__(self): return E(self.tokens + [(OP_NOT, 0, 0, 0, 0.0, None)])
    __hash__ = None


def col(index: int) -> E:
    return E([(OP_COLUMN, 0, int(index), 0, 0.0, None)])


def lit(value, dtype: str | None = None) -> E:
    if isinstance(value, bool):
        raise TypeError("boolean literals are not supported")
    if isinstance(value, int):
        dt = _DTYPE_BY_NAME[dtype] if dtype else INT64
        return E([(OP_LIT_I64, dt, 0, int(value) if value < (1 << 63) else int(value) - (1 << 64), 0.0, None)])
    if isinstance(value, float):
        return E([(OP_LIT_F64, FLOAT64, 0, 0, float(value), None)])
    if isinstance(value, str):
        return E([(OP_LIT_UTF8, UTF8, 0, 0, 0.0, value.encode("utf-8"))])
    raise TypeError(f"unsupported literal {value!r}")


class _CExpr:
    """Keeps the ctypes token array of one expression alive."""

    def __init__(self, e: E):
        n = len(e.tokens)
        self.arr = (_ffi.ExprToken * n)()
        self.keep = []
        for i, (op, dt, c, i64, f64, s) in enumerate(e.tokens):
            t = self.arr[i]
            t.op, t.dtype, t.col, t.i64, t.f64 = op, dt, c, i64, f64
            if s is not None:
                self.keep.append(s)
                t.str = s
                t.str_len = len(s)
        self.expr = _ffi.Expr(self.arr, n)


# ------------------------------------------------------------------------------------------------
# Arrow C Data Interface helpers
# ------------------------------------------------------------------------------------------------
def _export_batches(schema: pa.Schema, batches: Sequence[pa.RecordBatch]):
    c_schema = _ffi.ArrowSchema()
    schema._export_to_c(C.addressof(c_schema))
    arrays = (_ffi.ArrowArray * max(len(batches), 1))()
    ptrs = (C.POINTER(_ffi.ArrowArray) * max(len(batches), 1))()
    for i, b in enumerate(batches):
        if b.schema.names != schema.names:
            raise ValueError("all batches of a relation must share one schema")
        b._export_to_c(C.addressof(arrays[i]))
        ptrs[i] = C.pointer(arrays[i])
    return c_schema, arrays, ptrs


def _release_exported(c_schema, arrays, n):
    # we only lent the data: call the release callbacks pyarrow installed
    rel_t = C.CFUNCTYPE(None, C.c_void_p)
    for i in range(n):
        if arrays[i].release:
            rel_t(arrays[i].release)(C.addressof(arrays[i]))
    if c_schema.release:
        rel_t(c_schema.release)(C.addressof(c_schema))


class HostRelation:
    """One relation's record batches exported ONCE through the Arrow C Data Interface.

    Exporting a RecordBatch from Python costs ~10 us; a 10 M-row relation is 153 batches, so re-exporting per
    invocation would dominate the end-to-end time.  The Rust shim holds FFI_ArrowArray structs the same way.
    ``feed_data_sources`` accepts a HostRelation wherever it accepts a list of partitions."""

    def __init__(self, batches: Sequence[pa.RecordBatch]):
        self.batches = list(batches)
        if not self.batches:
            raise ValueError("a relation needs at least one (possibly empty) batch")
        self.schema = self.batches[0].schema
        self.c_schema, self.arrays, self.ptrs = _export_batches(self.schema, self.batches)
        self.n = len(self.batches)

    def release(self) -> None:
        if self.n:
            _release_exported(self.c_schema, self.arrays, self.n)
            self.n = 0

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class Table:
    """A device-resident relation (flockgpu_table)."""

    def __init__(self, ctx: "Context", handle: int):
        self.ctx = ctx
        self.handle = C.c_void_p(handle)

    @property
    def num_rows(self) -> int:
        return lib.flockgpu_table_num_rows(self.handle)

    @property
    def num_columns(self) -> int:
        return lib.flockgpu_table_num_columns(self.handle)

    @property
    def nbytes(self) -> int:
        return lib.flockgpu_table_nbytes(self.handle)

    @property
    def schema(self) -> pa.Schema:
        s = _ffi.ArrowSchema()
        check(lib.flockgpu_table_schema(self.ctx.handle, self.handle, C.byref(s)))
        return pa.Schema._import_from_c(C.addressof(s))

    def to_batch(self, row_begin: int = 0, row_count: int = -1) -> pa.RecordBatch:
        s, a = _ffi.ArrowSchema(), _ffi.ArrowArray()
        check(lib.flockgpu_table_export(self.ctx.handle, self.handle, row_begin, row_count, C.byref(s), C.byref(a)))
        return pa.RecordBatch._import_from_c(C.addressof(a), C.addressof(s))

    def to_arrow(self) -> pa.Table:
        return pa.Table.from_batches([self.to_batch()])

    def to_ipc(self, row_begin: int = 0, row_count: int = -1) -> tuple[bytes, bytes]:
        """(header, body) of one Arrow IPC record-batch message: the DataFrame the reference's `to_payload` would build."""
        h, b = C.c_void_p(), C.c_void_p()
        hl, bl = C.c_int64(), C.c_int64()
        check(lib.flockgpu_table_export_ipc(self.ctx.handle, self.handle, row_begin, row_count, C.byref(h), C.byref(hl), C.byref(b), C.byref(bl)))
        try:
            return C.string_at(h, hl.value), C.string_at(b, bl.value)
        finally:
            lib.flockgpu_ipc_free(h)
            lib.flockgpu_ipc_free(b)

    def release(self) -> None:
        if self.handle:
            lib.flockgpu_table_release(self.handle)
            self.handle = C.c_void_p(None)

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class Context:
    """A GPU context (flockgpu_ctx): one device, one stream."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        check(lib.flockgpu_open(device, C.byref(h)))
        self.handle = h
        self.device = device

    def close(self) -> None:
        if self.handle:
            check(lib.flockgpu_close(self.handle))
            self.handle = C.c_void_p(None)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- plumbing
    def synchronize(self) -> None:
        check(lib.flockgpu_synchronize(self.handle))

    def flush_l2(self) -> None:
        check(lib.flockgpu_flush_l2(self.handle))

    def timer_start(self, slot: int = 0) -> None:
        check(lib.flockgpu_timer_start(self.handle, slot))

    def timer_stop(self, slot: int = 0) -> None:
        check(lib.flockgpu_timer_stop(self.handle, slot))

    def timer_ms(self, slot: int = 0) -> float:
        ms = C.c_float()
        check(lib.flockgpu_timer_elapsed_ms(self.handle, slot, C.byref(ms)))
        return ms.value

    def set_option(self, name: str, value: int) -> None:
        check(lib.flockgpu_set_option(self.handle, name.encode(), int(value)))

    def profile_begin(self) -> None:
        check(lib.flockgpu_profile_begin(self.handle))

    def profile_end(self) -> dict:
        buf = C.create_string_buffer(1 << 16)
        check(lib.flockgpu_profile_end(self.handle, buf, len(buf)))
        return json.loads(buf.value.decode())

    @property
    def kernel_launches(self) -> int:
        return lib.flockgpu_kernel_launches(self.handle)

    def bytes_moved(self) -> tuple[int, int]:
        """(host -> device, device -> host) bytes this context has moved over the host link so far."""
        return lib.flockgpu_bytes_moved(self.handle, 0), lib.flockgpu_bytes_moved(self.handle, 1)

    def host_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        check(lib.flockgpu_host_alloc(self.handle, nbytes, C.byref(p)))
        return p.value

    def host_free(self, ptr: int) -> None:
        check(lib.flockgpu_host_free(self.handle, C.c_void_p(ptr)))

    def pinned_copy(self, batch: pa.RecordBatch) -> pa.RecordBatch:
        """Copies a record batch into page-locked host memory (the e2e leg of bench.py)."""
        cols = []
        for arr in batch.columns:
            bufs = []
            for b in arr.buffers():
                if b is None:
                    bufs.append(None)
                    continue
                p = self.host_alloc(max(b.size, 8))
                C.memmove(p, b.address, b.size)
                bufs.append(pa.foreign_buffer(p, b.size, base=_PinnedOwner(self, p)))
            cols.append(pa.Array.from_buffers(arr.type, len(arr), bufs, null_count=arr.null_count, offset=arr.offset))
        return pa.RecordBatch.from_arrays(cols, schema=batch.schema)

    # ---- tables
    def import_batches(self, batches: Sequence[pa.RecordBatch], projection: Sequence[int] | None = None,
                       schema: pa.Schema | None = None) -> Table:
        batches = list(batches)
        schema = schema or batches[0].schema
        c_schema, arrays, ptrs = _export_batches(schema, batches)
        try:
            proj = (C.c_int32 * len(projection))(*projection) if projection is not None else None
            out = C.c_void_p()
            check(lib.flockgpu_table_import(self.handle, C.byref(c_schema), ptrs, len(batches), proj,
                                            len(projection) if projection is not None else 0, C.byref(out)))
        finally:
            _release_exported(c_schema, arrays, len(batches))
        return Table(self, out.value)

    def import_ipc(self, schema: pa.Schema, frames: Sequence[tuple], projection: Sequence[int] | None = None) -> Table:
        """frames: [(header, body)] -- the data_header / data_body of Arrow-Flight messages (bytes-like or pyarrow buffers)."""
        n = len(frames)
        keep = [(pa.py_buffer(h) if not isinstance(h, pa.Buffer) else h, pa.py_buffer(b) if not isinstance(b, pa.Buffer) else b) for h, b in frames]
        hp = (C.c_void_p * max(n, 1))(*[h.address for h, _ in keep])
        hl = (C.c_int64 * max(n, 1))(*[h.size for h, _ in keep])
        bp = (C.c_void_p * max(n, 1))(*[b.address for _, b in keep])
        bl = (C.c_int64 * max(n, 1))(*[b.size for _, b in keep])
        c_schema = _ffi.ArrowSchema()
        schema._export_to_c(C.addressof(c_schema))
        try:
            proj = (C.c_int32 * len(projection))(*projection) if projection is not None else None
            out = C.c_void_p()
            check(lib.flockgpu_table_import_ipc(self.handle, C.byref(c_schema), hp, hl, bp, bl, n, proj, len(projection) if projection is not None else 0,
                                                C.byref(out)))
        finally:
            if c_schema.release:
                C.CFUNCTYPE(None, C.c_void_p)(c_schema.release)(C.addressof(c_schema))
        return Table(self, out.value)

    def import_ndjson(self, schema: pa.Schema, text: bytes) -> Table:
        """One flat JSON object per line -> table (event_bytes_to_batch, flock/src/transmute.rs:255-266)."""
        buf = pa.py_buffer(text)
        c_schema = _ffi.ArrowSchema()
        schema._export_to_c(C.addressof(c_schema))
        try:
            out = C.c_void_p()
            check(lib.flockgpu_table_import_ndjson(self.handle, C.byref(c_schema), C.c_void_p(buf.address), buf.size, C.byref(out)))
        finally:
            if c_schema.release:
                C.CFUNCTYPE(None, C.c_void_p)(c_schema.release)(C.addressof(c_schema))
        return Table(self, out.value)

    def concat(self, tables: Sequence[Table]) -> Table:
        hs = (C.c_void_p * len(tables))(*[t.handle for t in tables])
        out = C.c_void_p()
        check(lib.flockgpu_table_concat(self.handle, hs, len(tables), C.byref(out)))
        return Table(self, out.value)

    # ---- operators
    def filter_project(self, table: Table, predicate: E | None = None, projections: Sequence[E] | None = None,
                       names: Sequence[str] | None = None) -> Table:
        pred = _CExpr(predicate) if predicate is not None else None
        projs = [_CExpr(E.wrap(p)) for p in (projections or [])]
        parr = (_ffi.Expr * max(len(projs), 1))()
        for i, p in enumerate(projs):
            parr[i] = p.expr
        narr = None
        if names is not None:
            keep = [n.encode() if n is not None else None for n in names]
            narr = (C.c_char_p * len(keep))(*keep)
        out = C.c_void_p()
        check(lib.flockgpu_filter_project(self.handle, table.handle, C.byref(pred.expr) if pred else None,
                                          parr if projs else None, narr, len(projs), C.byref(out)))
        return Table(self, out.value)

    def hash_aggregate(self, table: Table, group_cols: Sequence[int], aggs: Sequence[tuple], mode: str | int = "single") -> Table:
        """aggs: [(func, col, name)], func in count/sum/min/max/avg, col = -1 for COUNT(*)."""
        m = _MODE_BY_NAME[mode] if isinstance(mode, str) else mode
        g = (C.c_int32 * max(len(group_cols), 1))(*group_cols)
        specs = (_ffi.AggSpec * max(len(aggs), 1))()
        keep = []
        for i, (f, c, name) in enumerate(aggs):
            specs[i].func = _AGG_BY_NAME[f] if isinstance(f, str) else f
            specs[i].col = c
            keep.append(name.encode())
            specs[i].name = keep[-1]
        out = C.c_void_p()
        check(lib.flockgpu_hash_aggregate(self.handle, table.handle, m, g, len(group_cols), specs, len(aggs), C.byref(out)))
        return Table(self, out.value)

    def hash_join(self, left: Table, right: Table, left_keys: Sequence[int], right_keys: Sequence[int], join_type: str = "inner") -> Table:
        """join_type: inner, left, right, full (output left ++ right columns) or semi, anti (left columns only, left order)."""
        jt = _ffi.JOIN_TYPES.get(join_type.lower()) if isinstance(join_type, str) else None
        if jt is None:
            raise ValueError(f"unknown join type {join_type!r}; expected one of {sorted(_ffi.JOIN_TYPES)}")
        lk = (C.c_int32 * len(left_keys))(*left_keys)
        rk = (C.c_int32 * len(right_keys))(*right_keys)
        out = C.c_void_p()
        if jt == 0:
            check(lib.flockgpu_hash_join(self.handle, left.handle, right.handle, lk, rk, len(left_keys), C.byref(out)))
        else:
            check(lib.flockgpu_hash_join_typed(self.handle, left.handle, right.handle, lk, rk, len(left_keys), jt, C.byref(out)))
        return Table(self, out.value)

    def hash_partition(self, table: Table, key_cols: Sequence[int], n_parts: int) -> list[Table]:
        k = (C.c_int32 * len(key_cols))(*key_cols)
        outs = (C.c_void_p * n_parts)()
        check(lib.flockgpu_hash_partition(self.handle, table.handle, k, len(key_cols), n_parts, outs))
        return [Table(self, h) for h in outs]

    def sort(self, table: Table, cols: Sequence[int], descending: Sequence[bool] | None = None) -> Table:
        k = (C.c_int32 * len(cols))(*cols)
        d = (C.c_int32 * len(cols))(*[1 if x else 0 for x in (descending or [False] * len(cols))])
        out = C.c_void_p()
        check(lib.flockgpu_sort(self.handle, table.handle, k, d, len(cols), C.byref(out)))
        return Table(self, out.value)

    def row_number(self, table: Table, partition_cols: Sequence[int], name: str = "ROW_NUMBER()") -> Table:
        k = (C.c_int32 * max(len(partition_cols), 1))(*partition_cols)
        out = C.c_void_p()
        check(lib.flockgpu_row_number(self.handle, table.handle, k, len(partition_cols), name.encode(), C.byref(out)))
        return Table(self, out.value)

    def limit(self, table: Table, n: int) -> Table:
        out = C.c_void_p()
        check(lib.flockgpu_limit(self.handle, table.handle, n, C.byref(out)))
        return Table(self, out.value)

    # ---- multi-GPU
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_uint8 * 128)()
        check(lib.flockgpu_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, unique_id: bytes, rank: int, world_size: int) -> None:
        buf = (C.c_uint8 * 128)(*unique_id)
        check(lib.flockgpu_comm_init(self.handle, buf, rank, world_size))

    def all_to_all(self, parts: Sequence[Table]) -> Table:
        hs = (C.c_void_p * len(parts))(*[t.handle for t in parts])
        out = C.c_void_p()
        check(lib.flockgpu_all_to_all(self.handle, hs, len(parts), C.byref(out)))
        return Table(self, out.value)

    def hash_exchange(self, table: Table, key_cols: Sequence[int]) -> Table:
        k = (C.c_int32 * len(key_cols))(*key_cols)
        out = C.c_void_p()
        check(lib.flockgpu_hash_exchange(self.handle, table.handle, k, len(key_cols), C.byref(out)))
        return Table(self, out.value)


class Window:
    """Hopping / tumbling window over epoch relations resident in HBM (flockgpu_window_*; hopping.rs:54-74)."""

    def __init__(self, ctx: Context, window_size: int, hop_size: int):
        self.ctx = ctx
        h = C.c_void_p()
        check(lib.flockgpu_window_open(ctx.handle, window_size, hop_size, C.byref(h)))
        self.handle = h

    def push(self, epoch: Table) -> None:
        check(lib.flockgpu_window_push(self.handle, epoch.handle))

    @property
    def ready(self) -> bool:
        v = C.c_int32()
        check(lib.flockgpu_window_ready(self.handle, C.byref(v)))
        return bool(v.value)

    def next(self) -> tuple[Table, int]:
        out, first = C.c_void_p(), C.c_int64()
        check(lib.flockgpu_window_next(self.handle, C.byref(out), C.byref(first)))
        return Table(self.ctx, out.value), first.value

    def close(self) -> None:
        if self.handle:
            lib.flockgpu_window_close(self.handle)
            self.handle = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def selftest_eval_predicate(batch: pa.RecordBatch, predicate: E):
    """CPU-only check of the expression compiler (flockgpu_selftest_eval_predicate): returns
    (mask: list[bool], fast_kind: int).  Not an execution path."""
    import numpy as np
    c_schema, arrays, ptrs = _export_batches(batch.schema, [batch])
    try:
        pred = _CExpr(predicate)
        mask = np.zeros(max(batch.num_rows, 1), np.uint8)
        fast = C.c_int32()
        check(lib.flockgpu_selftest_eval_predicate(C.byref(c_schema), ptrs[0], C.byref(pred.expr),
                                                   mask.ctypes.data_as(C.c_void_p), C.byref(fast)))
    finally:
        _release_exported(c_schema, arrays, 1)
    return mask[:batch.num_rows].astype(bool), fast.value


def selftest_pred_i32(x, modulus: int, cmp: int, rhs: int):
    """CPU-only: `CAST(x AS Int64) [% modulus] cmp rhs` (modulus 0 = no `%`) with the constants and the per-row test of the
    vectorised filter kernel (csrc/pred_i32.h).  Returns (bool mask, arithmetic mode 0 / 1 / 2)."""
    import numpy as np
    x = np.ascontiguousarray(x, dtype=np.int32)
    keep = np.zeros(max(len(x), 1), np.uint8)
    mode = C.c_int32()
    check(lib.flockgpu_selftest_pred_i32(modulus, cmp, rhs, x.ctypes.data_as(C.POINTER(C.c_int32)), len(x),
                                         keep.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(mode)))
    return keep[:len(x)].astype(bool), mode.value


def selftest_eval_value(batch: pa.RecordBatch, expr: E):
    """CPU-only check of value-expression lowering: returns (numpy values or None if pass-through, dtype code)."""
    import numpy as np
    c_schema, arrays, ptrs = _export_batches(batch.schema, [batch])
    try:
        ce = _CExpr(E.wrap(expr))
        out = np.zeros(max(batch.num_rows, 1), np.int64)
        dt, passthrough = C.c_int32(), C.c_int32()
        check(lib.flockgpu_selftest_eval_value(C.byref(c_schema), ptrs[0], C.byref(ce.expr), out.ctypes.data_as(C.c_void_p),
                                               C.byref(dt), C.byref(passthrough)))
    finally:
        _release_exported(c_schema, arrays, 1)
    if passthrough.value:
        return None, dt.value
    n = batch.num_rows
    if dt.value in (INT32, UINT32):
        return out.view(np.int32 if dt.value == INT32 else np.uint32)[:n].copy(), dt.value
    if dt.value == FLOAT64:
        return out.view(np.float64)[:n].copy(), dt.value
    if dt.value == UINT64:
        return out.view(np.uint64)[:n].copy(), dt.value
    return out[:n].copy(), dt.value


class _PinnedOwner:
    def __init__(self, ctx: Context, ptr: int):
        self.ctx, self.ptr = ctx, ptr

    def __del__(self):
        try:
            if self.ctx.handle:
                self.ctx.host_free(self.ptr)
        except Exception:
            pass


class ExecutionContext:
    """flock::runtime::context::ExecutionContext on the GPU (flock/src/runtime/context.rs).

    ``plans`` is the reference's serde-JSON physical plan (a dict / JSON string), a list of them, or
    a whole marshalled ExecutionContext object.
    """

    def __init__(self, ctx: Context, plans):
        self.ctx = ctx
        text = plans if isinstance(plans, str) else json.dumps(plans)
        h = C.c_void_p()
        # ctx=None gives a parse-only context (plan_str / is_shuffling), used by CPU-only tests
        check(lib.flock_context_unmarshal(ctx.handle if ctx is not None else None, text.encode("utf-8"), C.byref(h)))
        self.handle = h

    @property
    def num_plans(self) -> int:
        return lib.flock_context_num_plans(self.handle)

    def feed_data_sources(self, sources: Sequence[Sequence[Sequence[pa.RecordBatch]]]) -> None:
        """sources[relation][partition][batch] -- the Vec<Vec<Vec<RecordBatch>>> of context.rs:257."""
        n = len(sources)
        schemas = (C.POINTER(_ffi.ArrowSchema) * n)()
        batch_ptrs = (C.POINTER(C.POINTER(_ffi.ArrowArray)) * n)()
        counts = (C.c_int32 * n)()
        keep = []
        try:
            for i, rel in enumerate(sources):
                if isinstance(rel, HostRelation):
                    schemas[i], batch_ptrs[i], counts[i] = C.pointer(rel.c_schema), rel.ptrs, rel.n
                    continue
                flat = [b for part in rel for b in part]
                if not flat:
                    raise ValueError("feed_data_sources: a relation needs at least one (possibly empty) batch")
                cs, arrays, ptrs = _export_batches(flat[0].schema, flat)
                keep.append((cs, arrays, len(flat), ptrs))
                schemas[i] = C.pointer(cs)
                batch_ptrs[i] = ptrs
                counts[i] = len(flat)
            check(lib.flock_context_feed_data_sources(self.handle, schemas, batch_ptrs, counts, n))
        finally:
            for cs, arrays, k, _ in keep:
                _release_exported(cs, arrays, k)

    def feed_tables(self, tables: Sequence[Table]) -> None:
        hs = (C.c_void_p * len(tables))(*[t.handle for t in tables])
        check(lib.flock_context_feed_tables(self.handle, hs, len(tables)))

    def execute_device(self, plan_index: int = 0) -> Table:
        out = C.c_void_p()
        check(lib.flock_context_execute(self.handle, plan_index, C.byref(out)))
        return Table(self.ctx, out.value)

    def execute(self) -> list[list[pa.RecordBatch]]:
        """Vec<Vec<RecordBatch>>: one list of batches per plan (context.rs:172-191)."""
        return [[self.execute_device(i).to_batch()] for i in range(self.num_plans)]

    def execute_partitioned(self, max_parts: int = 64) -> list[list[list[pa.RecordBatch]]]:
        res = []
        for i in range(self.num_plans):
            outs = (C.c_void_p * max_parts)()
            n = C.c_int32()
            check(lib.flock_context_execute_partitioned(self.handle, i, outs, max_parts, C.byref(n)))
            res.append([[Table(self.ctx, outs[k]).to_batch()] for k in range(n.value)])
        return res

    def clean_data_sources(self) -> None:
        check(lib.flock_context_clean_data_sources(self.handle))

    def is_shuffling(self) -> bool:
        v = C.c_int32()
        check(lib.flock_context_is_shuffling(self.handle, C.byref(v)))
        return bool(v.value)

    def plan_str(self, plan_index: int = 0) -> str:
        s = lib.flock_context_plan_str(self.handle, plan_index)
        return s.decode() if s else ""

    def close(self) -> None:
        if self.handle:
            lib.flock_context_free(self.handle)
            self.handle = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
