"""Host logic that runs without a GPU (`-m "not gpu"`): the C ABI library loads and exports every symbol
include/flockgpu.h declares, fails loudly without a device, parses the reference's serde-JSON plans,
and lowers DataFusion expressions to the term/chain programs the kernels interpret."""
import ctypes as C
import json
import re
from pathlib import Path

import numpy as np
import pyarrow as pa
import pytest

import flock_b200 as fb
from flock_b200 import _ffi, nexgen, plans
from flock_b200 import col, lit

ROOT = Path(__file__).resolve().parent.parent
# the reference's own serialised plans (flock/src/tests/data/plan/*.json), stored verbatim
REFERENCE_PLANS = Path(__file__).resolve().parent / "golden" / "reference_plans"


def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "flockgpu.h").read_text()
    declared = set(re.findall(r"\b(flockgpu_[a-z0-9_]+|flock_context_[a-z0-9_]+)\s*\(", header))
    declared -= {"flockgpu_ctx", "flockgpu_table"}
    assert len(declared) >= 40
    lib = C.CDLL(str(_ffi.LIB_PATH))
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, f"libflockgpu.so does not export: {missing}"
    assert set(_ffi.PROTOTYPES) == declared, set(_ffi.PROTOTYPES) ^ declared


def test_version_and_no_cpu_fallback():
    assert b"sm_100a" in fb.lib.flockgpu_version()
    try:
        ctx = fb.Context(0)
    except fb.FlockGpuError as e:
        # CPU-only box: opening a context must fail loudly -- there is no CPU execution path
        assert e.code == _ffi.ERR_NO_DEVICE and "no CPU fallback" in e.message
        ec = fb.ExecutionContext(None, plans.q2())
        with pytest.raises(fb.FlockGpuError) as info:
            ec.execute_device(0)
        assert info.value.code == _ffi.ERR_NO_DEVICE
    else:
        ctx.close()


@pytest.mark.parametrize("query", ["q1", "q2", "q3", "q4", "q5", "q7", "q8"])
def test_unmarshal_nexmark_plans(query):
    ec = fb.ExecutionContext(None, plans.QUERIES[query]())
    assert ec.num_plans == 1 and not ec.is_shuffling()
    s = ec.plan_str(0)
    assert s.splitlines()[0].startswith("ProjectionExec: expr=[")
    assert "MemoryExec" in s
    if query == "q2":
        # the rendering of planner.rs:120-124
        assert "FilterExec: CAST(auction@0 AS Int64) % 123 = 0" in s
        assert "CoalesceBatchesExec: target_batch_size=4096" in s and "RepartitionExec: partitioning=RoundRobinBatch(8)" in s
    if query == "q3":
        assert "HashJoinExec: mode=Partitioned, join_type=Inner, on=[(seller, p_id)]" in s
        assert "FilterExec: state@3 = or OR state@3 = id OR state@3 = ca" in s
        assert s.count("RepartitionExec: partitioning=Hash") == 2 and s.count("FilterExec") == 2
    if query == "q5":
        assert s.count("HashAggregateExec: mode=Partial") == 3 and s.count("MemoryExec") == 2
    if query == "q4":
        assert "FilterExec: b_date_time@6 >= a_date_time@1 AND b_date_time@6 <= expires@2" in s       # BETWEEN, q4.sql
        assert "gby=[a_id@0 as a_id, category@3 as category], aggr=[MAX(bid.price)]" in s and "aggr=[AVG(Q.final)]" in s
    if query == "q7":
        assert "HashJoinExec: mode=Partitioned, join_type=Inner, on=[(price, maxprice)]" in s and "mode=Final, gby=[]" in s


def test_q6_plan_is_accepted():
    """q6 = SortExec + WindowAggExec(ROW_NUMBER) + the operators of q4: the GPU plan layer builds all of it."""
    s = fb.ExecutionContext(None, plans.q6()).plan_str()
    assert s.count("SortExec: [") == 3 and s.count("WindowAggExec: wdw=[ROW_NUMBER()") == 2
    assert "SortExec: [a_id@0 ASC, price@5 DESC]" in s and "aggr=[AVG(R.price)]" in s
    # other window functions are refused, not emulated
    bad = plans.row_number_window("r", [plans.column("a_id", 0)], [], plans.memory_exec(nexgen.auction_schema(), [0]))
    bad["window_expr"][0]["fun"] = "Rank"
    with pytest.raises(fb.FlockGpuError) as info:
        fb.ExecutionContext(None, bad)
    assert info.value.code == _ffi.ERR_UNSUPPORTED and "Rank" in info.value.message


def test_header_is_c_and_the_c_program_links(tmp_path):
    """include/flockgpu.h compiles as C11 (not only as C++), and tests/cabi/q2_cabi.c links against libflockgpu.so --
    every symbol it uses is exported with C linkage.  (It runs on the GPU box: tests/test_gpu_cabi.py.)"""
    import subprocess
    root = Path(__file__).resolve().parent.parent
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-x", "c", str(root / "include" / "flockgpu.h")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    from test_gpu_cabi import build_cabi_program
    build_cabi_program(tmp_path / "q2_cabi")
    assert (tmp_path / "q2_cabi").exists()


def test_shuffle_stage_and_marshalled_context():
    a, p = plans.q3_stage0()
    ec = fb.ExecutionContext(None, [a, p])
    assert ec.num_plans == 2 and ec.is_shuffling()       # context.rs:328-337
    wrapped = {"plan": {"execution_plans": [plans.q1()], "object_storage": None}, "name": "q1-00", "next": {"Sink": "Blackhole"}}
    assert fb.ExecutionContext(None, wrapped).num_plans == 1


def test_unsupported_nodes_fail_loudly():
    cross = {"execution_plan": "cross_join_exec", "left": plans.q2(), "right": plans.q2()}
    with pytest.raises(fb.FlockGpuError) as info:
        fb.ExecutionContext(None, cross)
    assert info.value.code == _ffi.ERR_UNSUPPORTED and "cross_join_exec" in info.value.message
    with pytest.raises(fb.FlockGpuError):
        fb.ExecutionContext(None, "{not json")


def test_reference_plan_fixtures_parse():
    """The reference's own serialised plans (older serde dialect: columns without index, on=[[\"a\",\"c\"]])."""
    ec = fb.ExecutionContext(None, (REFERENCE_PLANS / "simple_select.json").read_text())
    assert ec.plan_str(0).startswith("ProjectionExec: expr=[c1 as c1]")
    ec = fb.ExecutionContext(None, (REFERENCE_PLANS / "aggregate.json").read_text())
    s = ec.plan_str(0)
    assert "HashAggregateExec: mode=FinalPartitioned, gby=[c3 as c3], aggr=[MAX(c1), MIN(c2)]" in s
    assert "FilterExec: c2 < CAST(99 AS Float64)" in s
    s = fb.ExecutionContext(None, (REFERENCE_PLANS / "join.json").read_text()).plan_str(0)      # global_limit_exec <- sort_exec <- merge_exec <- ...
    assert s.startswith("GlobalLimitExec: limit=3\n  SortExec: [b ASC]\n    CoalescePartitionsExec")
    assert "HashJoinExec: mode=Partitioned, join_type=Inner, on=[(a, c)]" in s


# ---- expression lowering ---------------------------------------------------------------------------------
def expr_batch(n=1000, seed=0):
    rng = np.random.default_rng(seed)
    return pa.RecordBatch.from_arrays([
        pa.array(rng.integers(-5000, 5000, n).astype(np.int32)),
        pa.array(rng.integers(-(1 << 40), 1 << 40, n)),
        pa.array(rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2) + np.uint64(1)),
        pa.array(rng.normal(0, 100, n)),
        pa.array(rng.integers(1_436_918_400_000, 1_436_918_500_000, n), pa.timestamp("ms")),
        pa.array(rng.integers(1_436_918_400_000, 1_436_918_500_000, n), pa.timestamp("ms")),
        pa.array([["az", "ca", "id", "or", "wa", "wy", ""][k] for k in rng.integers(0, 7, n)]),
        pa.array(rng.integers(1, 50, n).astype(np.int32)),
    ], names=["i32", "i64", "u64", "f64", "t0", "t1", "state", "pos"])


def cols(b):
    return {name: b.column(i).to_numpy(zero_copy_only=False) for i, name in enumerate(b.schema.names)}


def test_predicate_lowering_matches_numpy():
    b = expr_batch()
    c = cols(b)
    i32, i64 = c["i32"].astype(np.int64), c["i64"]
    t0, t1 = c["t0"].astype("int64"), c["t1"].astype("int64")
    state = np.array(b.column(6).to_pylist())
    cases = [
        (col(0).cast("int64") % 123 == 0, np.fmod(i32, 123) == 0, 1),                       # q2, planner.rs:122
        (col(0).cast("int64") % 7 == -3, np.fmod(i32, 7) == -3, 1),
        (col(0).cast("int64") % -123 == 0, np.fmod(i32, 123) == 0, 1),
        (col(0).cast("int64") == 10, i32 == 10, 2),                                           # q3, planner.rs:155
        (col(0).cast("int64") >= -17, i32 >= -17, 2),
        (~(col(0).cast("int64") % 123 == 0), np.fmod(i32, 123) != 0, 1),                     # negation keeps the fast shape
        (~(col(0).cast("int64") < 5), i32 >= 5, 2),
        ((col(6) == "or") | (col(6) == "id") | (col(6) == "ca"), np.isin(state, ["or", "id", "ca"]), 0),  # planner.rs:162
        ((col(4) >= col(5)) & (col(4) <= col(5) + 20000), (t0 >= t1) & (t0 <= t1 + 20000), 0),  # q4 BETWEEN, planner.rs:237
        (col(3) < lit(99).cast("float64"), c["f64"] < 99.0, 0),                               # aggregate.json predicate
        (~((col(1) + 5) * 3 > col(0).cast("int64")), ~((i64 + 5) * 3 > i32), 0),
        ((col(1) - col(0).cast("int64")) / 7 != 0, np.trunc((i64 - i32) / 7).astype(np.int64) != 0, 0),
        (col(2) > lit(1 << 63, "uint64"), c["u64"] > np.uint64(1 << 63), 0),                  # unsigned domain
        (col(6) < "id", state < "id", 0),
        ((col(0) * 2 + 1).cast("int64") % col(7).cast("int64") == 1, np.fmod(i32 * 2 + 1, c["pos"].astype(np.int64)) == 1, 0),
        (lit(100) - col(0).cast("int64") > 5000, 100 - i32 > 5000, 0),
    ]
    for e, want, fast in cases:
        got, kind = fb.selftest_eval_predicate(b, e)
        assert kind == fast
        assert np.array_equal(got, want), fb.E.wrap(e).tokens


def test_truth_table_covers_and_or_not():
    b = expr_batch(256, seed=1)
    i32 = cols(b)["i32"].astype(np.int64)
    t = [i32 > 0, np.fmod(i32, 2) == 0, i32 < 1000, np.fmod(i32, 3) == 0]
    e = [col(0).cast("int64") > 0, col(0).cast("int64") % 2 == 0, col(0).cast("int64") < 1000, col(0).cast("int64") % 3 == 0]
    got, _ = fb.selftest_eval_predicate(b, (e[0] & ~e[1]) | (e[2] & (e[3] | ~e[0])))
    assert np.array_equal(got, (t[0] & ~t[1]) | (t[2] & (t[3] | ~t[0])))


def test_three_valued_predicates_match_arrow_kleene():
    """NULL operands: a comparison over a NULL is NULL, AND / OR / NOT follow Kleene's tables, and FilterExec keeps the rows
    whose predicate is TRUE (SURVEY.md Appendix C.3).  The truth table the kernels index is built by expr_compile.cc; here
    it runs on the host over bitmaps with a non-zero bit offset."""
    import pyarrow.compute as pc
    n = 300
    rng = np.random.default_rng(3)
    a = pa.array(rng.integers(-20, 20, n).astype(np.int32), mask=np.arange(n) % 5 == 0)
    b_ = pa.array(rng.integers(-20, 20, n), mask=np.arange(n) % 7 == 3)
    s_ = pa.array([None if k % 11 == 2 else ["or", "id", "ca", "wa"][k % 4] for k in range(n)])
    full = pa.RecordBatch.from_arrays([a, b_, s_, pa.array(np.arange(n, dtype=np.int32))], names=["a", "b", "s", "id"])
    b = full.slice(3, n - 9)                                                                   # bit offset 3 in every bitmap
    A, B, S, I = (b.column(i) for i in range(4))
    cases = [
        (col(0) > 3, pc.greater(A, 3)),
        ((col(0) > 3) | (col(1) < 0), pc.or_kleene(pc.greater(A, 3), pc.less(B, 0))),
        ((col(0) > 3) & (col(1) < 0), pc.and_kleene(pc.greater(A, 3), pc.less(B, 0))),
        (~((col(0) > 3) | (col(2) == "or")), pc.invert(pc.or_kleene(pc.greater(A, 3), pc.equal(S, "or")))),
        (((col(0) > 3) & ~(col(1) < 0)) | ((col(2) == "id") & (col(3) % 2 == 0)),
         pc.or_kleene(pc.and_kleene(pc.greater(A, 3), pc.invert(pc.less(B, 0))), pc.and_kleene(pc.equal(S, "id"), pc.equal(pc.bit_wise_and(I, 1), 0)))),
        (col(0).cast("int64") + col(1) > 0, pc.greater(pc.add(pc.cast(A, pa.int64()), B), 0)),
    ]
    for e, want in cases:
        got, _ = fb.selftest_eval_predicate(b, e)
        assert np.array_equal(got, want.fill_null(False).to_numpy(zero_copy_only=False)), fb.E.wrap(e).tokens


def test_value_lowering_matches_numpy():
    b = expr_batch(500, seed=2)
    c = cols(b)
    i32 = c["i32"]
    v, dt = fb.selftest_eval_value(b, 0.908 * col(0).cast("float64"))                        # q1, planner.rs:90
    assert dt == fb.FLOAT64 and np.array_equal(v.view(np.int64), (np.float64(0.908) * i32.astype(np.float64)).view(np.int64))
    v, dt = fb.selftest_eval_value(b, col(0) * col(7) + 7)                                   # Int32 arithmetic wraps to Int32
    assert dt == fb.INT64 or dt == fb.INT32
    v, dt = fb.selftest_eval_value(b, (col(1) - 3) * 2)
    assert dt == fb.INT64 and np.array_equal(v, (c["i64"] - 3) * 2)
    v, dt = fb.selftest_eval_value(b, col(3) / 4.0 - col(0).cast("float64"))
    assert dt == fb.FLOAT64 and np.array_equal(v.view(np.int64), (c["f64"] / 4.0 - i32.astype(np.float64)).view(np.int64))
    v, dt = fb.selftest_eval_value(b, col(4))
    assert v is None and dt == fb.TIMESTAMP                                                  # plain columns stay zero-copy
    v, dt = fb.selftest_eval_value(b, (col(3) * 2.5).cast("int64"))
    assert dt == fb.INT64 and np.array_equal(v, np.trunc(c["f64"] * 2.5).astype(np.int64))


def test_expression_errors():
    b = expr_batch(16)
    with pytest.raises(fb.FlockGpuError, match="Divide by zero") as info:
        fb.selftest_eval_predicate(b, col(0).cast("int64") % 0 == 0)
    assert info.value.code == _ffi.ERR_EXECUTION
    z = b.set_column(7, "pos", pa.array(np.zeros(16, np.int32)))
    with pytest.raises(fb.FlockGpuError, match="Divide by zero"):
        fb.selftest_eval_predicate(z, col(0).cast("int64") % col(7).cast("int64") == 0)
    with pytest.raises(fb.FlockGpuError) as info:      # (a+b)*(c+d): not a left-deep chain
        fb.selftest_eval_value(b, (col(0) + col(7)) * (col(0) - col(7)))
    assert info.value.code == _ffi.ERR_UNSUPPORTED
    with pytest.raises(fb.FlockGpuError) as info:
        fb.selftest_eval_predicate(b, col(99) == 1)
    assert info.value.code == _ffi.ERR_INVALID
    with pytest.raises(fb.FlockGpuError):
        fb.selftest_eval_predicate(b, col(0) + 1)      # not boolean


def test_nexgen_invariants():
    # generator counts (nexmark.rs:427-454 analogue): event mix 1:3:46
    assert nexgen.relation_counts(10_000) == (200, 600, 9200)
    ev = nexgen.generate(10_000, seed=5, batch_rows=4096)
    assert [sum(b.num_rows for b in ev[r]) for r in ("person", "auction", "bid")] == [200, 600, 9200]
    assert ev["bid"][0].schema.equals(nexgen.bid_schema()) and ev["bid"][0].num_rows == 4096
    assert ev["person"][0].schema.equals(nexgen.person_schema()) and ev["auction"][0].schema.equals(nexgen.auction_schema())
    p = pa.Table.from_batches(ev["person"])
    assert p["p_id"].to_pylist() == list(range(1000, 1200))
    assert set(p["state"].to_pylist()) <= set(nexgen.US_STATES)
    a = pa.Table.from_batches(ev["auction"])
    assert set(a["category"].to_pylist()) <= set(range(10, 15))
    assert all(1000 <= s < 1000 + 200 + 10 for s in a["seller"].to_pylist())


# ---- the arithmetic of the vectorised filter predicate (csrc/pred_i32.h), exactly as the GPU kernel runs it ---------------
@pytest.mark.parametrize("modulus", [0, 1, 2, 3, 6, 96, 123, 1000, 1 << 20, 3 << 29, (1 << 31) - 1])
def test_pred_i32_arithmetic_matches_truncated_remainder(modulus):
    """`CAST(x AS Int64) % m cmp c` with Rust / Arrow semantics (sign follows the dividend) for every comparison, boundary
    literals, negative dividends and INT_MIN -- through the same constants and per-row test the kernel uses."""
    import operator
    rng = np.random.default_rng(modulus + 1)
    n = 200_000
    x = rng.integers(-(1 << 31), 1 << 31, n).astype(np.int64)
    if modulus:
        x[::5] = rng.integers(-((1 << 31) // modulus), ((1 << 31) - 1) // modulus + 1, len(x[::5])) * modulus   # plenty of multiples
    x[:6] = [0, -(1 << 31), (1 << 31) - 1, -1, 1, -(1 << 31) + 1]
    lhs = np.fmod(x, modulus) if modulus else x
    ops = {fb.OP_EQ: operator.eq, fb.OP_NE: operator.ne, fb.OP_LT: operator.lt, fb.OP_LE: operator.le, fb.OP_GT: operator.gt, fb.OP_GE: operator.ge}
    literals = [0, 1, -1, 10, -7] + ([] if modulus else [-(1 << 31), (1 << 31) - 1, -(1 << 31) - 1, 1 << 31, 1 << 40, -(1 << 40)])
    modes = set()
    for cmp, fn in ops.items():
        for rhs in literals:
            keep, mode = fb.selftest_pred_i32(x, modulus, cmp, rhs)
            modes.add(mode)
            assert np.array_equal(keep, fn(lhs, rhs)), (modulus, cmp, rhs, mode)
    if modulus == 0:
        assert modes == {0}                      # every plain comparison is one affine range test
    elif modulus % 2:
        assert modes == {0, 1}                   # odd m: `% m (=|!=) 0` is the affine test, everything else Lemire
    else:
        assert modes == {1, 2}                   # even m: rotate test for divisibility


def test_stage_copy_is_exact(tmp_path):
    """The staging copy of the pageable feed uses non-temporal stores for the aligned body and memcpy for head and tail:
    every alignment / size combination must copy exactly n bytes (tests/cabi/stage_copy_test.cpp)."""
    import subprocess
    root = Path(__file__).resolve().parent.parent
    exe = tmp_path / "stage_copy_test"
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", str(root / "tests" / "cabi" / "stage_copy_test.cpp"),
                    str(root / "flock_b200" / "csrc" / "host" / "stream_copy.cpp"), "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr


def _import_ipc_without_a_device(schema: pa.Schema, frames) -> str:
    """flockgpu_table_import_ipc with a NULL context: the frames are validated BEFORE the context is looked at, so the error
    message tells whether validation passed ("null context handle") or what was wrong with the payload."""
    keep = [(pa.py_buffer(h), pa.py_buffer(b)) for h, b in frames]
    n = len(keep)
    hp = (C.c_void_p * max(n, 1))(*[h.address for h, _ in keep])
    hl = (C.c_int64 * max(n, 1))(*[h.size for h, _ in keep])
    bp = (C.c_void_p * max(n, 1))(*[b.address for _, b in keep])
    bl = (C.c_int64 * max(n, 1))(*[b.size for _, b in keep])
    c_schema = _ffi.ArrowSchema()
    schema._export_to_c(C.addressof(c_schema))
    out = C.c_void_p()
    try:
        rc = _ffi.lib.flockgpu_table_import_ipc(None, C.byref(c_schema), hp, hl, bp, bl, n, None, 0, C.byref(out))
    finally:
        if c_schema.release:
            C.CFUNCTYPE(None, C.c_void_p)(c_schema.release)(C.addressof(c_schema))
    assert rc == _ffi.ERR_INVALID or rc == _ffi.ERR_UNSUPPORTED, rc
    return _ffi.lib.flockgpu_last_error().decode()


def test_ipc_frames_are_validated_before_anything_reads_them():
    """A payload frame is untrusted input (flock/src/runtime/payload.rs:161-192 hands over what arrived in the Lambda
    event): lengths, offsets and buffer extents are checked against the bytes that came with them, on the host, before a
    device is involved."""
    import struct
    b = pa.RecordBatch.from_arrays([pa.array(np.arange(1000, dtype=np.int32)), pa.array(["s%d" % (i % 17) for i in range(1000)]),
                                    pa.array(np.arange(1000, dtype=np.int64), mask=np.arange(1000) % 3 == 0)], names=["a", "s", "v"])
    frame = lambda batch: (lambda m: (m.metadata.to_pybytes(), m.body.to_pybytes()))(pa.ipc.read_message(batch.serialize()))
    header, body = frame(b)
    ok = "null context handle"
    assert _import_ipc_without_a_device(b.schema, [(header, body)]) == ok
    assert _import_ipc_without_a_device(b.schema, [frame(b.slice(3, 200)), frame(b.slice(0, 0)), frame(b.slice(203))]) == ok
    # a body shorter than the buffers the header lists
    assert "outside the" in _import_ipc_without_a_device(b.schema, [(header, body[:len(body) // 2])])
    # a header cut short / garbage
    assert "flatbuffer" in _import_ipc_without_a_device(b.schema, [(header[:40], body)]) or "IPC header" in _import_ipc_without_a_device(b.schema, [(header[:40], body)])
    assert "IPC header" in _import_ipc_without_a_device(b.schema, [(b"\xff" * 64, body)])
    # a frame of another schema: fewer fields, or a narrower column where a wider one is declared
    assert "fields" in _import_ipc_without_a_device(b.schema, [frame(b.select(["a", "s"]))])
    wide = pa.schema([pa.field("a", pa.int64()), b.schema.field("s"), b.schema.field("v")])
    assert "value bytes" in _import_ipc_without_a_device(wide, [(header, body)])
    # Utf8 offsets that point past the value bytes: patch the LAST offset of column s inside the body
    off = np.frombuffer(pa.ipc.read_record_batch(pa.ipc.read_message(b.serialize()), b.schema).column(1).buffers()[1], dtype=np.int32)
    needle = struct.pack("<i", int(off[1000]))
    at = body.rfind(needle, 0, body.find(b"s0s1s2"))           # the offsets buffer sits right before the value bytes
    assert at > 0
    broken = body[:at] + struct.pack("<i", 1 << 30) + body[at + 4:]
    assert "offsets" in _import_ipc_without_a_device(b.schema, [(header, broken)])
    # a dictionary / schema message is not a data frame
    sink = pa.BufferOutputStream()
    with pa.ipc.new_stream(sink, b.schema):
        pass
    schema_msg = pa.ipc.read_message(sink.getvalue())
    assert "message type" in _import_ipc_without_a_device(b.schema, [(schema_msg.metadata.to_pybytes(), b"")])
