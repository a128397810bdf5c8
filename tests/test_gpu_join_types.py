"""HashJoinExec Left / Right / Full / Semi / Anti on the GPU against the CPU restatement (tests/join_oracle.py).

Every relation shape runs in both size orientations, so each type runs the form where its preserved (or filtered) side
is streamed and the form where it is hashed.  Left / Right / Full are compared as multisets, Semi / Anti in exact left
input order.  Also: the padded side's nullable flags, each type at the q8 one-GPU share, a q13-shaped plan (NULLs made by
the join flow through COUNT(col) and a Final aggregate), Inner through both C entry points, and the launch profile of the
Inner plans q3 / q5 / q8 against the one recorded before the other join types existed.
"""
from __future__ import annotations

import ctypes as C
import json
import sys
from pathlib import Path

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pytest

import flock_b200 as fb
from flock_b200 import _ffi, plans

sys.path.insert(0, str(Path(__file__).resolve().parent))
import join_oracle as jo  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
TYPES = ["Left", "Right", "Full", "Semi", "Anti"]


def _batches(t: pa.Table) -> list[pa.RecordBatch]:
    t = t.combine_chunks()
    if t.num_rows == 0:
        return [pa.RecordBatch.from_arrays([pa.array([], f.type) for f in t.schema], schema=t.schema)]
    return t.to_batches()


def _gpu_join(ctx, left: pa.Table, right: pa.Table, lk, rk, jt: str) -> pa.Table:
    tl, tr = ctx.import_batches(_batches(left)), ctx.import_batches(_batches(right))
    return ctx.hash_join(tl, tr, lk, rk, jt.lower()).to_arrow()


_SYNTH = jo.synthetic_cases()


@pytest.mark.parametrize("jt", TYPES)
@pytest.mark.parametrize("case", sorted(_SYNTH))
def test_join_type_matches_oracle(gpu_ctx, case, jt):
    left, right, lk, rk = _SYNTH[case]
    got = _gpu_join(gpu_ctx, left, right, lk, rk, jt)
    want = jo.join_tables(left, right, lk, rk, jt)
    jo.assert_same_rows(got, want, ordered=jt in ("Semi", "Anti"))
    # the padded side is nullable whatever the data; Semi / Anti return the left columns only
    n_left = left.num_columns
    assert got.num_columns == (n_left if jt in ("Semi", "Anti") else n_left + right.num_columns)
    if jt in ("Right", "Full"):
        assert all(f.nullable for f in list(got.schema)[:n_left])
    if jt in ("Left", "Full"):
        assert all(f.nullable for f in list(got.schema)[n_left:])


@pytest.mark.parametrize("jt", TYPES)
def test_join_type_nexmark(gpu_ctx, events_small, jt):
    for name, (left, right, lk, rk) in jo.nexmark_cases(events_small).items():
        got = _gpu_join(gpu_ctx, left, right, lk, rk, jt)
        want = jo.join_tables(left, right, lk, rk, jt)
        jo.assert_same_rows(got, want, ordered=jt in ("Semi", "Anti"))


def test_join_type_q8_share(gpu_ctx):
    """Each type once at the q8 one-GPU share: 2.5 M persons, 7.5 M auctions (sellers drawn past the last person too,
    so that both sides have rows without a partner)."""
    rng = np.random.default_rng(5)
    n_p, n_a = 2_500_000, 7_500_000
    person = pa.table({"p_id": pa.array(rng.permutation(n_p).astype(np.int32)), "v": pa.array(rng.integers(0, 1 << 30, n_p).astype(np.int64))})
    auction = pa.table({"a_id": pa.array(np.arange(n_a, dtype=np.int32)), "seller": pa.array(rng.integers(0, n_p + n_p // 4, n_a).astype(np.int32))})
    for jt in TYPES:
        for left, right, lk, rk in ((person, auction, [0], [1]), (auction, person, [1], [0])):
            got = _gpu_join(gpu_ctx, left, right, lk, rk, jt)
            li, ri = jo.join_indices(jo.oracle._concat(left.to_batches(), left.schema), jo.oracle._concat(right.to_batches(), right.schema), lk, rk, jt)
            assert got.num_rows == len(li), (jt, got.num_rows, len(li))
            if ri is None:
                # exact order: the left rows selected, as row numbers of `left` through its unique first column / a_id
                key = got.column(0).to_numpy()
                assert np.array_equal(key, left.column(0).to_numpy()[li]), jt
            else:
                lid = np.where(li >= 0, left.column(0).to_numpy()[np.maximum(li, 0)], -1)
                rid = np.where(ri >= 0, right.column(0).to_numpy()[np.maximum(ri, 0)], -1)
                g_l = got.column(0).fill_null(-1).to_numpy()
                g_r = got.column(left.num_columns).fill_null(-1).to_numpy()
                w = np.lexsort((rid, lid))
                g = np.lexsort((g_r, g_l))
                assert np.array_equal(g_l[g], lid[w]) and np.array_equal(g_r[g], rid[w]), jt


def _q13_plan(n: int) -> dict:
    """persons LEFT JOIN auctions ON p_id = seller -> COUNT(a_id) per p_id -> COUNT(*) per count (TPC-H q13's shape)."""
    p = plans.coalesce_batches_exec(plans.repartition_hash(plans.repartition_rr(plans.memory_exec(plans.PERSON, [0]), n), [plans.column("p_id", 0)], n))
    a = plans.coalesce_batches_exec(plans.repartition_hash(plans.repartition_rr(plans.memory_exec(plans.AUCTION, [0, 7]), n), [plans.column("seller", 1)], n))
    join = plans.hash_join_exec(p, a, [(plans.column("p_id", 0), plans.column("seller", 1))], join_type="Left")
    cnt = plans.aggregate_expr("count", "COUNT(a_id)", plans.column("a_id", 1), "UInt64")
    per_person = plans.two_phase_aggregate([("p_id", 0)], [cnt], plans.coalesce_batches_exec(join), n)
    c = plans.projection_exec([(plans.column("COUNT(a_id)", 1), "c_count")], per_person)
    star = plans.aggregate_expr("count", "COUNT(UInt8(1))", plans.literal("UInt8", 1), "UInt64")
    return plans.two_phase_aggregate([("c_count", 0)], [star], c, n)


@pytest.mark.parametrize("n", [1, 8])
def test_q13_shaped_plan(gpu_ctx, events_small, n):
    ec = fb.ExecutionContext(gpu_ctx, _q13_plan(n))
    ec.feed_data_sources([[events_small["person"]], [events_small["auction"]]])
    got = pa.Table.from_batches(ec.execute()[0]).combine_chunks()
    ec.close()
    person = pa.Table.from_batches(events_small["person"]).select(["p_id"])
    auction = pa.Table.from_batches(events_small["auction"]).select(["a_id", "seller"])
    j = person.join(auction, keys="p_id", right_keys="seller", join_type="left outer", coalesce_keys=False)
    per = j.group_by("p_id").aggregate([("a_id", "count")])                       # COUNT(col): NULLs not counted
    dist = per.group_by("a_id_count").aggregate([([], "count_all")])
    want = sorted(zip(pc.cast(dist["a_id_count"], pa.uint64()).to_pylist(), dist["count_all"].to_pylist()))
    have = sorted(zip(got.column(0).to_pylist(), got.column(1).to_pylist()))
    assert have == want
    assert any(c == 0 for c, _ in have), "no person without auctions: the padded rows were not exercised"


def _both_entry_points(ctx, left, right, lk, rk):
    tl, tr = ctx.import_batches(_batches(left)), ctx.import_batches(_batches(right))
    lka, rka = (C.c_int32 * len(lk))(*lk), (C.c_int32 * len(rk))(*rk)
    a, b = C.c_void_p(), C.c_void_p()
    _ffi.check(_ffi.lib.flockgpu_hash_join(ctx.handle, tl.handle, tr.handle, lka, rka, len(lk), C.byref(a)))
    _ffi.check(_ffi.lib.flockgpu_hash_join_typed(ctx.handle, tl.handle, tr.handle, lka, rka, len(lk), 0, C.byref(b)))
    return fb.Table(ctx, a.value).to_arrow(), fb.Table(ctx, b.value).to_arrow()


def test_inner_entry_points_bit_identical(gpu_ctx, events_small):
    # unique keys on the hashed side (persons): the output order is fixed by the probe order, so the bytes must agree
    ta, tb = _both_entry_points(gpu_ctx, *jo.nexmark_cases(events_small)["persons_auctions"])
    assert ta.schema == tb.schema and ta.equals(tb)
    # duplicate keys: the order of a key's build rows is whatever the build's atomics made it, in either entry point
    ta, tb = _both_entry_points(gpu_ctx, *_SYNTH["utf8_null_keys_both_sl"])
    assert ta.schema == tb.schema and jo.canonical(ta).equals(jo.canonical(tb))
    tl, tr = gpu_ctx.import_batches(_batches(_SYNTH["one_row_left"][0])), gpu_ctx.import_batches(_batches(_SYNTH["one_row_left"][1]))
    lka = (C.c_int32 * 1)(0)
    with pytest.raises(fb.FlockGpuError) as info:
        c = C.c_void_p()
        _ffi.check(_ffi.lib.flockgpu_hash_join_typed(gpu_ctx.handle, tl.handle, tr.handle, lka, lka, 1, 6, C.byref(c)))
    assert info.value.code == _ffi.ERR_INVALID


@pytest.mark.parametrize("jt", TYPES)
def test_reference_format_plan_on_gpu(gpu_ctx, events_small, jt):
    """A join plan of every type through unmarshal -> feed -> execute equals the restatement, at 8 partitions."""
    plan = join_plan(jt, 8)
    srcs = [[events_small["person"]], [events_small["auction"]]]
    ec = fb.ExecutionContext(gpu_ctx, plan)
    ec.feed_data_sources(srcs)
    got = pa.Table.from_batches(ec.execute()[0])
    ec.close()
    want = jo.execute_plan(plan, srcs)
    jo.assert_same_rows(got, want, ordered=False)


def join_plan(jt: str, n: int) -> dict:
    p = plans.coalesce_batches_exec(plans.repartition_hash(plans.memory_exec(plans.PERSON, [0, 1, 4]), [plans.column("p_id", 0)], n))
    a = plans.coalesce_batches_exec(plans.repartition_hash(plans.memory_exec(plans.AUCTION, [0, 7, 8]), [plans.column("seller", 1)], n))
    return plans.hash_join_exec(p, a, [(plans.column("p_id", 0), plans.column("seller", 1))], join_type=jt)


def test_inner_launch_profile_unchanged():
    """q3, q5 and q8 launch the same kernels the same number of times as before the other join types existed."""
    sys.path.insert(0, str(ROOT / "tools"))
    import launch_profile
    from flock_b200 import nexgen
    have = launch_profile.profile(fb, nexgen, plans)
    want = json.loads((ROOT / "tests" / "golden" / "launch_profile_q3_q5_q8.json").read_text())
    assert have == want
