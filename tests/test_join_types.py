"""HashJoinExec Left / Right / Full / Semi / Anti without a GPU: the restatement (tests/join_oracle.py) against Acero over
the relation matrix, through plans at 1 and 8 Hash partitions, and the plan layer's unmarshal of every type."""
from __future__ import annotations

import json
import sys
from pathlib import Path

import pyarrow as pa
import pytest

import flock_b200 as fb
from flock_b200 import _ffi, plans

sys.path.insert(0, str(Path(__file__).resolve().parent))
import join_oracle as jo  # noqa: E402

TYPES = ["Left", "Right", "Full", "Semi", "Anti"]
REFERENCE_PLANS = Path(__file__).resolve().parent / "golden" / "reference_plans"
_SYNTH = jo.synthetic_cases()


@pytest.mark.parametrize("jt", TYPES)
@pytest.mark.parametrize("case", sorted(_SYNTH))
def test_oracle_matches_acero(case, jt):
    left, right, lk, rk = _SYNTH[case]
    want = jo.acero_join(left, right, lk, rk, jt)
    got = jo.join_tables(left, right, lk, rk, jt)
    jo.assert_same_rows(got, want, ordered=False)
    if jt in ("Semi", "Anti"):
        # left rows, once each, in left input order
        li, ri = jo.join_indices(jo.oracle._concat(left.to_batches(), left.schema), jo.oracle._concat(right.to_batches(), right.schema), lk, rk, jt)
        assert ri is None and (len(li) < 2 or (li[1:] > li[:-1]).all())


@pytest.mark.parametrize("jt", TYPES)
def test_oracle_matches_acero_nexmark(events_small, jt):
    for name, (left, right, lk, rk) in jo.nexmark_cases(events_small).items():
        jo.assert_same_rows(jo.join_tables(left, right, lk, rk, jt), jo.acero_join(left, right, lk, rk, jt), ordered=False)


def _join_plan(jt: str, n: int) -> dict:
    p = plans.coalesce_batches_exec(plans.repartition_hash(plans.memory_exec(plans.PERSON, [0, 1, 4]), [plans.column("p_id", 0)], n))
    a = plans.coalesce_batches_exec(plans.repartition_hash(plans.memory_exec(plans.AUCTION, [0, 7, 8]), [plans.column("seller", 1)], n))
    return plans.hash_join_exec(p, a, [(plans.column("p_id", 0), plans.column("seller", 1))], join_type=jt)


@pytest.mark.parametrize("n", [1, 8])
@pytest.mark.parametrize("jt", TYPES)
def test_plan_partitions(events_small, jt, n):
    """Hash-repartitioned on the keys, the partition-wise joins together equal the join of the whole relations."""
    srcs = [[events_small["person"]], [events_small["auction"]]]
    got = jo.execute_plan(_join_plan(jt, n), srcs)
    person = pa.Table.from_batches(events_small["person"]).select(["p_id", "name", "city"])
    auction = pa.Table.from_batches(events_small["auction"]).select(["a_id", "seller", "category"])
    jo.assert_same_rows(got, jo.acero_join(person, auction, [0], [1], jt), ordered=False)


@pytest.mark.parametrize("jt", TYPES)
def test_plan_with_an_empty_side(events_small, jt):
    """An empty input is still a side: Left / Full keep every person, Anti returns them all, Semi none."""
    srcs = [[events_small["person"]], [[pa.RecordBatch.from_arrays([pa.array([], f.type) for f in plans.AUCTION], schema=plans.AUCTION)]]]
    got = jo.execute_plan(_join_plan(jt, 8), srcs)
    n_p = sum(b.num_rows for b in events_small["person"])
    assert got.num_rows == {"Left": n_p, "Full": n_p, "Anti": n_p, "Right": 0, "Semi": 0}[jt]


def test_collect_left_over_partitions_is_refused(events_small):
    plan = _join_plan("Left", 8)
    plan["mode"] = "CollectLeft"
    plan["left"] = plans.coalesce_partitions_exec(plan["left"])
    with pytest.raises(jo.oracle.OracleError, match="CollectLeft"):
        jo.execute_plan(plan, [[events_small["person"]], [events_small["auction"]]])


def test_plans_keep_inner_by_default():
    """Existing plans serialise as before: the keyword defaults to Inner."""
    assert json.dumps(plans.q3()).count('"join_type": "Inner"') == 1
    assert plans.hash_join_exec({}, {}, [])["join_type"] == "Inner"


@pytest.mark.parametrize("jt", TYPES + ["Inner"])
def test_host_unmarshals_every_type(jt):
    s = fb.ExecutionContext(None, _join_plan(jt, 8)).plan_str(0)
    assert s.startswith(f"HashJoinExec: mode=Partitioned, join_type={jt}, on=[(p_id, seller)]")
    # the reference's own serialised join plan with its join_type replaced (the parse-only unmarshal the shim uses)
    ref = (REFERENCE_PLANS / "join.json").read_text()
    assert ref.count('"Inner"') == 1
    s = fb.ExecutionContext(None, ref.replace('"Inner"', f'"{jt}"')).plan_str(0)
    assert f"HashJoinExec: mode=Partitioned, join_type={jt}, on=[(a, c)]" in s


def test_host_refuses_unknown_join_type_and_cross_join():
    with pytest.raises(fb.FlockGpuError) as info:
        fb.ExecutionContext(None, _join_plan("LeftOuter", 8))
    assert info.value.code == _ffi.ERR_INVALID and "LeftOuter" in info.value.message
    cross = {"execution_plan": "cross_join_exec", "left": plans.q2(), "right": plans.q2()}
    with pytest.raises(fb.FlockGpuError) as info:
        fb.ExecutionContext(None, cross)
    assert info.value.code == _ffi.ERR_UNSUPPORTED


def test_python_join_type_names():
    with pytest.raises(ValueError, match="unknown join type"):
        fb.Context.hash_join(None, None, None, [0], [0], "outer")
