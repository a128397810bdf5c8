"""NEXMark physical plans in the reference's own serde-JSON plan format.

The reference serialises ``Arc<dyn ExecutionPlan>`` with typetag tags ("execution_plan": "filter_exec",
"physical_expr": "binary_expr", ...; fixtures flock/src/tests/data/plan/{simple_select,aggregate,join}.json)
and ships the string in the Lambda environment (flock/src/runtime/context.rs:366-398).  No Rust
toolchain exists here, so these builders write the same JSON by hand, following the physical plans the
reference's own tests print (flock/src/distributed_plan/planner.rs:86-255) and SURVEY.md Appendix B.
Both the GPU executor (flock_b200.ExecutionContext) and the CPU oracle execute exactly this JSON.
"""
from __future__ import annotations

import pyarrow as pa

from . import nexgen

TARGET_PARTITIONS = 8     # flock/src/configs/flock.toml:113
TARGET_BATCH_SIZE = 4096  # CoalesceBatchesExec default seen in every plan dump


# ---- data types / schema ---------------------------------------------------------------------------
def data_type_json(t: pa.DataType):
    if pa.types.is_int32(t): return "Int32"
    if pa.types.is_uint32(t): return "UInt32"
    if pa.types.is_int64(t): return "Int64"
    if pa.types.is_uint64(t): return "UInt64"
    if pa.types.is_float64(t): return "Float64"
    if pa.types.is_string(t): return "Utf8"
    if pa.types.is_timestamp(t):
        unit = {"s": "Second", "ms": "Millisecond", "us": "Microsecond", "ns": "Nanosecond"}[t.unit]
        return {"Timestamp": [unit, t.tz]}
    raise TypeError(f"unsupported type {t}")


def schema_json(schema: pa.Schema) -> dict:
    md = {k.decode(): v.decode() for k, v in (schema.metadata or {}).items()}
    return {"fields": [{"name": f.name, "data_type": data_type_json(f.type), "nullable": f.nullable,
                        "dict_id": 0, "dict_is_ordered": False} for f in schema],
            "metadata": md}


# ---- physical expressions ----------------------------------------------------------------------------
def column(name: str, index: int) -> dict:
    return {"physical_expr": "column", "name": name, "index": index}


def literal(type_name: str, value) -> dict:
    return {"physical_expr": "literal", "value": {type_name: value}}


def binary(left: dict, op: str, right: dict) -> dict:
    return {"physical_expr": "binary_expr", "left": left, "op": op, "right": right}


def cast(expr: dict, type_json) -> dict:
    return {"physical_expr": "cast_expr", "expr": expr, "cast_type": type_json}


def try_cast(expr: dict, type_json) -> dict:
    return {"physical_expr": "try_cast_expr", "expr": expr, "cast_type": type_json}


# ---- execution plans -------------------------------------------------------------------------------------
def memory_exec(schema: pa.Schema, projection: list[int] | None) -> dict:
    return {"execution_plan": "memory_exec", "schema": schema_json(schema), "projection": projection}


def projection_exec(exprs: list[tuple[dict, str]], input: dict) -> dict:
    return {"execution_plan": "projection_exec", "expr": [[e, n] for e, n in exprs], "input": input}


def filter_exec(predicate: dict, input: dict) -> dict:
    return {"execution_plan": "filter_exec", "predicate": predicate, "input": input}


def coalesce_batches_exec(input: dict, target_batch_size: int = TARGET_BATCH_SIZE) -> dict:
    return {"execution_plan": "coalesce_batches_exec", "input": input, "target_batch_size": target_batch_size}


def coalesce_partitions_exec(input: dict) -> dict:
    return {"execution_plan": "coalesce_partitions_exec", "input": input}


def repartition_rr(input: dict, n: int = TARGET_PARTITIONS) -> dict:
    return {"execution_plan": "repartition_exec", "input": input, "partitioning": {"RoundRobinBatch": n}}


def repartition_hash(input: dict, exprs: list[dict], n: int = TARGET_PARTITIONS) -> dict:
    return {"execution_plan": "repartition_exec", "input": input, "partitioning": {"Hash": [exprs, n]}}


def aggregate_expr(func: str, name: str, expr: dict, data_type) -> dict:
    return {"aggregate_expr": func, "name": name, "expr": expr, "data_type": data_type, "nullable": True}


def hash_aggregate_exec(mode: str, group_expr: list[tuple[dict, str]], aggr_expr: list[dict], input: dict) -> dict:
    return {"execution_plan": "hash_aggregate_exec", "mode": mode, "group_expr": [[e, n] for e, n in group_expr],
            "aggr_expr": aggr_expr, "input": input}


def hash_join_exec(left: dict, right: dict, on: list[tuple[dict, dict]], mode: str = "Partitioned", join_type: str = "Inner") -> dict:
    """join_type: DataFusion 6 JoinType -- Inner, Left, Right, Full, Semi or Anti."""
    return {"execution_plan": "hash_join_exec", "join_type": join_type, "mode": mode, "left": left, "right": right,
            "on": [[{"name": l["name"], "index": l["index"]}, {"name": r["name"], "index": r["index"]}] for l, r in on]}


def sort_exec(exprs: list[tuple[dict, bool, bool]], input: dict) -> dict:
    """flock/src/tests/data/plan/join.json: {"expr": [{"expr": column, "options": {"descending", "nulls_first"}}]}."""
    return {"execution_plan": "sort_exec", "input": input,
            "expr": [{"expr": e, "options": {"descending": desc, "nulls_first": nf}} for e, desc, nf in exprs]}


def global_limit_exec(input: dict, limit: int) -> dict:
    return {"execution_plan": "global_limit_exec", "input": input, "limit": limit}


def row_number_window(name: str, partition_by: list[dict], order_by: list[tuple[dict, bool, bool]], input: dict) -> dict:
    """WindowAggExec with one ROW_NUMBER() (the only window function NEXMark q6 uses).  No fixture of the reference
    serialises this node; the layout follows DataFusion 6's WindowAggExec { input, window_expr } and its
    BuiltInWindowExpr { fun, name, partition_by, order_by } fields."""
    return {"execution_plan": "window_agg_exec", "input": input,
            "window_expr": [{"window_expr": "built_in_window_expr", "fun": "RowNumber", "name": name, "partition_by": partition_by,
                             "order_by": [{"expr": e, "options": {"descending": desc, "nulls_first": nf}} for e, desc, nf in order_by]}]}


def two_phase_aggregate(group: list[tuple[str, int]], aggrs: list[dict], input: dict, n: int = TARGET_PARTITIONS) -> dict:
    """Partial -> RepartitionExec(Hash[group]) -> CoalesceBatches -> FinalPartitioned (stage.rs:597-601);
    without group columns: Partial -> CoalescePartitions -> Final (stage.rs:535-537)."""
    gexpr = [(column(nm, ix), nm) for nm, ix in group]
    partial = hash_aggregate_exec("Partial", gexpr, aggrs, input)
    if not group:
        return hash_aggregate_exec("Final", [], aggrs, coalesce_partitions_exec(partial))
    gfinal = [(column(nm, i), nm) for i, (nm, _) in enumerate(group)]
    shuffled = coalesce_batches_exec(repartition_hash(partial, [column(nm, i) for i, (nm, _) in enumerate(group)], n))
    return hash_aggregate_exec("FinalPartitioned", gfinal, aggrs, shuffled)


# ---- NEXMark q1..q8 (benchmarks/src/nexmark/query/qN.sql) -------------------------------------------------
BID, AUCTION, PERSON = nexgen.bid_schema(), nexgen.auction_schema(), nexgen.person_schema()
TS_MS = {"Timestamp": ["Millisecond", None]}


def q1(n: int = TARGET_PARTITIONS) -> dict:
    """planner.rs:90-92  SELECT auction, bidder, 0.908 * price AS price, b_date_time FROM bid"""
    scan = repartition_rr(memory_exec(BID, [0, 1, 2, 3]), n)
    return projection_exec([
        (column("auction", 0), "auction"), (column("bidder", 1), "bidder"),
        (binary(literal("Float64", 0.908), "Multiply", cast(column("price", 2), "Float64")), "price"),
        (column("b_date_time", 3), "b_date_time")], scan)


def q2(n: int = TARGET_PARTITIONS) -> dict:
    """planner.rs:120-124  SELECT auction, price FROM bid WHERE auction % 123 = 0"""
    scan = repartition_rr(memory_exec(BID, [0, 2]), n)
    pred = binary(binary(cast(column("auction", 0), "Int64"), "Modulo", literal("Int64", 123)), "Eq", literal("Int64", 0))
    return projection_exec([(column("auction", 0), "auction"), (column("price", 1), "price")],
                           coalesce_batches_exec(filter_exec(pred, scan)))


def q3_stage0(n: int = TARGET_PARTITIONS) -> list[dict]:
    """planner.rs:151-163: the two shuffle stages (auction side, person side)."""
    a_scan = repartition_rr(memory_exec(AUCTION, [0, 7, 8]), n)
    a_pred = binary(cast(column("category", 2), "Int64"), "Eq", literal("Int64", 10))
    a = coalesce_batches_exec(repartition_hash(coalesce_batches_exec(filter_exec(a_pred, a_scan)), [column("seller", 1)], n))
    p_scan = repartition_rr(memory_exec(PERSON, [0, 1, 4, 5]), n)
    st = column("state", 3)
    p_pred = binary(binary(binary(st, "Eq", literal("Utf8", "or")), "Or", binary(st, "Eq", literal("Utf8", "id"))),
                    "Or", binary(st, "Eq", literal("Utf8", "ca")))
    p = coalesce_batches_exec(repartition_hash(coalesce_batches_exec(filter_exec(p_pred, p_scan)), [column("p_id", 0)], n))
    return [a, p]


def q3(n: int = TARGET_PARTITIONS) -> dict:
    """planner.rs:151-171 as ONE plan (centralized mode runs the whole plan in one worker,
    benchmarks/src/nexmark/main.rs:209-214): auction JOIN person ON seller = p_id."""
    a, p = q3_stage0(n)
    join = hash_join_exec(a, p, [(column("seller", 1), column("p_id", 0))])
    return projection_exec([(column("name", 4), "name"), (column("city", 5), "city"), (column("state", 6), "state"),
                            (column("a_id", 0), "a_id")], coalesce_batches_exec(join))


def _count_by_auction(n: int) -> dict:
    scan = repartition_rr(memory_exec(BID, [0]), n)
    cnt = aggregate_expr("count", "COUNT(UInt8(1))", literal("UInt8", 1), "UInt64")
    return two_phase_aggregate([("auction", 0)], [cnt], scan, n)


def q5(n: int = TARGET_PARTITIONS) -> dict:
    """SURVEY.md Appendix B (types q5_plan.fmt): AuctionBids JOIN MaxBids ON num = maxn.  The COUNT-by-auction
    subtree appears twice, exactly as DataFusion 6 plans it (no common-subexpression elimination)."""
    left = projection_exec([(column("auction", 0), "auction"), (column("COUNT(UInt8(1))", 1), "num")], _count_by_auction(n))
    nums = projection_exec([(column("COUNT(UInt8(1))", 1), "num")], _count_by_auction(n))
    mx = aggregate_expr("max", "MAX(CountBids.num)", column("num", 0), "UInt64")
    right = projection_exec([(column("MAX(CountBids.num)", 0), "maxn")], two_phase_aggregate([], [mx], nums, n))
    lsh = coalesce_batches_exec(repartition_hash(left, [column("num", 1)], n))
    rsh = coalesce_batches_exec(repartition_hash(right, [column("maxn", 0)], n))
    join = hash_join_exec(lsh, rsh, [(column("num", 1), column("maxn", 0))])
    return projection_exec([(column("auction", 0), "auction"), (column("num", 1), "num")], coalesce_batches_exec(join))


def q8(n: int = TARGET_PARTITIONS) -> dict:
    """SURVEY.md Appendix B (q8_plan.fmt): P(p_id, name GROUP BY) JOIN A(seller GROUP BY) ON p_id = seller."""
    p_scan = repartition_rr(memory_exec(PERSON, [0, 1]), n)
    P = two_phase_aggregate([("p_id", 0), ("name", 1)], [], p_scan, n)
    a_scan = repartition_rr(memory_exec(AUCTION, [7]), n)
    A = two_phase_aggregate([("seller", 0)], [], a_scan, n)
    lsh = coalesce_batches_exec(repartition_hash(P, [column("p_id", 0)], n))
    rsh = coalesce_batches_exec(repartition_hash(A, [column("seller", 0)], n))
    join = hash_join_exec(lsh, rsh, [(column("p_id", 0), column("seller", 0))])
    return projection_exec([(column("p_id", 0), "p_id"), (column("name", 1), "name")], coalesce_batches_exec(join))


def q4(n: int = TARGET_PARTITIONS) -> dict:
    """benchmarks/src/nexmark/query/q4.sql, types q4_plan.fmt:
       SELECT category, AVG(final) FROM (SELECT MAX(price) AS final, category FROM auction JOIN bid ON a_id = auction
       WHERE b_date_time BETWEEN a_date_time AND expires GROUP BY a_id, category) GROUP BY category.
    Physical shape as DataFusion 6 builds it: Hash-repartitioned Partitioned join, Filter (BETWEEN = two comparisons),
    two two-phase aggregates."""
    a_scan = repartition_rr(memory_exec(AUCTION, [0, 5, 6, 8]), n)     # a_id, a_date_time, expires, category
    b_scan = repartition_rr(memory_exec(BID, [0, 2, 3]), n)            # auction, price, b_date_time
    lsh = coalesce_batches_exec(repartition_hash(a_scan, [column("a_id", 0)], n))
    rsh = coalesce_batches_exec(repartition_hash(b_scan, [column("auction", 0)], n))
    join = coalesce_batches_exec(hash_join_exec(lsh, rsh, [(column("a_id", 0), column("auction", 0))]))
    # a_id 0, a_date_time 1, expires 2, category 3, auction 4, price 5, b_date_time 6
    between = binary(binary(column("b_date_time", 6), "GtEq", column("a_date_time", 1)), "And",
                     binary(column("b_date_time", 6), "LtEq", column("expires", 2)))
    filt = coalesce_batches_exec(filter_exec(between, join))
    mx = aggregate_expr("max", "MAX(bid.price)", column("price", 5), "Int32")
    inner = two_phase_aggregate([("a_id", 0), ("category", 3)], [mx], filt, n)           # a_id, category, MAX(bid.price)
    q = projection_exec([(column("MAX(bid.price)", 2), "final"), (column("category", 1), "category")], inner)
    avg = aggregate_expr("avg", "AVG(Q.final)", column("final", 0), "Float64")
    outer = two_phase_aggregate([("category", 1)], [avg], q, n)
    return projection_exec([(column("category", 0), "category"), (column("AVG(Q.final)", 1), "AVG(Q.final)")], outer)


def q7(n: int = TARGET_PARTITIONS) -> dict:
    """benchmarks/src/nexmark/query/q7.sql, types q7_plan.fmt:
       SELECT auction, price, bidder, b_date_time FROM bid JOIN (SELECT MAX(price) AS maxprice FROM bid) ON price = maxprice."""
    bid = repartition_rr(memory_exec(BID, [0, 1, 2, 3]), n)
    mx = aggregate_expr("max", "MAX(bid.price)", column("price", 2), "Int32")
    b1 = projection_exec([(column("MAX(bid.price)", 0), "maxprice")],
                         two_phase_aggregate([], [mx], repartition_rr(memory_exec(BID, [0, 1, 2, 3]), n), n))
    lsh = coalesce_batches_exec(repartition_hash(bid, [column("price", 2)], n))
    rsh = coalesce_batches_exec(repartition_hash(b1, [column("maxprice", 0)], n))
    join = hash_join_exec(lsh, rsh, [(column("price", 2), column("maxprice", 0))])
    return projection_exec([(column("auction", 0), "auction"), (column("price", 2), "price"), (column("bidder", 1), "bidder"),
                            (column("b_date_time", 3), "b_date_time")], coalesce_batches_exec(join))


def q6(n: int = TARGET_PARTITIONS) -> dict:
    """benchmarks/src/nexmark/query/q6.sql, types q6_plan.fmt: average selling price of each seller's last ten closed
    auctions.  SortExec + WindowAggExec(ROW_NUMBER) on top of q4's join and BETWEEN filter (SURVEY section 8f rank 3)."""
    a_scan = repartition_rr(memory_exec(AUCTION, [0, 5, 6, 7]), n)     # a_id, a_date_time, expires, seller
    b_scan = repartition_rr(memory_exec(BID, [0, 2, 3]), n)            # auction, price, b_date_time
    lsh = coalesce_batches_exec(repartition_hash(a_scan, [column("a_id", 0)], n))
    rsh = coalesce_batches_exec(repartition_hash(b_scan, [column("auction", 0)], n))
    join = coalesce_batches_exec(hash_join_exec(lsh, rsh, [(column("a_id", 0), column("auction", 0))]))
    # a_id 0, a_date_time 1, expires 2, seller 3, auction 4, price 5, b_date_time 6
    between = binary(binary(column("b_date_time", 6), "GtEq", column("a_date_time", 1)), "And",
                     binary(column("b_date_time", 6), "LtEq", column("expires", 2)))
    filt = coalesce_partitions_exec(coalesce_batches_exec(filter_exec(between, join)))
    w1_name = "ROW_NUMBER() PARTITION BY [#auction.a_id] ORDER BY [#bid.price DESC NULLS FIRST]"
    w1 = row_number_window(w1_name, [column("a_id", 0)], [(column("price", 5), True, True)],
                           sort_exec([(column("a_id", 0), False, False), (column("price", 5), True, True)], filt))
    # window column first: rn 0, a_id 1, a_date_time 2, expires 3, seller 4, auction 5, price 6, b_date_time 7
    winners = coalesce_batches_exec(filter_exec(binary(column(w1_name, 0), "Eq", literal("UInt64", 1)), w1))
    q = projection_exec([(column("seller", 4), "seller"), (column("a_id", 1), "a_id"), (column("price", 6), "price"),
                         (column("b_date_time", 7), "b_date_time"), (column(w1_name, 0), "price_rank")], winners)
    q_sorted = sort_exec([(column("a_id", 1), False, False), (column("price", 2), True, True)], q)       # ORDER BY a_id, price DESC of subquery Q
    q2 = projection_exec([(column("seller", 0), "seller"), (column("price", 2), "price"), (column("b_date_time", 3), "b_date_time"),
                          (column("price_rank", 4), "price_rank")], q_sorted)
    w2_name = "ROW_NUMBER() PARTITION BY [#Q.seller] ORDER BY [#Q.b_date_time DESC NULLS FIRST]"
    w2 = row_number_window(w2_name, [column("seller", 0)], [(column("b_date_time", 2), True, True)],
                           sort_exec([(column("seller", 0), False, False), (column("b_date_time", 2), True, True)], q2))
    # rn 0, seller 1, price 2, b_date_time 3, price_rank 4
    last10 = coalesce_batches_exec(filter_exec(binary(column(w2_name, 0), "LtEq", literal("UInt64", 10)), w2))
    r = projection_exec([(column("seller", 1), "seller"), (column("price", 2), "price"), (column(w2_name, 0), "time_rank")], last10)
    avg = aggregate_expr("avg", "AVG(R.price)", column("price", 1), "Float64")
    outer = two_phase_aggregate([("seller", 0)], [avg], repartition_rr(r, n), n)
    return projection_exec([(column("seller", 0), "seller"), (column("AVG(R.price)", 1), "AVG(R.price)")], outer)


QUERIES = {"q1": q1, "q2": q2, "q3": q3, "q4": q4, "q5": q5, "q6": q6, "q7": q7, "q8": q8}
GPU_QUERIES = list(QUERIES)
# relations each query feeds, in feed order (flock/src/datasource/nexmark/nexmark.rs:181-203); q5 scans bid
# twice, and feed_data_sources hands one source to one leaf (context.rs:293-303), so bid is fed twice.
SOURCES = {"q1": ["bid"], "q2": ["bid"], "q3": ["auction", "person"], "q4": ["auction", "bid"], "q5": ["bid", "bid"],
           "q6": ["auction", "bid"], "q7": ["bid", "bid"], "q8": ["person", "auction"]}
