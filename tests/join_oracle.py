"""Restatement of HashJoinExec for every DataFusion 6 join type, and Acero as its independent second implementation.

TEST INFRASTRUCTURE ONLY.  The row pairs come from the oracle's Inner join (oracle.hash_join over the rows whose keys
are not NULL, with each side's row numbers carried along as one more column); the join types are derived from those
pairs exactly as SURVEY.md Appendix C states them:

    Inner   the pairs
    Left    the pairs, then every left row in no pair (right side NULL), in left order
    Right   the pairs, then every right row in no pair (left side NULL), in right order
    Full    the pairs, the unmatched right rows, the unmatched left rows
    Semi    every left row in some pair, once, in left order (left columns only)
    Anti    every left row in no pair, in left order (left columns only)

A row whose key is NULL is in no pair (NULL != NULL) but is still a row of its side.  The padded side's fields are
nullable.  `TypedPlanExecutor` runs plans whose HashJoinExec nodes carry any of these types; every other node is the
oracle's own.
"""
from __future__ import annotations

import numpy as np
import pyarrow as pa

import oracle

JOIN_TYPES = ("Inner", "Left", "Right", "Full", "Semi", "Anti")
LEFT_PRESERVING = ("Left", "Full", "Semi", "Anti")      # types whose output depends on the left rows without a match
ACERO_TYPES = {"Inner": "inner", "Left": "left outer", "Right": "right outer", "Full": "full outer",
               "Semi": "left semi", "Anti": "left anti"}


def _null_key_rows(batch: pa.RecordBatch, keys: list[int]) -> np.ndarray:
    null = np.zeros(batch.num_rows, bool)
    for k in keys:
        c = batch.column(k)
        if c.null_count:
            null |= c.is_null().to_numpy(zero_copy_only=False)
    return null


def _key_batch(batch: pa.RecordBatch, keys: list[int], rows: np.ndarray) -> pa.RecordBatch:
    idx = pa.array(rows, pa.int64())
    cols = [batch.column(k).take(idx) for k in keys] + [pa.array(rows, pa.int64())]
    return pa.RecordBatch.from_arrays(cols, names=[f"k{i}" for i in range(len(keys))] + ["row"])


def join_indices(left: pa.RecordBatch, right: pa.RecordBatch, lkeys: list[int], rkeys: list[int], join_type: str):
    """(left rows, right rows) as int64 arrays, -1 where that side is padded; Semi / Anti: (left rows, None)."""
    if join_type not in JOIN_TYPES:
        raise oracle.OracleError(f"oracle: unknown join type {join_type}")
    lsel = np.nonzero(~_null_key_rows(left, lkeys))[0]
    rsel = np.nonzero(~_null_key_rows(right, rkeys))[0]
    n = len(lkeys)
    if len(lsel) and len(rsel):
        pairs = oracle.hash_join(_key_batch(left, lkeys, lsel), _key_batch(right, rkeys, rsel), list(range(n)), list(range(n)))
        li = pairs.column(n).to_numpy().astype(np.int64)
        ri = pairs.column(2 * n + 1).to_numpy().astype(np.int64)
    else:
        li = ri = np.zeros(0, np.int64)
    l_matched = np.zeros(left.num_rows, bool)
    l_matched[li] = True
    r_matched = np.zeros(right.num_rows, bool)
    r_matched[ri] = True
    if join_type == "Semi":
        return np.nonzero(l_matched)[0].astype(np.int64), None
    if join_type == "Anti":
        return np.nonzero(~l_matched)[0].astype(np.int64), None
    parts_l, parts_r = [li], [ri]
    if join_type in ("Right", "Full"):
        un = np.nonzero(~r_matched)[0].astype(np.int64)
        parts_l.append(np.full(len(un), -1, np.int64))
        parts_r.append(un)
    if join_type in ("Left", "Full"):
        un = np.nonzero(~l_matched)[0].astype(np.int64)
        parts_l.append(un)
        parts_r.append(np.full(len(un), -1, np.int64))
    return np.concatenate(parts_l), np.concatenate(parts_r)


def _take(batch: pa.RecordBatch, rows: np.ndarray, padded: bool) -> tuple[list[pa.Array], list[pa.Field]]:
    idx = pa.array(rows, pa.int64(), mask=rows < 0)
    cols = [c.take(idx) for c in batch.columns]
    fields = [f.with_nullable(True) if padded else f for f in batch.schema]
    return cols, fields


def join_batches(left: pa.RecordBatch, right: pa.RecordBatch, lkeys: list[int], rkeys: list[int], join_type: str) -> pa.RecordBatch:
    li, ri = join_indices(left, right, lkeys, rkeys, join_type)
    lcols, lfields = _take(left, li, join_type in ("Right", "Full"))
    if ri is None:
        return pa.RecordBatch.from_arrays(lcols, schema=pa.schema(lfields))
    rcols, rfields = _take(right, ri, join_type in ("Left", "Full"))
    return pa.RecordBatch.from_arrays(lcols + rcols, schema=pa.schema(lfields + rfields))


def join_tables(left: pa.Table, right: pa.Table, lkeys: list[int], rkeys: list[int], join_type: str) -> pa.Table:
    lb = oracle._concat(left.combine_chunks().to_batches(), left.schema)
    rb = oracle._concat(right.combine_chunks().to_batches(), right.schema)
    return pa.Table.from_batches([join_batches(lb, rb, lkeys, rkeys, join_type)])


def acero_join(left: pa.Table, right: pa.Table, lkeys: list[int], rkeys: list[int], join_type: str) -> pa.Table:
    """The same join by Arrow C++'s Acero hash join (NULL keys match nothing there too).  Row order is Acero's."""
    ln = [f"l{i}" for i in range(left.num_columns)]
    rn = [f"r{i}" for i in range(right.num_columns)]
    lt, rt = left.rename_columns(ln), right.rename_columns(rn)
    j = lt.join(rt, keys=[ln[k] for k in lkeys], right_keys=[rn[k] for k in rkeys], join_type=ACERO_TYPES[join_type],
                coalesce_keys=False, use_threads=False)
    names = ln if join_type in ("Semi", "Anti") else ln + rn
    out = j.select(names)
    return out.rename_columns(left.schema.names + ([] if join_type in ("Semi", "Anti") else right.schema.names))


# ---- plans ----------------------------------------------------------------------------------------------------------
def _static_schema(node: dict) -> pa.Schema:
    """Schema of a subtree that produced no batch at all (a Hash repartition of no rows)."""
    tag = node["execution_plan"]
    if tag == "memory_exec":
        sch = oracle._schema_from_json(node["schema"])
        return pa.schema([sch.field(n) for n in oracle.PlanExecutor._projected_names(node)], metadata=sch.metadata)
    if tag in ("repartition_exec", "coalesce_batches_exec", "coalesce_partitions_exec", "merge_exec", "filter_exec"):
        return _static_schema(node["input"])
    raise oracle.OracleError(f"oracle: cannot type the empty input {tag} of a join")


class TypedPlanExecutor(oracle.PlanExecutor):
    """oracle.PlanExecutor, with HashJoinExec of every join type."""

    def _exec(self, p: dict):
        if p["execution_plan"] != "hash_join_exec" or p.get("join_type", "Inner") == "Inner":
            return super()._exec(p)
        jt = p["join_type"]
        if jt not in JOIN_TYPES:
            raise oracle.OracleError(f"oracle: unknown join type {jt}")
        lparts, rparts = self._exec(p["left"]), self._exec(p["right"])
        if p.get("mode", "Partitioned") == "CollectLeft" or len(lparts) != len(rparts):
            # every right partition sees the whole left side: its unmatched left rows would depend on the partition count
            if jt in LEFT_PRESERVING and len(rparts) > 1:
                raise oracle.OracleError(f"oracle: CollectLeft {jt} join over {len(rparts)} right partitions is not restated")
            lparts = [[b for src in lparts for b in src]] * len(rparts)
        lschema = next((b.schema for src in lparts for b in src), None) or _static_schema(p["left"])
        rschema = next((b.schema for src in rparts for b in src), None) or _static_schema(p["right"])

        def on_idx(o, names):
            return names.index(o) if isinstance(o, str) else oracle._resolve(names, o)

        def run(pair):
            lsrc, rsrc = pair
            lb = oracle._concat([b for b in lsrc if b.num_rows], lschema)
            rb = oracle._concat([b for b in rsrc if b.num_rows], rschema)
            if lb.num_rows == 0 and rb.num_rows == 0:
                return []
            lk = [on_idx(l, lb.schema.names) for l, _ in p["on"]]
            rk = [on_idx(r, rb.schema.names) for _, r in p["on"]]
            return [join_batches(lb, rb, lk, rk, jt)]
        return self._map(run, list(zip(lparts, rparts)))


def execute_plan(plan, sources, threads: int = 1) -> pa.Table:
    """oracle.execute_plan with TypedPlanExecutor."""
    ex = TypedPlanExecutor(plan, threads)
    ex.feed_data_sources(sources)
    batches = [b for b in ex.execute()[0]]
    nonempty = [b for b in batches if b.num_rows]
    if nonempty:
        return pa.Table.from_batches(nonempty)
    return pa.Table.from_batches(batches[:1]) if batches else pa.table({})


# ---- the relations the join-type tests run over ---------------------------------------------------------------------
def _holes(values, every: int, phase: int = 0, type=None) -> pa.Array:
    """`values` with every `every`-th entry (from `phase`) NULL; every = 0: no NULL."""
    n = len(values)
    mask = np.zeros(n, bool) if not every else (np.arange(n) % every) == phase
    return pa.array(values, type=type, mask=mask)


def synthetic_cases(n_big: int = 6000, n_small: int = 700, seed: int = 11) -> dict:
    """name -> (left, right, left keys, right keys).  Every shape comes in both size orientations ("_sl": the left side is
    the smaller one, so it is hashed; "_sr": the right side is), so each join type runs both of its kernel forms."""
    rng = np.random.default_rng(seed)
    words = np.array(["ab", "cd", "efg", "", "hijkl", "m", "nopqrstu", "vw", "xyz", "0123456789abcdef"])
    out = {}

    def rel(n, key_range, key_nulls=0, payload_nulls=0, offset=0, utf8=False, two=False, phase=0):
        k = rng.integers(0, key_range, n) + offset
        cols = {}
        if utf8:
            cols["k"] = _holes([words[i % len(words)] + str(i // len(words)) for i in k], key_nulls, phase, pa.utf8())
        else:
            cols["k"] = _holes(k.astype(np.int64), key_nulls, phase, pa.int64())
        if two:
            cols["k2"] = _holes((k % 3).astype(np.int32), key_nulls and key_nulls + 1, phase, pa.int32())
        cols["v"] = _holes(rng.integers(-1000, 1000, n).astype(np.int32), payload_nulls, 1, pa.int32())
        cols["s"] = _holes([words[i] for i in rng.integers(0, len(words), n)], payload_nulls and payload_nulls + 2, 0, pa.utf8())
        cols["f"] = pa.array(rng.normal(0, 10, n).round(2))
        return pa.table(cols)

    shapes = {
        "i64_dups": dict(l=dict(key_range=400), r=dict(key_range=400)),
        "utf8_keys": dict(l=dict(key_range=300, utf8=True), r=dict(key_range=300, utf8=True)),
        "i64_null_keys_left": dict(l=dict(key_range=300, key_nulls=5, payload_nulls=7), r=dict(key_range=300)),
        "i64_null_keys_right": dict(l=dict(key_range=300), r=dict(key_range=300, key_nulls=4, payload_nulls=6)),
        "utf8_null_keys_both": dict(l=dict(key_range=250, utf8=True, key_nulls=6), r=dict(key_range=250, utf8=True, key_nulls=5, phase=2)),
        "no_matches": dict(l=dict(key_range=1000), r=dict(key_range=1000, offset=5000)),
        "all_match": dict(l=dict(key_range=50), r=dict(key_range=50)),
        "two_keys_i64_i32": dict(l=dict(key_range=200, two=True), r=dict(key_range=200, two=True)),
        "two_keys_null": dict(l=dict(key_range=200, two=True, key_nulls=9), r=dict(key_range=200, two=True, key_nulls=7)),
    }
    for name, sh in shapes.items():
        two = sh["l"].get("two", False)
        keys = [0, 1] if two else [0]
        for orient, (nl, nr) in (("_sl", (n_small, n_big)), ("_sr", (n_big, n_small))):
            out[name + orient] = (rel(nl, **sh["l"]), rel(nr, **sh["r"]), keys, keys)
    # Int32 + Int32 and Int32 + Utf8 keys (packed / row-comparison forms)
    for orient, (nl, nr) in (("_sl", (n_small, n_big)), ("_sr", (n_big, n_small))):
        def rel2(n, utf8):
            a = rng.integers(0, 40, n).astype(np.int32)
            b = rng.integers(0, 12, n)
            second = pa.array([words[i % len(words)] for i in b]) if utf8 else pa.array(b.astype(np.int32))
            return pa.table({"a": pa.array(a), "b": second, "v": pa.array(rng.integers(0, 99, n).astype(np.int64))})
        out["i32_i32" + orient] = (rel2(nl, False), rel2(nr, False), [0, 1], [0, 1])
        out["i32_utf8" + orient] = (rel2(nl, True), rel2(nr, True), [0, 1], [0, 1])
    base = rel(n_small, key_range=100)
    out["empty_left"] = (base.slice(0, 0), base, [0], [0])
    out["empty_right"] = (base, base.slice(0, 0), [0], [0])
    out["empty_both"] = (base.slice(0, 0), base.slice(0, 0), [0], [0])
    one = base.slice(3, 1)
    out["one_row_left"] = (one, base, [0], [0])
    out["one_row_right"] = (base, one, [0], [0])
    miss = pa.table({"k": pa.array([10 ** 9], pa.int64()), "v": pa.array([1], pa.int32()), "s": pa.array(["x"]), "f": pa.array([0.5])})
    out["one_row_no_match"] = (miss, base, [0], [0])
    return out


def nexmark_cases(events: dict) -> dict:
    """NEXMark persons vs auctions on p_id = seller, auctions vs bids on a_id = auction (both orders of the sides)."""
    t = {r: pa.Table.from_batches(events[r]).combine_chunks() for r in ("person", "auction", "bid")}
    person = t["person"].select(["p_id", "name", "city"])
    auction = t["auction"].select(["a_id", "seller", "category"])
    bid = t["bid"].select(["auction", "price"])
    return {"persons_auctions": (person, auction, [0], [1]), "auctions_persons": (auction, person, [1], [0]),
            "auctions_bids": (auction, bid, [0], [0]), "bids_auctions": (bid, auction, [0], [0])}


def canonical(t: pa.Table) -> pa.Table:
    """Rows in a canonical order (NULLs last), for comparing joins whose row order is unspecified."""
    t = t.combine_chunks()
    if t.num_rows == 0:
        return t
    tmp = pa.table({f"c{i}": t.column(i) for i in range(t.num_columns)})
    import pyarrow.compute as pc
    return t.take(pc.sort_indices(tmp, sort_keys=[(f"c{i}", "ascending") for i in range(t.num_columns)], null_placement="at_end"))


def assert_same_rows(actual: pa.Table, expected: pa.Table, ordered: bool) -> None:
    """Equal column types and rows: as multisets, or in order (Semi / Anti).  Names are not compared."""
    assert [f.type for f in actual.schema] == [f.type for f in expected.schema], (actual.schema, expected.schema)
    assert actual.num_rows == expected.num_rows, f"row counts differ: {actual.num_rows} vs {expected.num_rows}"
    a, e = (actual.combine_chunks(), expected.combine_chunks()) if ordered else (canonical(actual), canonical(expected))
    for i in range(a.num_columns):
        assert a.column(i).equals(e.column(i)), f"column {i} ({a.schema.names[i]}) differs"
