"""Device time of HashJoinExec per join type at the q8 one-GPU share (the persons and auctions of 125 M NEXMark events:
2.5 M persons, 7.5 M auctions), one JSON line.

    python tools/join_types_bench.py [--reps 20] [--out FILE]

Per join: median and best of `reps` executions (CUDA events on the library stream around one hash_join call, L2 flushed
before each -- the protocol of bench.py's `queries`), kernel launches, output rows, algorithmic bytes (every input column
read once + every output column written once) and the CPU restatement's time for the same join (tests/join_oracle.py:
single-threaded C++ hash join + numpy, a restatement, NOT a tuned CPU baseline).  The card name and its power limit are
read in the same run and written beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import numpy as np  # noqa: E402
import pyarrow as pa  # noqa: E402

EVENTS = 125_000_000
# (label, join type, left relation, right relation, left key, right key)
JOINS = (
    ("persons_inner_auctions", "inner", "person", "auction", 0, 1),
    ("persons_left_auctions", "left", "person", "auction", 0, 1),      # preserved side (persons) is the smaller: hashed
    ("auctions_left_persons", "left", "auction", "person", 1, 0),      # preserved side (auctions) is the larger: streamed
    ("persons_full_auctions", "full", "person", "auction", 0, 1),
    ("persons_semi_auctions", "semi", "person", "auction", 0, 1),
    ("persons_anti_auctions", "anti", "person", "auction", 0, 1),
)


def card() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, power = (r.stdout.strip().split(", ") + ["?"])[:2] if r.returncode == 0 else ("unknown", "unknown")
    return {"gpu": name, "power_limit": power}


def relations() -> dict:
    from flock_b200 import nexgen
    n_p, n_a, _ = nexgen.relation_counts(EVENTS)
    def pieces(total, fn, cols):
        parts = [fn(min(4_000_000, total - o), 42, o, cols) for o in range(0, total, 4_000_000)]
        return pa.Table.from_batches(parts).combine_chunks()
    return {"person": pieces(n_p, nexgen.persons, ["p_id", "name"]), "auction": pieces(n_a, nexgen.auctions, ["a_id", "seller"])}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out")
    args = ap.parse_args()
    import flock_b200 as fb
    import join_oracle as jo
    rel = relations()
    res = {"workload": "q8 one-GPU share: persons and auctions of 125 M NEXMark events (seed 42)",
           "rows_in": {k: v.num_rows for k, v in rel.items()}, **card(), "joins": {}}
    with fb.Context(0) as ctx:
        dev = {k: ctx.import_batches(v.to_batches()) for k, v in rel.items()}
        for label, jt, lname, rname, lk, rk in JOINS:
            L, R = dev[lname], dev[rname]
            for _ in range(2):
                ctx.hash_join(L, R, [lk], [rk], jt).num_rows
            times = []
            for _ in range(args.reps):
                ctx.flush_l2()
                ctx.timer_start(2)
                out = ctx.hash_join(L, R, [lk], [rk], jt)
                ctx.timer_stop(2)
                rows = out.num_rows
                times.append(ctx.timer_ms(2))
                nbytes = out.nbytes
                del out
            l0 = ctx.kernel_launches
            ctx.hash_join(L, R, [lk], [rk], jt).num_rows
            launches = ctx.kernel_launches - l0
            lb, rb = jo.oracle._concat(rel[lname].to_batches(), rel[lname].schema), jo.oracle._concat(rel[rname].to_batches(), rel[rname].schema)
            t = time.perf_counter()
            li, _ = jo.join_indices(lb, rb, [lk], [rk], jt.capitalize())
            oracle_s = time.perf_counter() - t
            assert len(li) == rows, (label, len(li), rows)
            alg = rel[lname].nbytes + rel[rname].nbytes + nbytes
            res["joins"][label] = {"join_type": jt, "ms": round(statistics.median(times), 4), "ms_best": round(min(times), 4),
                                   "kernel_launches": launches, "rows_out": rows, "algorithmic_bytes": int(alg),
                                   "oracle_s": round(oracle_s, 3)}
    res["timing"] = (f"device-resident inputs, CUDA events around one hash_join call, L2 flushed before each of {args.reps} repetitions; "
                     "oracle_s: single-threaded CPU restatement (tests/join_oracle.py), not a tuned CPU baseline")
    line = json.dumps(res)
    if args.out:
        Path(args.out).write_text(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
