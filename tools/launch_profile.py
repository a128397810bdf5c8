"""Kernel launch profile (kernel label -> launches) of one execution of NEXMark q3, q5 and q8 at a fixed, seeded size.

Every operator labels its launches (LaunchTimer), so two builds that launch the same kernels the same number of times
print the same JSON.  tests/golden/launch_profile_q3_q5_q8.json holds the profile of the commit before the join types
other than Inner existed; tests/test_gpu_join_types.py checks that the Inner plans still launch exactly that.

    python tools/launch_profile.py [--root TREE] [--out FILE]

--root runs another checkout's build of the package (an A/B against an older commit).
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

# (query, relations fed, events): small enough to run in seconds, large enough for multi-tile scans in every kernel
WORKLOAD = (("q3", 1_000_000), ("q5", 2_000_000), ("q8", 2_000_000))


def profile(fb, nexgen, plans) -> dict:
    out = {}
    with fb.Context(0) as ctx:
        for q, events in WORKLOAD:
            if q == "q5":
                ev = {"bid": nexgen.bids_chunked(events, seed=42, columns=["auction"])}
            else:
                ev = nexgen.generate(events, seed=42, relations=("person", "auction"))
            tables = {r: ctx.import_batches(b) for r, b in ev.items()}
            ec = fb.ExecutionContext(ctx, plans.QUERIES[q]())
            feed = [tables[r] for r in plans.SOURCES[q]]
            ec.feed_tables(feed)
            ec.execute_device(0).num_rows          # warm-up: resident-CTA caches, allocator blocks
            ec.feed_tables(feed)
            ctx.profile_begin()
            ec.execute_device(0).num_rows
            prof = ctx.profile_end()
            out[q] = {k: int(v["launches"]) for k, v in sorted(prof.items())}
            ec.close()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=str(Path(__file__).resolve().parent.parent))
    ap.add_argument("--out")
    args = ap.parse_args()
    sys.path.insert(0, str(Path(args.root).resolve()))
    import flock_b200 as fb
    from flock_b200 import nexgen, plans
    res = profile(fb, nexgen, plans)
    text = json.dumps(res, indent=1, sort_keys=True)
    if args.out:
        Path(args.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
