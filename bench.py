#!/usr/bin/env python
"""bench.py -- NEXMark events/sec through the B200-native executor (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's GPU path
    python bench.py --gpus 1 ... --dump-outputs DIR          # + the q2 result of the last timed step as DIR/<column>.npy
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores

N = 1  headline workload "nexmark_q2_10M_bids" = BASELINE.json configs[1]: NEXMark q2 (SELECT auction, price FROM bid
       WHERE auction % 123 = 0) over 10 M bids cut into 64 Ki-row Arrow batches; one step = one pass of the whole plan
       over all batches.  The same line carries a `queries` object with the other single-GPU configurations (q1 one
       batch, q3 10 M events, q5 100 M bids, q8 at the per-GPU share of the 1 B-event configuration), each timed
       device-resident with the L2 flushed between repetitions and each CHECKED against an independent numpy
       statement of the SQL (`parity_check`).
N > 1  headline workload "nexmark_q8_125M_events_per_gpu" = BASELINE.json configs[4] weak-scaled: every rank scans its
       own 125 M-event slice of the stream (2.5 M persons + 7.5 M auctions; 8 ranks = the 1 B-event configuration),
       the plan's Hash repartitions run as NVLink peer-window exchanges INSIDE the timed region, and the union of the
       ranks' results is compared (row count + order-independent 128-bit digest) with an independent reference
       computed from the rank-local generators.  `queries.q8` of the N = 1 line is the same share on one GPU, so the
       per-GPU work is identical at every N ("scaling": "weak").  q2 (round-robin sharding, no collective) stays in
       `queries`.

One JSON line on stdout (rank 0).  Keys beyond the base contract:
  value        events/s of the headline workload with the relations resident in HBM: K back-to-back executions of the
               plan through ExecutionContext::execute, CUDA events on the library's stream, max over ranks.
  e2e          the same metric through the reference-facing call sequence with HOST buffers every step:
               feed_data_sources -> execute -> export of the result to host Arrow memory -> clean_data_sources.
               The headline e2e feeds ORDINARY (pageable) Arrow buffers, as arrow-rs allocates them; `e2e.variants`
               adds the page-locked zero-copy feed and a cudaHostRegister-on-feed path (registration inside the timed
               region).  Byte counts come from the library (flockgpu_bytes_moved).
  roofline     dominant kernel of the headline workload: algorithmic bytes per launch / mean launch duration from
               per-launch CUDA events (flockgpu_profile_begin/_end) against the measured HBM copy bandwidth.  At N = 1
               the K steps run twice back to back: once bare (`value`, `ms_per_step`) and once with the event pairs
               (`roofline.kernel_ms`, `ms_per_step_instrumented`) -- the pairs cost ~3 us per 25 us step.
  cpu_baseline the CPU arm on the host cores in the same run (native threads inside liboracle.so, no Python per batch):
               all cores, target_partitions = 8 (flock/src/configs/flock.toml:113) and one thread.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np          # noqa: E402
import pyarrow as pa        # noqa: E402

N_BIDS = 10_000_000          # BASELINE.json configs[1]
EVENTS_PER_GPU = 125_000_000  # BASELINE.json configs[4] / 8
BATCH_ROWS = 65536
RING = 4                     # distinct resident relations rotated through (defeats the 126 MB L2)
UNIT = "events/s"
DUMP_BYTES = 64_000_000      # --dump-outputs: at most this many bytes of .npy data in all


# Libraries write to fd 1 behind Python's back (NCCL prints "NCCL version ..." there): keep the real stdout for the
# JSON line(s) only and point fd 1 at stderr for everything else.
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak_gbs() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def workload_config(world: int, bids: int) -> tuple[str, dict]:
    """(metric, config) -- identical in both arms (the driver compares the dicts)."""
    if world == 1:
        name = "nexmark_q2_10M_bids" if bids == N_BIDS else f"nexmark_q2_{bids}_bids"
        return "nexmark_q2_events_per_sec", {"workload": name, "query": "q2", "bids_per_gpu": bids, "batch_rows": BATCH_ROWS,
                                             "batches_per_step": (bids + BATCH_ROWS - 1) // BATCH_ROWS}
    from flock_b200 import nexgen
    n_p, n_a, _ = nexgen.relation_counts(EVENTS_PER_GPU)
    return "nexmark_q8_events_per_sec", {"workload": "nexmark_q8_125M_events_per_gpu", "query": "q8", "events_per_gpu": EVENTS_PER_GPU,
                                         "persons_per_gpu": n_p, "auctions_per_gpu": n_a, "batch_rows": BATCH_ROWS,
                                         "batches_per_step": (n_p + BATCH_ROWS - 1) // BATCH_ROWS + (n_a + BATCH_ROWS - 1) // BATCH_ROWS}


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons of one GPU through NVML while the timed regions run."""

    def __init__(self, device: int):
        super().__init__(daemon=True)
        self.device, self.samples, self.reasons, self.max_mhz = device, [], set(), None
        self._stop_evt = threading.Event()
        self.active = threading.Event()
        self.ok = False
        # seconds between samples: 2 ms while the short device-resident regions run (a K = 200 region lasts ~5 ms); the
        # host-buffer legs last 100+ ms and are sampled every 20 ms -- NVML queries take driver locks and the sampling
        # thread takes the interpreter lock, both of which the host side of an e2e step would otherwise wait for
        # (execute + export read 0.40 ms per step under 2 ms sampling against 0.07 ms without a sampler, run 37)
        self.interval = 0.002
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:      # NVML missing: report that honestly
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"} \
            if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else \
                {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self._stop_evt.is_set():
            if self.active.is_set():
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                    mask = get(self.h)
                    for bit, name in names.items():
                        if mask & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(self.interval)

    def stop(self) -> dict:
        self._stop_evt.set()
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable: " + getattr(self, "err", "")}
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


class Dist:
    """torch.distributed (NCCL) as the control plane: barriers, max/sum over ranks, the NCCL id broadcast."""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank, self.local, self.d = 0, 0, None
        if self.world > 1:
            import torch
            import torch.distributed as dist
            self.local = int(os.environ.get("LOCAL_RANK", "0"))
            torch.cuda.set_device(self.local)
            dist.init_process_group(backend="nccl", device_id=torch.device("cuda", self.local))
            self.d, self.rank = dist, dist.get_rank()

    def barrier(self):
        if self.d is not None:
            import torch
            self.d.barrier(device_ids=[self.local])
            torch.cuda.synchronize(self.local)

    def _reduce(self, values, op):
        if self.d is None:
            return list(values)
        import torch
        t = torch.tensor(list(values), dtype=torch.float64, device=torch.device("cuda", self.local))
        self.d.all_reduce(t, op=op)
        return t.tolist()

    def max(self, *values):
        return self._reduce(values, self.d.ReduceOp.MAX if self.d else None)

    def sum(self, *values):
        return self._reduce(values, self.d.ReduceOp.SUM if self.d else None)

    def sum_u64(self, values):
        """exact sum modulo 2^64 of unsigned words over the ranks (the digests): 16-bit limbs in int64 lanes"""
        if self.d is None:
            return [int(v) & (2**64 - 1) for v in values]
        import torch
        limbs = []
        for v in values:
            limbs += [(int(v) >> s) & 0xffff for s in (0, 16, 32, 48)]
        t = torch.tensor(limbs, dtype=torch.int64, device=torch.device("cuda", self.local))
        self.d.all_reduce(t, op=self.d.ReduceOp.SUM)
        lst, out = t.tolist(), []
        for i in range(len(values)):
            out.append(sum(lst[4 * i + k] << (16 * k) for k in range(4)) & (2**64 - 1))
        return out

    def gather_objects(self, obj):
        if self.d is None:
            return [obj]
        out = [None] * self.world
        self.d.all_gather_object(out, obj)
        return out

    def broadcast_object(self, obj):
        if self.d is None:
            return obj
        box = [obj]
        self.d.broadcast_object_list(box, src=0)
        return box[0]

    def close(self):
        if self.d is not None:
            self.d.destroy_process_group()


# ---- order-independent 128-bit digest of (p_id, name) rows (the multi-rank q8 check) --------------------------------
_M64 = (1 << 64) - 1


def _fmix64(k: np.ndarray) -> np.ndarray:
    k = k.astype(np.uint64, copy=True)
    with np.errstate(over="ignore"):
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xFF51AFD7ED558CCD)
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xC4CEB9FE1A85EC53)
        k ^= k >> np.uint64(33)
    return k


def digest_rows(p_id: np.ndarray, name: pa.Array) -> tuple[int, int, int]:
    """(rows, h1, h2): two independent 64-bit sums over per-row hashes of (p_id, name bytes).  A sum is order- and
    partition-independent, so the ranks' partial digests add up to the digest of the union."""
    n = len(p_id)
    if n == 0:
        return 0, 0, 0
    name = name.combine_chunks() if isinstance(name, pa.ChunkedArray) else name
    off = np.frombuffer(name.buffers()[1], dtype=np.int32, count=n + 1 + name.offset)[name.offset:]
    data = np.frombuffer(name.buffers()[2], dtype=np.uint8) if name.buffers()[2] is not None else np.zeros(0, np.uint8)
    lens = np.diff(off).astype(np.int64)
    total = int(lens.sum())
    body = data[int(off[0]):int(off[0]) + total].astype(np.uint64)
    starts = np.cumsum(lens) - lens
    pos = np.arange(total, dtype=np.int64) - np.repeat(starts, lens)
    out = []
    with np.errstate(over="ignore"):
        for mult, seed in ((np.uint64(0x100000001B3), np.uint64(0x9E3779B97F4A7C15)), (np.uint64(0xD6E8FEB86659FD93), np.uint64(0xC2B2AE3D27D4EB4F))):
            table = np.ones(int(lens.max()) + 1, np.uint64)
            for i in range(1, table.size):
                table[i] = table[i - 1] * mult
            contrib = (body + np.uint64(1)) * table[pos]
            sh = np.zeros(n, np.uint64)
            nz = lens > 0
            if total:
                sh[nz] = np.add.reduceat(contrib, starts[nz])
            row = _fmix64(_fmix64(p_id.astype(np.int64).view(np.uint64) ^ seed) + sh * np.uint64(0x9FB21C651E98DF25) + lens.astype(np.uint64))
            out.append(int(row.sum(dtype=np.uint64)))
    return n, out[0], out[1]


# ---- inputs ------------------------------------------------------------------------------------------------------
def q8_slice(rank: int, seed: int = 42):
    """The persons and auctions of rank `rank`'s contiguous 125 M-event slice of the stream, as 64 Ki-row batches."""
    from flock_b200 import nexgen
    n_p, n_a, _ = nexgen.relation_counts(EVENTS_PER_GPU)
    def pieces(total, first, fn, cols):
        parts = [fn(min(4_000_000, total - o), seed, first + o, cols) for o in range(0, total, 4_000_000)]
        tbl = pa.Table.from_batches(parts).combine_chunks()
        return nexgen.split_batches(tbl.to_batches()[0], BATCH_ROWS)
    return pieces(n_p, rank * n_p, nexgen.persons, ["p_id", "name"]), pieces(n_a, rank * n_a, nexgen.auctions, ["seller"])


def time_plan(ctx, ec, tables, reps: int, dist: Dist | None = None, flush: bool = True):
    """Median / best device time of one execution of plan 0 with `tables` fed (CUDA events on the library stream; L2
    flushed before every repetition; max over ranks when distributed) + the per-kernel profile of one more run."""
    def run():
        ec.feed_tables(tables)
        return ec.execute_device(0)
    out = run()
    rows = out.num_rows
    for _ in range(2):
        run().num_rows
    times = []
    for _ in range(reps):
        if flush:
            ctx.flush_l2()
        if dist is not None:
            dist.barrier()
        ctx.timer_start(2)
        o = run()
        ctx.timer_stop(2)
        o.num_rows
        ms = ctx.timer_ms(2)
        times.append(dist.max(ms)[0] if dist is not None else ms)
    if dist is not None:
        dist.barrier()
    ctx.profile_begin()
    launches0 = ctx.kernel_launches
    run().num_rows
    launches = ctx.kernel_launches - launches0
    prof = ctx.profile_end()
    return out, rows, statistics.median(times), min(times), prof, launches


def dump_outputs(table: pa.Table, out_dir: str) -> None:
    """Writes every column of `table` as out_dir/<column>.npy in float64 (exact for the int32 columns of q2), so that two
    builds can be compared array for array.  Beyond DUMP_BYTES in all, the same fixed, seeded sample of rows (in row
    order) is taken from every column."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    n, cap = table.num_rows, DUMP_BYTES // (8 * max(table.num_columns, 1))
    rows = np.sort(np.random.default_rng(0).choice(n, cap, replace=False)) if n > cap else None
    for name in table.column_names:
        v = table[name].to_numpy().astype(np.float64)
        np.save(d / f"{name}.npy", v if rows is None else v[rows])
    log(f"dumped {table.column_names} of the last timed step ({n} rows{'' if rows is None else f', {cap} sampled'}) to {d}")


def dominant(prof: dict) -> tuple[str | None, float]:
    if not prof:
        return None, 0.0
    k = max(prof, key=lambda n: prof[n]["ms"])
    return k, prof[k]["ms"]


# ---- the single-GPU side queries (N = 1) ---------------------------------------------------------------------------
def side_queries(ctx, fb, reps: int, peak: float, parity: dict) -> dict:
    from flock_b200 import nexgen, plans
    res = {}

    def record(q, events, rows_in, alg_bytes, ms, best, prof, launches, rows_out, extra=None):
        k, k_ms = dominant(prof)
        res[q] = {"ms": round(ms, 5), "ms_best": round(best, 5), "events_per_sec": events / (ms * 1e-3), "rows_in": rows_in, "rows_out": rows_out,
                  "algorithmic_bytes": int(alg_bytes), "roofline": {"bound": "hbm", "achieved": round(alg_bytes / (ms * 1e-3) / 1e9, 1), "peak": peak,
                                                                   "unit": "GB/s", "frac": round(alg_bytes / (ms * 1e-3) / 1e9 / peak, 4)},
                  "dominant_kernel": k, "dominant_kernel_ms": round(k_ms, 5), "kernel_launches": launches, "kernels": prof,
                  "timing": "device-resident inputs, CUDA events around one plan execution, L2 flushed (384 MB memset) before each of "
                            f"{reps} repetitions, median"}
        if extra:
            res[q].update(extra)

    # ---- q1: one 64 Ki-row bid batch (configs[0])
    b1 = nexgen.bids(BATCH_ROWS, seed=42)
    t1 = ctx.import_batches([b1])
    ec = fb.ExecutionContext(ctx, plans.q1())
    out, rows, ms, best, prof, launches = time_plan(ctx, ec, [t1], reps)
    got = out.to_arrow()
    ok = (got.num_rows == BATCH_ROWS and np.array_equal(got["price"].to_numpy(), 0.908 * b1["price"].to_numpy().astype(np.float64))
          and got["auction"].equals(pa.chunked_array([b1["auction"]])) and got["b_date_time"].equals(pa.chunked_array([b1["b_date_time"]])))
    parity["q1"] = "ok" if ok else "MISMATCH"
    record("q1", BATCH_ROWS, {"bid": BATCH_ROWS}, 12.0 * BATCH_ROWS, ms, best, prof, launches, rows)
    ec.close()
    del t1, out

    # ---- q3: 10 M events = 200 K persons + 600 K auctions (configs[2])
    ev = nexgen.generate(10_000_000, seed=42, relations=("person", "auction"),
                         columns={"person": ["p_id", "name", "city", "state"], "auction": ["a_id", "seller", "category"]})
    src = {r: ctx.import_batches(ev[r]) for r in ("auction", "person")}
    ec = fb.ExecutionContext(ctx, plans.q3())
    out, rows, ms, best, prof, launches = time_plan(ctx, ec, [src[r] for r in plans.SOURCES["q3"]], reps)
    got = out.to_arrow()
    a, p = pa.Table.from_batches(ev["auction"]), pa.Table.from_batches(ev["person"])
    pid = p["p_id"].to_numpy()
    okst = np.isin(np.array(p["state"].to_pylist()), ["or", "id", "ca"])
    sel = a["category"].to_numpy() == 10
    sellers, a_ids = a["seller"].to_numpy()[sel], a["a_id"].to_numpy()[sel]
    pos = np.minimum(np.searchsorted(pid, sellers), pid.size - 1)
    hit = (pid[pos] == sellers) & okst[pos]
    order = np.argsort(got["a_id"].to_numpy(), kind="stable")
    ok = (got.num_rows == int(hit.sum()) and np.array_equal(got["a_id"].to_numpy()[order], np.sort(a_ids[hit]))
          and got["name"].take(pa.array(order)).to_pylist() == p["name"].take(pa.array(pos[hit][np.argsort(a_ids[hit], kind="stable")])).to_pylist())
    parity["q3"] = "ok" if ok else "MISMATCH"
    n_p, n_a = p.num_rows, a.num_rows
    utf8 = sum(p[c].nbytes for c in ("name", "city", "state"))
    out_utf8 = sum(got[c].nbytes for c in ("name", "city", "state"))
    record("q3", 10_000_000, {"person": n_p, "auction": n_a}, 12.0 * n_a + 4.0 * n_p + utf8 + 4.0 * rows + out_utf8, ms, best, prof, launches, rows,
           {"note": "events/s counts all 10 M events of the stream; the plan scans their 800 K persons + auctions"})
    ec.close()
    del src, out, ev

    # ---- q5: 100 M bids (configs[3])
    t0 = time.time()
    batches = nexgen.bids_chunked(100_000_000, seed=42, columns=["auction"])
    auction = np.concatenate([b["auction"].to_numpy() for b in batches])
    bids = ctx.import_batches(batches)
    del batches
    log(f"q5 input generated + uploaded in {time.time() - t0:.1f}s")
    ec = fb.ExecutionContext(ctx, plans.q5())
    out, rows, ms, best, prof, launches = time_plan(ctx, ec, [bids, bids], reps)
    got = out.to_arrow()
    counts = np.bincount(auction)
    winners = np.nonzero(counts == counts.max())[0]
    ok = sorted(got["auction"].to_pylist()) == winners.tolist() and set(got["num"].to_pylist()) == {int(counts.max())}
    parity["q5"] = "ok" if ok else "MISMATCH"
    groups = int((counts > 0).sum())
    record("q5", 100_000_000, {"bid": 100_000_000}, 4.0 * 100_000_000 + 12.0 * groups, ms, best, prof, launches, rows, {"groups": groups})
    ec.close()
    del bids, out, auction, counts

    # ---- q8: the per-GPU share of the 1 B-event configuration (configs[4] / 8)
    persons, auctions = q8_slice(0)
    src = {"person": ctx.import_batches(persons), "auction": ctx.import_batches(auctions)}
    ec = fb.ExecutionContext(ctx, plans.q8())
    out, rows, ms, best, prof, launches = time_plan(ctx, ec, [src[r] for r in plans.SOURCES["q8"]], reps)
    got = out.to_arrow()
    p = pa.Table.from_batches(persons)
    sellers = np.unique(np.concatenate([b["seller"].to_numpy() for b in auctions]))
    keep = np.isin(p["p_id"].to_numpy(), sellers)
    want = digest_rows(p["p_id"].to_numpy()[keep], p["name"].filter(pa.array(keep)))
    have = digest_rows(got["p_id"].to_numpy(), got["name"])
    parity["q8"] = "ok" if want == have else f"MISMATCH rows {have[0]} vs {want[0]}"
    n_p, n_a = p.num_rows, sum(b.num_rows for b in auctions)
    record("q8", EVENTS_PER_GPU, {"person": n_p, "auction": n_a}, 4.0 * n_p + p["name"].nbytes + 4.0 * n_a + 4.0 * rows + got["name"].nbytes, ms, best, prof,
           launches, rows, {"note": "125 M events = the per-GPU share of the 1 B-event configuration; the N > 1 lines time the same share per rank with the exchange"})
    ec.close()
    return res


# ---- N = 1: q2 headline ----------------------------------------------------------------------------------------------
def run_gpu_q2(args, dist: Dist) -> dict:
    import flock_b200 as fb
    from flock_b200 import nexgen, plans

    rank, world, local = dist.rank, dist.world, dist.local
    ctx = fb.Context(local)
    sampler = ClockSampler(local)
    sampler.start()
    metric, config = workload_config(1, args.bids)
    parity = {}

    t0 = time.time()
    relations = [nexgen.bids_chunked(args.bids, seed=42 + 1000 * rank + r, columns=None if r == 0 else ["auction", "price"]) for r in range(RING)]
    n_batches = len(relations[0])
    resident = [ctx.import_batches(rel) for rel in relations]
    pageable = relations[0]                                          # ordinary Arrow buffers, as arrow-rs allocates them
    pinned = [ctx.pinned_copy(b) for b in relations[0]]              # the same batches in page-locked host memory
    log(f"[rank {rank}] generated + uploaded {RING} x {args.bids} bids in {time.time() - t0:.1f}s ({n_batches} batches of <= {BATCH_ROWS} rows)")
    ec = fb.ExecutionContext(ctx, plans.q2())

    def step_device(i: int):
        ec.feed_tables([resident[i % RING]])
        return ec.execute_device(0)         # one filter_compact_kernel launch; the survivor count stays in flight

    n_sel = [step_device(r).num_rows for r in range(RING)]
    # parity of the headline workload: exact arrays against numpy's truncated remainder
    got = step_device(0).to_arrow()
    au = np.concatenate([b["auction"].to_numpy() for b in relations[0]])
    pr = np.concatenate([b["price"].to_numpy() for b in relations[0]])
    keep = np.fmod(au.astype(np.int64), 123) == 0
    parity["q2"] = "ok" if (np.array_equal(got["auction"].to_numpy(), au[keep]) and np.array_equal(got["price"].to_numpy(), pr[keep])) else "MISMATCH"
    del got, au, pr, keep

    keep = []
    for i in range(args.warmup):
        keep = (keep + [step_device(i)])[-2:]
    ctx.synchronize()
    dist.barrier()
    # ---- timed region A: the K steps, nothing between the launches but the library's own work -> `value`
    launches0 = ctx.kernel_launches
    sampler.active.set()
    ctx.timer_start(0)
    t_host = time.perf_counter()
    for i in range(args.steps):
        keep = (keep + [step_device(args.warmup + i)])[-2:]
    host_us = (time.perf_counter() - t_host) * 1e6 / args.steps
    ctx.timer_stop(0)
    ctx.synchronize()
    dist.barrier()
    dev_ms = ctx.timer_ms(0)
    launches = ctx.kernel_launches - launches0
    assert keep[-1].num_rows == n_sel[(args.warmup + args.steps - 1) % RING]
    last_step = keep[-1] if args.dump_outputs else None     # the result of the last step of `value`'s region
    # ---- timed region B: the same K steps again with a CUDA-event pair around every launch (flockgpu_profile_*) -> the
    # kernel's mean duration for `roofline`.  Kept apart from A because the event pairs themselves cost ~3 us per step
    # (27.8 vs 24.4 us per step, runs 28 / 32); `ms_per_step_instrumented` reports B next to A.
    dist.barrier()
    ctx.profile_begin()
    ctx.timer_start(0)
    for i in range(args.steps):
        keep = (keep + [step_device(args.warmup + args.steps + i)])[-2:]
    ctx.timer_stop(0)
    ctx.synchronize()
    dist.barrier()
    sampler.active.clear()
    dev_ms_instrumented = dist.max(ctx.timer_ms(0))[0]
    prof = ctx.profile_end()
    del keep
    dev_ms = dist.max(dev_ms)[0]

    # ---- e2e legs: host batches -> plan -> host result, every step
    def e2e_leg(source_batches, zero_copy: bool, register: bool, steps: int) -> dict:
        src = [fb.HostRelation(source_batches)]
        ctx.set_option("feed_zero_copy", 1 if zero_copy else 0)
        ctx.set_option("feed_register", 1 if register else 0)
        for _ in range(2):
            ec.feed_data_sources(src)
            ec.execute()
            ec.clean_data_sources()
        dist.barrier()
        h0, d0 = ctx.bytes_moved()
        sampler.interval = 0.02
        sampler.active.set()
        ctx.timer_start(1)
        t_wall = time.perf_counter()
        t_feed = t_exec = t_clean = 0.0
        for _ in range(steps):
            a = time.perf_counter()
            ec.feed_data_sources(src)
            b = time.perf_counter()
            res = ec.execute()
            c = time.perf_counter()
            ec.clean_data_sources()
            d = time.perf_counter()
            t_feed += b - a
            t_exec += c - b
            t_clean += d - c
        ctx.timer_stop(1)
        ctx.synchronize()
        ms = max(ctx.timer_ms(1), (time.perf_counter() - t_wall) * 1e3)      # host-side work counts too
        sampler.active.clear()
        h1, d1 = ctx.bytes_moved()
        ms = dist.max(ms)[0]
        assert res[0][0].num_rows == n_sel[0]
        ctx.set_option("feed_zero_copy", 0)
        ctx.set_option("feed_register", 0)
        src[0].release()
        return {"value": world * args.bids * steps / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": (h1 - h0) // steps, "d2h_bytes_per_step": (d1 - d0) // steps,
                "steps": steps, "ms_per_step": ms / steps,
                "host_ms_per_step": {"feed_data_sources": round(t_feed * 1e3 / steps, 4), "execute+export": round(t_exec * 1e3 / steps, 4),
                                     "clean_data_sources": round(t_clean * 1e3 / steps, 4)}}

    e2e_steps = args.steps if args.e2e_steps is None else args.e2e_steps
    e2e_pageable = e2e_leg(pageable, False, False, max(3, min(e2e_steps, 40)))
    e2e_pageable["feed"] = "pageable Arrow buffers (as arrow-rs allocates them): staged through the library's page-locked ring by host threads, then DMA"
    e2e_registered = e2e_leg(pageable, True, True, max(3, min(e2e_steps, 10)))
    e2e_registered["feed"] = "pageable Arrow buffers page-locked in place by cudaHostRegister at feed time and released at clean time (both inside the timed region), read in place over PCIe"
    e2e_pinned = e2e_leg(pinned, True, False, e2e_steps)
    e2e_pinned["feed"] = ("batches allocated page-locked (flockgpu_host_alloc, the allocator hook of rust/flock-gpu-exec): the filter reads `auction` in place "
                          "over PCIe and fetches `price` for survivors only")
    e2e = dict(e2e_pageable)
    e2e["variants"] = {"pageable": e2e_pageable, "host_register": e2e_registered, "page_locked_zero_copy": e2e_pinned}
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(last_step.to_arrow(), args.dump_outputs)
    del last_step

    # ---- roofline of the dominant kernel
    peak, peak_src = measured_peak_gbs()
    k = next((v for name, v in prof.items() if name.startswith("filter_compact")), None)
    mean_sel = float(np.mean(n_sel)) if n_sel else 0.0
    alg_bytes = 4.0 * args.bids + 12.0 * mean_sel          # SURVEY.md 8(d): read auction 4 B x N; per survivor read price 4 B, write 8 B
    roofline, traffic, tsrc = None, None, None
    for name in ("r2_filter_dram_traffic.json", "r1_filter_dram_traffic.json"):
        tp = ROOT / "profiles" / name                        # dram__bytes_{read,write}.sum of one ncu --set full capture of this kernel
        if tp.exists() and args.bids == N_BIDS:
            try:
                tj = json.loads(tp.read_text())
                traffic, tsrc = int(tj["dram_bytes_read_per_launch"]) + int(tj["dram_bytes_write_per_launch"]), f"profiles/{name} (ncu --set full, one launch)"
                break
            except Exception:
                pass
    if k and k["launches"]:
        # Two CUDA-event measurements of the kernel's average launch duration, both on the launching stream:
        #   back to back  region A / K: the region holds exactly K launches of this kernel and nothing else (one launch per
        #                 step, `gpu_launches` == `steps`), so its length / K bounds a launch from above, gaps included;
        #   event pairs   region B: an event pair around every launch -- what an isolated launch costs; the pairs
        #                 serialise the launches and read ~2.5 us longer (25.1 vs 22.6 us, run 34; ncu's cold, serialised
        #                 launch: 24.3 us).
        # `achieved` / `frac` use the back-to-back figure (the sustained rate the workload actually runs at, the same
        # measurement as `value`); the event-pair figure stays beside it.
        k_pairs_ms = k["ms"] / k["launches"]
        one_per_step = launches == args.steps
        k_ms = min(k_pairs_ms, dev_ms / args.steps) if one_per_step else k_pairs_ms
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        pairs = alg_bytes / (k_pairs_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                    "traffic": traffic, "traffic_source": tsrc, "kernel": "filter_compact_kernel", "kernel_ms": round(k_ms, 5),
                    "kernel_ms_source": "timed region / launches (back to back)" if k_ms < k_pairs_ms else "event pair around every launch",
                    "event_pairs": {"kernel_ms": round(k_pairs_ms, 5), "achieved": round(pairs, 1), "frac": round(pairs / peak, 4)},
                    "launches_timed": k["launches"], "algorithmic_bytes_per_launch": int(alg_bytes), "peak_source": peak_src}

    result = {
        "metric": metric, "value": world * args.bids * args.steps / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config,
        "notes": {"sharding": "one GPU", "cache": f"inputs rotate over {RING} resident relations ({RING} x {8 * args.bids / 1e6:.0f} MB > 126 MB L2)",
                  "selectivity": mean_sel / args.bids},
        "e2e": e2e, "gpu_launches": int(launches), "host_enqueue_us_per_step": round(host_us, 2),
        "ms_per_step_instrumented": dev_ms_instrumented / args.steps, "kernels": prof, "clocks": clocks, "roofline": roofline,
        "stream_events_per_sec": world * args.bids * (50 / 46) * args.steps / (dev_ms * 1e-3),
    }
    ec.close()
    del resident, pinned, relations
    if not args.no_queries:
        try:
            result["queries"] = side_queries(ctx, fb, max(5, min(args.steps, 20)), peak, parity)
        except Exception as e:                      # the headline numbers above must still be reported
            log(f"side queries failed: {e!r}")
            result["queries"] = {"error": repr(e)[:400]}
    result["parity_check"] = parity
    if not args.no_cpu_baseline:
        try:
            result["cpu_baseline"] = cpu_baseline(args, 1)
        except Exception as e:
            log(f"cpu_baseline failed: {e}")
            result["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port", "sample": f"failed: {e}"[:300]}
    ctx.close()
    return result


# ---- N > 1: q8 sharded over the ranks, the exchange in the timed region --------------------------------------------------
PHASES = {"scan+aggregate": ("agg_",), "partition+push (exchange)": ("partition_", "exchange_"), "join build/probe": ("join_",), "take (gather)": ("gather_",),
          "filter/project": ("filter_", "project_")}


def phase_times(prof: dict) -> dict:
    out = {}
    for name, v in prof.items():
        ph = next((p for p, pre in PHASES.items() if name.startswith(pre)), "other")
        out[ph] = round(out.get(ph, 0.0) + v["ms"], 5)
    return out


def bind_to_gpu_numa_node(device: int, dist: "Dist | None" = None) -> str:
    """Pins this process to CPU cores next to its GPU (NVML's ideal affinity: `nvidia-smi topo -m` shows GPUs 0-3 on NUMA
    node 0 and 4-7 on node 1 on these boxes); torchrun does not bind ranks.  With `dist`, the ranks that share a node
    split its cores into disjoint, contiguous slices (physical cores and their hyper-thread siblings together), so that
    no two ranks' host threads ever share a core -- what `numactl --physcpubind` would do per rank.  FLOCK_BENCH_BIND=node
    keeps the whole node, =off leaves the process unbound."""
    mode = os.environ.get("FLOCK_BENCH_BIND", "slice")
    if mode == "off":
        return "unbound (FLOCK_BENCH_BIND=off)"
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(device))
        node = sorted(os.sched_getaffinity(0))
        if dist is None or dist.world == 1 or mode == "node":
            return f"{len(node)} cpus (node)"
        masks = dist.gather_objects(tuple(node))
        same = [r for r in range(dist.world) if masks[r] == masks[dist.rank]]
        j, k = same.index(dist.rank), len(same)
        half = len(node) // 2                         # "0-31,64-95": first half physical cores, second half their siblings
        per = max(1, half // k)
        mine = node[j * per:(j + 1) * per] + node[half + j * per:half + (j + 1) * per]
        if mine:
            os.sched_setaffinity(0, mine)
        return f"{len(mine)} cpus (slice {j + 1} of {k} of a {len(node)}-cpu node)"
    except Exception as e:                           # affinity is a tuning aid, never a requirement
        return f"unbound ({type(e).__name__})"


def run_gpu_q8(args, dist: Dist) -> dict | None:
    import flock_b200 as fb
    from flock_b200 import nexgen, plans

    rank, world, local = dist.rank, dist.world, dist.local
    numa = bind_to_gpu_numa_node(local, dist)
    ctx = fb.Context(local)
    ctx.comm_init(dist.broadcast_object(fb.Context.comm_unique_id() if rank == 0 else None), rank, world)
    alone = fb.Context(local)                       # the same share WITHOUT a communicator: what one GPU does on its own
    sampler = ClockSampler(local)
    sampler.interval = float(os.environ.get("FLOCK_BENCH_SAMPLE_MS", "2")) * 1e-3
    sampler.start()
    metric, config = workload_config(world, args.bids)
    peak, peak_src = measured_peak_gbs()
    parity = {}

    t0 = time.time()
    persons, auctions = q8_slice(rank)
    host = {"person": persons, "auction": auctions}
    order = plans.SOURCES["q8"]
    resident = {k: ctx.import_batches(v) for k, v in host.items()}
    resident_alone = {k: alone.import_batches(v) for k, v in host.items()}
    log(f"[rank {rank}] generated + uploaded {sum(b.num_rows for b in persons)} persons + {sum(b.num_rows for b in auctions)} auctions in {time.time() - t0:.1f}s")
    ec = fb.ExecutionContext(ctx, plans.q8())
    ec_alone = fb.ExecutionContext(alone, plans.q8())

    def step():
        ec.feed_tables([resident[r] for r in order])
        return ec.execute_device(0)

    # ---- parity: union of the ranks' results against an independent reference built from the rank-local generators
    dist.barrier()
    out = step()
    got = out.to_arrow()
    my_sellers = np.unique(np.concatenate([b["seller"].to_numpy() for b in auctions]))
    sellers = np.unique(np.concatenate(dist.gather_objects(my_sellers)))
    p = pa.Table.from_batches(persons)
    keepm = np.isin(p["p_id"].to_numpy(), sellers)
    want = digest_rows(p["p_id"].to_numpy()[keepm], p["name"].filter(pa.array(keepm)))
    have = digest_rows(got["p_id"].to_numpy(), got["name"])
    tot = dist.sum_u64([want[0], want[1], want[2], have[0], have[1], have[2]])
    parity["q8"] = "ok" if tot[:3] == tot[3:] else f"MISMATCH rows {tot[3]} vs {tot[0]}"
    parity["q8_detail"] = {"rows_union": tot[3], "rows_expected": tot[0], "digest_union": f"{tot[4]:016x}{tot[5]:016x}", "digest_expected": f"{tot[1]:016x}{tot[2]:016x}",
                           "method": "sum over ranks of per-row 2 x 64-bit hashes of (p_id, name); expected side = numpy isin() of each rank's persons against the all-gathered sellers"}
    rows_out = tot[3]
    del out, got

    # ---- device leg: W warm-up steps, then EXACTLY K timed steps between barriers (inputs: 80 MB per rank; the L2 is
    # flushed before every step, outside nothing -- the flush memset is part of the region and costs ~60 us; see notes)
    keep = []
    for _ in range(args.warmup):
        keep = (keep + [step()])[-2:]
    ctx.synchronize()
    dist.barrier()
    launches0 = ctx.kernel_launches
    sampler.active.set()
    ctx.timer_start(0)
    for _ in range(args.steps):
        keep = (keep + [step()])[-2:]
    ctx.timer_stop(0)
    ctx.synchronize()
    dist.barrier()
    sampler.active.clear()
    dev_ms = dist.max(ctx.timer_ms(0))[0]
    launches = ctx.kernel_launches - launches0
    del keep
    # per-phase kernel times of one more step (max over ranks per phase)
    # (five steps, per-step mean: the ranks leave the barrier tens of microseconds apart, and a single profiled step
    # books that skew as waiting time inside the first exchange -- run 23 showed 150 us on rank 0 against 27 us on rank 1)
    PROFILED_STEPS = 5
    dist.barrier()
    ctx.profile_begin()
    for _ in range(PROFILED_STEPS):
        step().num_rows
    prof = {k: {"launches": v["launches"] / PROFILED_STEPS, "ms": v["ms"] / PROFILED_STEPS} for k, v in ctx.profile_end().items()}
    ph = phase_times(prof)
    names = sorted(PHASES) + ["other"]
    mx = dist.max(*[ph.get(n, 0.0) for n in names])
    phases = {n: round(v, 5) for n, v in zip(names, mx) if v}
    # how long each rank sat in the exchange waiting for its peers' counts (exchange_place_kernel = push my counts,
    # wait for everybody's, lay the windows out) and its own step time: rank skew shows up here, not in the kernels
    per_rank = dist.gather_objects({"rank": dist.rank, "step_ms": round(ctx.timer_ms(0) / args.steps, 5),
                                    "exchange_place_ms": round(prof.get("exchange_place_kernel", {}).get("ms", 0.0), 5),
                                    "exchange_finish_ms": round(prof.get("exchange_finish_kernel", {}).get("ms", 0.0), 5),
                                    "kernels_us": {k: round(v["ms"] * 1e3, 1) for k, v in prof.items()}})

    # ---- the same share on one GPU, no communicator (what weak scaling is measured against), same protocol
    def step_alone():
        ec_alone.feed_tables([resident_alone[r] for r in order])
        return ec_alone.execute_device(0)
    for _ in range(args.warmup):
        step_alone().num_rows
    alone.synchronize()
    dist.barrier()
    alone.timer_start(0)
    for _ in range(args.steps):
        step_alone().num_rows
    alone.timer_stop(0)
    alone.synchronize()
    alone_ms = dist.max(alone.timer_ms(0))[0]

    # ---- e2e: host batches every step (pageable Arrow buffers), result exported to the host
    src = [[host[r]] for r in order]
    for _ in range(2):
        dist.barrier()
        ec.feed_data_sources(src)
        ec.execute()
        ec.clean_data_sources()
    e2e_steps = max(3, min(args.steps if args.e2e_steps is None else args.e2e_steps, 20))
    dist.barrier()
    h0, d0 = ctx.bytes_moved()
    sampler.interval = 0.02
    sampler.active.set()
    t_wall = time.perf_counter()
    for _ in range(e2e_steps):
        ec.feed_data_sources(src)
        ec.execute()
        ec.clean_data_sources()
    ctx.synchronize()
    e2e_ms = dist.max((time.perf_counter() - t_wall) * 1e3)[0]
    sampler.active.clear()
    h1, d1 = ctx.bytes_moved()
    clocks = sampler.stop()

    events = world * EVENTS_PER_GPU
    n_p, n_a = sum(b.num_rows for b in persons), sum(b.num_rows for b in auctions)
    alg = dist.sum(4.0 * n_p + p["name"].nbytes + 4.0 * n_a)[0]
    k, k_ms = dominant(prof)
    # ---- q2 weak-scaled next to it (round-robin sharding, no collective)
    q2 = None
    if not args.no_queries:
        # the protocol of the N = 1 headline: K back-to-back executions over RING distinct resident relations (> L2),
        # CUDA events on the library stream, barrier + sync on both sides, max over ranks
        ring = [alone.import_batches(nexgen.bids_chunked(args.bids, seed=42 + 1000 * rank + r, columns=["auction", "price"])) for r in range(RING)]
        ec2 = fb.ExecutionContext(alone, plans.q2())

        def q2_step(i: int):
            ec2.feed_tables([ring[i % RING]])
            return ec2.execute_device(0)
        keep2 = []
        for i in range(max(args.warmup, 3)):
            keep2 = (keep2 + [q2_step(i)])[-2:]
        alone.synchronize()
        dist.barrier()
        alone.timer_start(0)
        for i in range(args.steps):
            keep2 = (keep2 + [q2_step(i)])[-2:]
        alone.timer_stop(0)
        alone.synchronize()
        dist.barrier()
        keep2[-1].num_rows
        ms2 = dist.max(alone.timer_ms(0))[0] / args.steps
        q2 = {"ms": round(ms2, 5), "events_per_sec": world * args.bids / (ms2 * 1e-3), "bids_per_gpu": args.bids, "sharding": "round-robin, no collective",
              "timing": f"{args.steps} back-to-back executions per rank over {RING} resident relations, max over ranks (the N = 1 headline's protocol)"}
        del keep2, ring
        ec2.close()
    result = {
        "metric": metric, "value": events * args.steps / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32+utf8", "data": "synthetic",
        "config": config,
        "notes": {"sharding": f"every rank scans its own contiguous 125 M-event slice; Hash repartitions = NVLink peer-window exchanges ({world} ranks)",
                  "cache": "per-rank inputs (~80 MB) stay resident between steps; intermediate tables (~150 MB per step) exceed nothing: see queries.q8 of the N = 1 line for the L2-flushed figure",
                  "single_share_ms_per_step": alone_ms / args.steps, "rows_out": rows_out},
        "e2e": {"value": events * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": (h1 - h0) // e2e_steps, "d2h_bytes_per_step": (d1 - d0) // e2e_steps,
                "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps, "feed": "pageable Arrow batches per rank, result exported per rank"},
        "gpu_launches": int(launches), "launches_per_step_rank0": launches / args.steps, "kernels": prof, "phases_ms": phases, "per_rank": per_rank, "cpu_affinity": numa, "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": round(alg / (dev_ms / args.steps * 1e-3) / 1e9, 1), "peak": peak * world, "unit": "GB/s",
                     "frac": round(alg / (dev_ms / args.steps * 1e-3) / 1e9 / (peak * world), 4), "traffic": None, "kernel": k, "kernel_ms": round(k_ms, 5),
                     "algorithmic_bytes_per_launch": int(alg), "peak_source": peak_src + f" x {world} GPUs",
                     "note": "whole-query figure: compulsory input bytes of all ranks / step time; q8 is a chain of small launches, not one streaming kernel"},
        "queries": {"q8": {"ms": dev_ms / args.steps, "events_per_sec": events * args.steps / (dev_ms * 1e-3), "single_share_ms": alone_ms / args.steps,
                           "phases_ms": phases}, **({"q2": q2} if q2 else {})},
        "parity_check": parity,
    }
    ec.close()
    ec_alone.close()
    ctx.close()
    alone.close()
    return result if rank == 0 else None


# ---- the reference's CPU path (oracle port) -----------------------------------------------------------------------
def run_reference(args) -> dict | None:
    """--impl reference: the reference's CPU implementation of the path (oracle port; the Rust original cannot be built
    here) on the host cores.  Never maps libflockgpu.so.  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    if rank != 0:
        return None
    import oracle
    from flock_b200 import nexgen, plans, _ffi
    oracle.lib()
    cores = os.cpu_count() or 1
    metric, config = workload_config(world if world > 1 else args.gpus, args.bids)
    if config["query"] == "q2":
        batches = nexgen.bids_chunked(args.bids, seed=42, columns=["auction", "price"])
        figures = {}
        for label, parts, threads in (("all_cores", min(cores, len(batches)), cores), ("target_partitions_8", 8, min(8, cores)), ("single_thread", 1, 1)):
            tbl, times = oracle.q2_collect(batches, parts, threads, repeat=max(args.warmup, 1) + args.steps)
            times = times[max(args.warmup, 1):]
            figures[label] = {"value": args.bids * len(times) / sum(times), "ms_per_step": sum(times) * 1e3 / len(times),
                              "ms_median": statistics.median(times) * 1e3, "ms_best": min(times) * 1e3, "partitions": parts, "threads": threads}
        au = np.concatenate([b["auction"].to_numpy() for b in batches])
        assert tbl.num_rows == int((np.fmod(au.astype(np.int64), 123) == 0).sum())
        # a second CPU reference point (SURVEY.md 8d): the same query on Arrow C++'s compute kernels through Acero -- the
        # SIMD-vectorised engine of the Arrow project, NOT DataFusion; same batches, all of Arrow's threads
        try:
            import pyarrow.compute as pc
            import pyarrow.dataset as ds
            tab = pa.Table.from_batches(batches)
            a64 = pc.field("auction").cast(pa.int64())
            pred = pc.equal(pc.subtract(a64, pc.multiply(pc.divide(a64, 123), 123)), 0)        # truncated remainder = 0
            ts = []
            for _ in range(1 + min(args.steps, 10)):
                t = time.perf_counter()
                got = ds.dataset(tab).to_table(filter=pred, columns=["auction", "price"], use_threads=True)
                ts.append(time.perf_counter() - t)
            assert got.num_rows == tbl.num_rows
            ts = ts[1:]
            figures["arrow_acero"] = {"value": args.bids * len(ts) / sum(ts), "ms_per_step": sum(ts) * 1e3 / len(ts), "threads": pa.cpu_count(),
                                      "note": "Arrow C++ compute kernels via Acero (pyarrow %s): a SIMD CPU engine, not the reference's DataFusion; not the headline" % pa.__version__}
        except Exception as e:                       # a reference point, never a requirement
            figures["arrow_acero"] = {"value": None, "note": f"failed: {e!r}"[:200]}
        # ---- the other BASELINE configurations on the same host cores (the CPU side of the GPU arm's `queries`): q5 over
        # 100 M bids and q8 over the one-GPU share of 1 B events, native threads, all cores and target_partitions = 8
        by_query = {}
        if not args.no_queries:
            def arm(fn, events):
                out = {}
                for label, parts, threads in (("all_cores", cores, cores), ("target_partitions_8", 8, min(8, cores))):
                    res, ts = fn(parts, threads, 1 + max(1, min(args.steps, 3)))
                    ts = ts[1:]
                    out[label] = {"events_per_sec": events * len(ts) / sum(ts), "ms": sum(ts) * 1e3 / len(ts), "ms_best": min(ts) * 1e3, "partitions": parts,
                                  "threads": threads, "rows_out": res.num_rows}
                return out
            try:
                q1_bids = nexgen.bids_chunked(BATCH_ROWS, seed=42)                     # configs[0]: one 64 Ki-row bid batch
                by_query["q1"] = arm(lambda p, t, r: ((lambda res, ts: (pa.Table.from_batches(res), ts))(*oracle.q1_collect(q1_bids, p, t, repeat=r))), BATCH_ROWS)
                ev3 = nexgen.generate(10_000_000, seed=42, relations=("person", "auction"),
                                      columns={"person": ["p_id", "name", "city", "state"], "auction": ["a_id", "seller", "category"]})
                by_query["q3"] = arm(lambda p, t, r: oracle.q3_collect(ev3["auction"], ev3["person"], p, t, repeat=r), 10_000_000)
                del ev3
                q5_bids = nexgen.bids_chunked(100_000_000, seed=42, columns=["auction"])
                by_query["q5"] = arm(lambda p, t, r: oracle.q5_collect(q5_bids, p, t, repeat=r), 100_000_000)
                del q5_bids
                q8_p, q8_a = q8_slice(0)
                by_query["q8"] = arm(lambda p, t, r: oracle.q8_collect(q8_p, q8_a, p, t, repeat=r), EVENTS_PER_GPU)
                del q8_p, q8_a
            except Exception as e:                   # reference points beside `queries`, never a requirement
                by_query["error"] = repr(e)[:300]
        best = max((k for k in figures if k != "arrow_acero"), key=lambda k: figures[k]["value"])
        value, ms = figures[best]["value"], figures[best]["ms_per_step"]
        sample = (f"all {args.bids} bids per step, {args.steps} steps; native threads inside liboracle.so (orc_q2_collect), one task per partition; "
                  f"headline = {best}")
        used = figures[best]["threads"]
        rows_out = tbl.num_rows
    else:
        persons, auctions = q8_slice(0)
        figures, by_query = {}, {}
        n_steps = max(1, min(args.steps, 10))
        for label, parts, threads in (("all_cores", cores, cores), ("target_partitions_8", 8, min(8, cores)), ("single_thread", 1, 1)):
            out, times = oracle.q8_collect(persons, auctions, parts, threads, repeat=1 + (n_steps if threads > 1 else min(n_steps, 2)))
            times = times[1:]
            figures[label] = {"value": EVENTS_PER_GPU * len(times) / sum(times), "ms_per_step": sum(times) * 1e3 / len(times),
                              "ms_median": statistics.median(times) * 1e3, "ms_best": min(times) * 1e3, "partitions": parts, "threads": threads}
        best = max(figures, key=lambda k: figures[k]["value"])
        value, ms = figures[best]["value"], figures[best]["ms_per_step"]
        sample = (f"ONE rank's share (125 M events = 2.5 M persons + 7.5 M auctions) per step, {n_steps} steps: the CPU has one socket whatever N is; "
                  f"native threads inside liboracle.so (orc_q8_collect: Partial DISTINCT -> hash repartition -> FinalPartitioned DISTINCT -> "
                  f"partitioned join, one task per partition); headline = {best}")
        used, rows_out = figures[best]["threads"], out.num_rows
    assert not _ffi.lib.loaded, "the reference arm must not map the product library"
    return {"impl": "reference", "metric": metric, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32" if config["query"] == "q2" else "int32+utf8",
            "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port", "sample": sample, "figures": figures, "host_cores": cores,
                             **({"queries": by_query} if by_query else {})},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "rows_out": rows_out}


def cpu_baseline(args, world: int, steps: int = 5) -> dict:
    """The CPU arm timed beside the GPU run: `bench.py --impl reference` in a child process, a bounded sample."""
    import subprocess
    cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", str(world), "--steps", str(steps), "--warmup", "1", "--bids", str(args.bids)]
    if args.no_queries:
        cmd.append("--no-queries")
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    if world > 1:
        env["WORLD_SIZE"] = str(world)
        env["RANK"] = "0"
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    line = next((l for l in r.stdout.splitlines() if l.startswith("{")), None)
    if r.returncode != 0 or line is None:
        raise RuntimeError(f"reference arm failed (rc={r.returncode}): {r.stderr[-400:]}")
    d = json.loads(line)
    cb = d["cpu_baseline"]
    cb["sample"] += f"; {d['ms_per_step']:.2f} ms per step"
    cb["rows_out"] = d.get("rows_out")
    return cb


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="gpu", choices=["gpu", "reference"])
    ap.add_argument("--bids", type=int, default=N_BIDS, help="q2: bids per GPU per step (default: the BASELINE.json configuration)")
    ap.add_argument("--e2e-steps", type=int, default=None, help="steps of the host-buffer legs (default: --steps, capped per variant)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-queries", action="store_true", help="skip the `queries` object (q1 / q3 / q5 / q8 on one GPU, q2 on N GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the q2 result of the last timed step as DIR/<column>.npy (float64; seeded sample above 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "gpu" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs applies to the one-GPU q2 run (--impl gpu, one process)")
    if args.impl == "reference":
        res = run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        dist = Dist()
        res = run_gpu_q2(args, dist) if dist.world == 1 else run_gpu_q8(args, dist)
        if dist.world > 1 and res is not None and not args.no_cpu_baseline:
            pass          # cpu_baseline is reported at N = 1 only (tier rule 4)
        dist.close()
    if res is not None:
        print(json.dumps(res), file=_JSON_OUT, flush=True)


if __name__ == "__main__":
    main()
