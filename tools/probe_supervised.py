"""Supervised emission counts: the per-interval path (one _emission.fastUpdateCounts per interval,
as the reference's loop calls it) against the batched path (IndependentMultinomialEmissionModel.
supervisedTrain: host mapping, one upload, one tehmm_supervised_counts).

Shape: K = 10 tracks with bench.py's symbol widths, N = 30 states, 24 tables of ~10^8 rows in all,
10^6 labelled intervals; once without ratios (unit weights, integer histograms) and once with
segmented tables and an effective segment length (weighted chains).  The per-interval path is
timed on the first --sample intervals and reported per interval only.  The batched path is timed
end to end (host mapping included, ends in a device synchronise); its kernel time comes from a
separate torch.profiler run.  Both paths run on the shared subset and their counts are compared
bit for bit.  Writes one JSON line per case to --out, with the card's name and power limit.

    python tools/probe_supervised.py [--out profiles/r03_supervised.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tehmm_b200 import _emission, synth  # noqa: E402
from tehmm_b200.emission import IndependentMultinomialEmissionModel  # noqa: E402
from tehmm_b200.engine import get_engine  # noqa: E402
from tehmm_b200.track import IntegerTrackTable  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:                       # noqa: BLE001
        return {"gpu": "unknown (%s)" % e, "power_limit": "unknown"}


def make_tables(rng, syms, ntab, rows_per_table, segmented):
    """ntab tables on chr1..chrN; segmented ones span ~2x their rows in genome coordinates"""
    tables = []
    for i in range(ntab):
        if segmented:
            lens = rng.integers(1, 4, size=rows_per_table)
            offs = np.concatenate([[0], np.cumsum(lens[:-1])]).astype(np.int64)
            span = int(offs[-1] + lens[-1])
            t = IntegerTrackTable(len(syms), "chr%d" % (i + 1), 0, span)
            t.segOffsets = offs
            t.data = np.empty((rows_per_table, len(syms)), dtype=np.uint8)
            t.shape = (rows_per_table, len(syms))
        else:
            t = IntegerTrackTable(len(syms), "chr%d" % (i + 1), 0, rows_per_table)
        for k, s in enumerate(syms):
            t.data[:, k] = rng.integers(0, s + 1, size=t.data.shape[0], dtype=np.uint8)
        tables.append(t)
    return tables


def make_intervals(rng, tables, n, N):
    """n sorted, disjoint intervals spread over the tables in genome coordinates"""
    per = n // len(tables)
    out = []
    for t in tables:
        span = t.getEnd() - t.getStart()
        starts = np.sort(rng.choice(span - 1, size=per, replace=False))
        ends = np.minimum(np.append(starts[1:], span), starts + rng.integers(1, 2 * (span // per), size=per))
        st = rng.integers(0, N, size=per)
        out.extend(zip([t.getChrom()] * per, starts.tolist(), ends.tolist(), st.tolist()))
    return out


def batched(model, tables, intervals):
    seen = {}
    model.maximize = lambda obsStats, trackList=None: seen.setdefault("stats", obsStats.copy())
    model.supervisedTrain(types.SimpleNamespace(getTrackTableList=lambda: tables, getTrackList=lambda: None), intervals)
    return seen["stats"]


def per_interval(model, tables, intervals):
    """emission.py:293-331 with fastUpdateCounts per interval"""
    obsStats = model.initStats()
    lastTable, lastRatios, lastHit, lastOverlapEnd = None, None, 0, -1
    for interval in intervals:
        hit = False
        for tableIdx in range(lastHit, len(tables)):
            table = tables[tableIdx]
            overlap = table.getOverlapInTableCoords(interval, lastOverlapEnd)
            if overlap is not None:
                lastHit, hit = tableIdx, True
                lastOverlapEnd = max(0, overlap[2] - 1)
                if table is not lastTable:
                    lastRatios, lastTable = model.getSegmentRatios(table), table
                _emission.fastUpdateCounts(overlap, table, obsStats, lastRatios)
            elif hit is True:
                break
    return obsStats


def kernel_ms(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "sup_" in e.key)
    return us / 1000.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_supervised.jsonl"))
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--tables", type=int, default=24)
    ap.add_argument("--intervals", type=int, default=1_000_000)
    ap.add_argument("--sample", type=int, default=10_000)
    ap.add_argument("--sample-segmented", type=int, default=1_000,
                    help="per-interval sample with segmented tables (each call scans the whole table's offsets)")
    ap.add_argument("--N", type=int, default=30)
    args = ap.parse_args()
    import torch
    info = card()
    syms = list(synth.BENCH_SYMS)
    K, N = len(syms), args.N
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    eng = get_engine(0)
    with open(args.out, "a") as f:
        for ratios in (False, True):
            rng = np.random.default_rng(1 + ratios)
            tables = make_tables(rng, syms, args.tables, args.rows // args.tables, ratios)
            intervals = make_intervals(rng, tables, args.intervals, N)
            model = lambda: IndependentMultinomialEmissionModel(N, syms, effectiveSegmentLength=2 if ratios else None)  # noqa: E731
            batched(model(), tables, intervals[:1000])           # warm-up: module load, allocations
            torch.cuda.synchronize()
            launches0 = eng.ctx.launches
            t0 = time.perf_counter()
            full = batched(model(), tables, intervals)
            torch.cuda.synchronize()
            t_new = time.perf_counter() - t0
            launches = eng.ctx.launches - launches0
            from tehmm_b200.supervised import interval_triples
            t0 = time.perf_counter()
            trip = interval_triples(tables, intervals)
            t_map = time.perf_counter() - t0
            kms = kernel_ms(lambda: batched(model(), tables, intervals))
            ns = args.sample_segmented if ratios else args.sample
            sub = intervals[:ns]
            t0 = time.perf_counter()
            old = per_interval(model(), tables, sub)
            t_old = time.perf_counter() - t0
            new_sub = batched(model(), tables, sub)
            rec = dict(info, case="ratios" if ratios else "unit", K=K, N=N, syms=syms, tables=args.tables,
                       rows=int(sum(t.shape[0] for t in tables)), intervals=len(intervals),
                       counted_rows=int((trip[2] - trip[1]).sum()),
                       batched_s=round(t_new, 4), host_mapping_s=round(t_map, 4), kernel_ms=round(kms, 3),
                       batched_launches=launches, per_interval_sample=ns,
                       per_interval_us=round(1e6 * t_old / ns, 2),
                       sample_equal=bool(np.array_equal(old, new_sub)), total_counts=float(full.sum()))
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")
            assert rec["sample_equal"], "batched and per-interval counts differ"


if __name__ == "__main__":
    main()
