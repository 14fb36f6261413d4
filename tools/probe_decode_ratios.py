#!/usr/bin/env python
"""Decoding of segmented tables with host buffers (tehmm_decode_host_ratios / _both_ratios).

Three measurements on one GPU, with the card's name and power limit read in the same run:

  viterbi  C3-shaped batch (350 sequences, 3.5 M steps, 30 states, uint8, segments of up to 100
           bins, ratio = segment length / 100 as bench.py builds it), end to end from NumPy in to
           int64 states out: the device-pointer route (upload_batch + Engine.viterbi(ratios_dp=...))
           against Engine.decode_host(..., ratios=...).  The two calls alternate; median of --reps.
  both     the same batch as segmented IntegerTrackTables: MultitrackHmm.decode_both_batch against
           decode_batch(viterbi) + decode_batch(map).
  dp50     one 10 M-step sequence, 50 states: kernel time of the fp32 Viterbi DP with ratios
           (viterbi_wide_kernel<true>) against without (<false>), from the library's CUDA events
           (option "timing", mean over the launches).

Outputs of the routes being compared are checked for equality.  One JSON line per measurement to --out.

    python tools/probe_decode_ratios.py [--out profiles/r03_decode_ratios.jsonl] [--reps 7]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tehmm_b200 import _lib, synth  # noqa: E402
from tehmm_b200.emission import IndependentMultinomialEmissionModel  # noqa: E402
from tehmm_b200.engine import get_engine  # noqa: E402
from tehmm_b200.hmm import MultitrackHmm  # noqa: E402
from tehmm_b200.track import IntegerTrackTable  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power}


def sync():
    import torch
    torch.cuda.synchronize()


def timed(fn):
    sync()
    t0 = time.perf_counter()
    out = fn()
    sync()
    return time.perf_counter() - t0, out


def c3_batch(m):
    lens = synth.bench_lengths("c3")
    rng = np.random.RandomState(3)
    obs, tables = [], []
    for i, n in enumerate(lens):
        o = synth.sample_obs(m, n, seed=100 + i)[0]
        seg = np.minimum(rng.geometric(1.0 / 60.0, size=n), 100).astype(np.int64)
        t = IntegerTrackTable(o.shape[1], "chrG", 0, int(seg.sum()))
        t.segOffsets = np.concatenate([[0], np.cumsum(seg)[:-1]]).astype(np.int64)
        t.data = o
        t.shape = (len(t), o.shape[1])
        obs.append(o)
        tables.append(t)
    return obs, tables


def make_hmm(m, **kw):
    em = IndependentMultinomialEmissionModel(m["N"], list(m["syms"]), zeroAsMissingData=True, fudge=0.0,
                                             effectiveSegmentLength=100)
    em.logProbs = m["table"].copy()
    return MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy(), **kw), em


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_decode_ratios.jsonl"))
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--dp-steps", type=int, default=10_000_000)
    args = ap.parse_args()
    info = card()
    eng = get_engine(0)
    lines = []

    def emit(d):
        d = dict(info, **d)
        print(json.dumps(d), flush=True)
        lines.append(d)

    # ---- Viterbi with ratios, end to end
    m = synth.make_model(N=30, seed=0)
    obs, tables = c3_batch(m)
    hv, em = make_hmm(m)
    hm, _ = make_hmm(m, algorithm="map")
    hb, _ = make_hmm(m)
    ratios = [em.getSegmentRatios(t) for t in tables]
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])

    def old():
        eng.upload_batch(obs)
        return eng.viterbi(ratios_em=None, ratios_dp=ratios)

    def new():
        lp, _, st = eng.decode_host(obs, _lib.DECODE_VITERBI, ratios=ratios)
        return lp, st
    for _ in range(2):
        old(), new()
    t_old, t_new = [], []
    for _ in range(args.reps):
        a, out_old = timed(old)
        b, out_new = timed(new)
        t_old.append(a)
        t_new.append(b)
    same = bool(np.array_equal(out_old[0], out_new[0]) and all(np.array_equal(x, y) for x, y in zip(out_old[1], out_new[1])))
    emit({"case": "viterbi_with_ratios_end_to_end", "N": 30, "nseq": len(obs), "steps": int(sum(len(o) for o in obs)),
          "device_pointer_route_ms": 1e3 * float(np.median(t_old)), "host_call_ms": 1e3 * float(np.median(t_new)),
          "device_pointer_route_ms_all": [round(1e3 * x, 2) for x in t_old],
          "host_call_ms_all": [round(1e3 * x, 2) for x in t_new], "reps": args.reps, "outputs_identical": same})

    # ---- both decodings
    def two():
        return hv.decode_batch(tables), hm.decode_batch(tables)

    def one():
        return hb.decode_both_batch(tables)
    for _ in range(2):
        two(), one()
    t_two, t_one = [], []
    for _ in range(args.reps):
        a, (v, mp) = timed(two)
        b, bo = timed(one)
        t_two.append(a)
        t_one.append(b)
    same = all(x[0] == y[0] and x[2] == z[0] and np.array_equal(x[1], y[1]) and np.array_equal(x[3], z[1])
               for x, y, z in zip(bo, v, mp))
    emit({"case": "decode_both_with_ratios", "N": 30, "nseq": len(obs), "steps": int(sum(len(o) for o in obs)),
          "two_calls_ms": 1e3 * float(np.median(t_two)), "decode_both_batch_ms": 1e3 * float(np.median(t_one)),
          "two_calls_ms_all": [round(1e3 * x, 2) for x in t_two],
          "decode_both_batch_ms_all": [round(1e3 * x, 2) for x in t_one],
          "reps": args.reps, "outputs_identical": bool(same)})
    del obs, tables, ratios, out_old, out_new, v, mp, bo

    # ---- the 50-state DP with and without ratios
    m = synth.make_model(N=50, seed=0)
    T = args.dp_steps
    o = synth.sample_obs(m, T, seed=1)[0]
    r = np.minimum(np.random.RandomState(4).geometric(1.0 / 60.0, size=T), 100) / 100.0
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([o])
    prec, tdt = eng._prec("f32")
    elog, _, rowmax = eng.run_emission(prec, tdt, None, True, False)
    d_r = eng.upload_ratios([r])
    ctx = eng.ctx
    res = {}
    for name, dr in (("with_ratios", d_r), ("without_ratios", None), ("with_ratios_again", d_r)):
        for _ in range(2):
            ctx.optimistic(lambda: eng.run_viterbi(prec, elog, None, dr, want64=False, rowmax=rowmax))
        sync()
        rep0 = ctx.stat("repaired_chunks_viterbi")
        ctx.set_option("timing", 1)
        for _ in range(5):
            ctx.optimistic(lambda: eng.run_viterbi(prec, elog, None, dr, want64=False, rowmax=rowmax))
        sync()
        res[name] = {"dp_us": ctx.stat("us_viterbi_dp"), "traceback_us": ctx.stat("us_traceback"),
                     "rescore_us": ctx.stat("us_rescore"),
                     "repaired_chunks": ctx.stat("repaired_chunks_viterbi") - rep0}
        ctx.set_option("timing", 0)
    emit({"case": "dp_50_states", "N": 50, "steps": T, "kernel_with": "viterbi_wide_kernel<true>",
          "kernel_without": "viterbi_wide_kernel<false>", "launches_timed": 5, **res})
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
