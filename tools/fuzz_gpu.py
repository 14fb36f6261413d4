#!/usr/bin/env python
"""Randomised parity sweep of the batched device path against the CPU oracle: random state counts,
track counts / alphabet sizes, sequence raggedness, chunking options.  Prints one line per case and a
summary; exit code 1 on any mismatch.   python tools/fuzz_gpu.py [ncases] [seed]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np
import oracle as orc
from tehmm_b200 import _lib, synth
from tehmm_b200.engine import get_engine

orc.build()
ncases = int(sys.argv[1]) if len(sys.argv) > 1 else 40
rng = np.random.RandomState(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
eng = get_engine(0)
bad = 0
for case in range(ncases):
    N = int(rng.choice([2, 3, 5, 8, 17, 30, 31, 32, 33, 40, 50, 64]))
    K = int(rng.randint(1, 13))
    syms = tuple(int(rng.choice([1, 2, 3, 4, 7, 16, 33, 64, 120, 250])) for _ in range(K))
    m = synth.make_model(N=N, syms=syms, seed=int(rng.randint(1 << 30)), zero_frac=float(rng.choice([0.0, 0.2, 0.5])))
    nseq = int(rng.randint(1, 6))
    lens = [int(rng.choice([1, 2, 17, 63, 64, 65, 300, 1000, 4097, 20000])) for _ in range(nseq)]
    dtype = rng.choice([np.uint8, np.uint16, np.int32])
    seqs = [synth.sample_obs(m, n, seed=int(rng.randint(1 << 30)))[0].astype(dtype) for n in lens]
    opts = dict(chunk_tiles=int(rng.choice([0, 1, 4])), warmup=int(rng.choice([0, 8, 64])),
                fine_len=int(rng.choice([0, 64, 100])), tile=int(rng.choice([1, 1, 0])))
    for k, v in opts.items():
        eng.ctx.set_option(k, v)
    prec = str(rng.choice(["f32", "f32", "f64"]))
    only = os.environ.get("FUZZ_ONLY")          # replay ONE case of a seed (the draws above keep the generator in step)
    if only is not None and int(only) != case:
        continue
    tol = 1e-5 if prec == "f32" else 1e-10
    # absolute floor of a log-likelihood: a model that explains every observation with probability 1 (one symbol per
    # track) has log P = 0, and float32 carries ~3e-10 per step of rounding in the transition rows
    # (3e-10 on the CUDA-core kernels; the tensor-core forward kernels accumulate with round-toward-zero: a
    #  systematic -2.2e-7 nat per step, DESIGN.md section 6)
    floor = 1e-9 + (5e-7 * sum(lens) if prec == "f32" else 0.0)
    msg = []
    try:
        eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
        lpv, _, st = eng.decode_host(seqs, _lib.DECODE_VITERBI, precision=prec)
        flp, sc, ms = eng.decode_host(seqs, _lib.DECODE_MAP, precision=prec)
        eng.upload_batch(seqs)
        es = eng.estep(precision=prec)
        Kk, Nn, S = m["table"].shape
        s0, tr, ob = np.zeros(Nn), np.zeros((Nn, Nn)), np.zeros((Kk, Nn, S))
        lp_sum = 0.0
        for i, o in enumerate(seqs):
            ref = orc.sweep_sequence(o, m["table"], 1.0, m["log_start"], m["log_trans"])
            lp_sum += orc.estep_sequence(o, m["table"], 1.0, m["log_start"], m["log_trans"], None, s0, tr, ob)
            if abs(lpv[i] - ref["vit_logprob"]) > 1e-6 * abs(ref["vit_logprob"]) + 1e-9:
                msg.append("viterbi logprob seq %d: %r vs %r" % (i, lpv[i], ref["vit_logprob"]))
            if abs(flp[i] - ref["logprob"]) > tol * abs(ref["logprob"]) + floor:
                msg.append("logprob seq %d: %r vs %r" % (i, flp[i], ref["logprob"]))
            agree = float(np.mean(st[i] == ref["vit_states"]))
            # float32 near-ties: 3 % of the steps -- at least one step from 8 steps on, none on shorter sequences
            slack = max(1.0, 0.03 * len(o)) / len(o) if len(o) >= 8 else 0.0
            if (prec == "f64" and agree < 1.0) or agree < 1.0 - slack:
                msg.append("viterbi path seq %d agreement %.4f" % (i, agree))
            if float(np.mean(ms[i] == ref["map_states"])) < 1.0 - slack:
                msg.append("map path seq %d agreement %.4f" % (i, float(np.mean(ms[i] == ref["map_states"]))))
        if abs(es["logprob"] - lp_sum) > tol * abs(lp_sum) + floor:
            msg.append("estep logprob %r vs %r" % (es["logprob"], lp_sum))
        for name, got, want in (("start", es["start"], s0), ("trans", es["trans"], tr), ("obs", es["obs"], ob)):
            # float64: the oracle's (= the reference's) LOG-space lattices and normaliser carry absolute rounding that
            # grows with |log alpha|: at T = 2e4 its raw counts are off by a uniform 1.1e-7 relative against an
            # extended-precision evaluation while ours agree with it to 1e-15 (seed 13 case 56 of this tool as of
            # commit 029b7fc, whose option draws differ from today's; replayed there with FUZZ_ONLY=56:
            # profiles/r02_fuzz.txt) -- so 1e-6 against the oracle here, 1e-10 on the short golden vectors
            if not np.allclose(got, want, rtol=10 * tol if prec == "f32" else 1e-6, atol=2e-5 if prec == "f32" else 1e-9):
                msg.append("estep %s max abs err %.3g" % (name, float(np.abs(got - want).max())))
                if only is not None and name == "trans":
                    # who is right: an extended-precision (64-bit mantissa) evaluation in scaled space
                    sys.path.insert(0, os.path.join(ROOT, "tests"))
                    from parity import oracle_frame, trans_counts_extended
                    truth = trans_counts_extended([oracle_frame(orc, o, m["table"]) for o in seqs], m["log_start"], m["log_trans"])
                    with np.errstate(divide="ignore", invalid="ignore"):
                        print("trans counts (extended-precision arbiter):\n", truth)
                        print("ours   - arbiter, relative:\n", (got - truth) / truth)
                        print("oracle - arbiter, relative:\n", (want - truth) / truth)
    except Exception as e:                      # noqa: BLE001
        msg.append("EXCEPTION %r" % (e,))
    bad += bool(msg)
    print("case %2d N=%2d K=%2d syms=%s lens=%s %s %s %s -> %s" % (case, N, K, syms, lens, np.dtype(dtype).name, prec, opts,
                                                                   "OK" if not msg else "; ".join(msg)), flush=True)
for k in ("chunk_tiles", "warmup", "fine_len"):
    eng.ctx.set_option(k, 0)
eng.ctx.set_option("tile", 1)
print("%d of %d cases failed" % (bad, ncases))
sys.exit(1 if bad else 0)
