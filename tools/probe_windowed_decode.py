"""Viterbi and MAP decoding in time windows (DESIGN.md section 11) on one GPU; one JSON line per case.

    python tools/probe_windowed_decode.py [--c5] > profiles/r03_windowed_decode.jsonl

case 1: 20 M steps x 50 states.  Engine.viterbi in 4 windows against the unwindowed call, and
        Engine.decode_host_both (Viterbi, then MAP, each in 4 windows) against the one-call host decode:
        time ratios (CUDA events around whole calls, mean of 3 after a warm-up), divergent Viterbi
        steps, MAP state agreement and log-probability differences.
case 2 (--c5): config 5, MultitrackHmm.decode_both of one 250 M-step, 50-state sequence from host
        arrays.  The one-call decode's arena (three lattices) does not fit, the library returns
        TEHMM_ENOMEM and the engine decodes the uploaded batch, in windows where free memory asks for
        them: seconds and peak device memory, and the Viterbi path against the unwindowed Engine.viterbi.
The card's name and power limit are read in the same run."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from probe_windowed import card, timed   # noqa: E402


def divergent(a, b):
    return int(sum(int(np.count_nonzero(x != y)) for x, y in zip(a, b)))


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b)))


def case1():
    import torch
    from run_configs import sample_long
    from tehmm_b200 import synth
    from tehmm_b200.engine import get_engine
    m = synth.make_model(N=50, seed=0)
    T = 20_000_000
    obs = sample_long(synth, m, T, seed=301)
    eng = get_engine(0)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    t_plain, (lp_a, st_a) = timed(torch, lambda: eng.viterbi())
    t_win, (lp_b, st_b) = timed(torch, lambda: eng.viterbi(max_window_steps=T // 4))
    out = {"case": "20M_x_50_decode", "steps": T, "states": 50, "windows": 4,
           "viterbi_ms_unwindowed": t_plain, "viterbi_ms_windowed": t_win, "viterbi_time_ratio": t_win / t_plain,
           "viterbi_divergent_steps": divergent(st_b, st_a), "viterbi_logprob_rel_diff": rel(lp_b, lp_a)}
    t_plain, a = timed(torch, lambda: eng.decode_host_both([obs]))
    t_win, b = timed(torch, lambda: eng.decode_host_both([obs], max_window_steps=T // 4))
    out.update({"both_ms_one_call": t_plain, "both_ms_windowed": t_win, "both_time_ratio": t_win / t_plain,
                "both_viterbi_divergent_steps": divergent(b[1], a[1]),
                "both_viterbi_logprob_rel_diff": rel(b[0], a[0]),
                "both_map_agreement": 1.0 - divergent(b[3], a[3]) / T,
                "both_map_score_rel_diff": rel(b[2], a[2]), "both_forward_logprob_rel_diff": rel(b[4], a[4])})
    return out


def case2():
    import torch
    from run_configs import sample_long
    from tehmm_b200 import synth
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    from tehmm_b200.engine import get_engine
    from tehmm_b200.hmm import MultitrackHmm
    m = synth.make_model(N=50, seed=0)
    T = 250_000_000
    obs = sample_long(synth, m, T, seed=300)
    em = IndependentMultinomialEmissionModel(50, list(m["syms"]), zeroAsMissingData=True)
    em.logProbs = m["table"].copy()
    h = MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy())
    eng = get_engine(0)
    calls = []
    plain = type(eng)._decode_windows

    def spy(self, *args):
        calls.append(args[1])
        return plain(self, *args)
    type(eng)._decode_windows = spy
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(eng.device)
    t0 = time.perf_counter()
    vlp, vst, msc, mst = h.decode_both(obs)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    peak = torch.cuda.max_memory_allocated(eng.device) / 1e9
    type(eng)._decode_windows = plain
    out = {"case": "c5_decode_both", "steps": T, "states": 50, "decode_both_seconds": sec,
           "out_of_memory_route": len(calls) == 1, "peak_gb_torch": peak,
           "viterbi_logprob": vlp, "map_score": msc}
    eng.upload_batch([obs])
    lp_u, st_u = eng.viterbi()
    out.update({"unwindowed_viterbi_logprob": float(lp_u[0]), "viterbi_divergent_steps": divergent([vst], st_u),
                "viterbi_logprob_rel_diff": rel([vlp], lp_u)})
    return out


if __name__ == "__main__":
    gpu = card()
    for fn in [case1] + ([case2] if "--c5" in sys.argv else []):
        r = fn()
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)
