"""Windowed forward-backward (DESIGN.md section 11) on one GPU; one JSON line per case.

    python tools/probe_windowed.py [--c5] > profiles/r03_windowed.jsonl

case 1: 20 M steps x 50 states, E-step in 4 windows against the unwindowed E-step: time ratio
        (CUDA events around whole E-steps, mean of 3 after a warm-up) and the largest relative
        difference of the statistics.
case 2 (--c5): config 5, one sequence of 250 M steps at 50 states, whose lattices do not fit:
        one E-step (windows planned from free memory), its time and peak device memory, and
        its log-likelihood against Engine.score (forward only, which fits).
The card's name and power limit are read in the same run."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(torch, fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.mean(ts)), out


def rel_diff(a, b):
    worst = 0.0
    for k in ("start", "trans", "obs"):
        x, y = np.asarray(a[k]), np.asarray(b[k])
        big = np.abs(y) > 1e-6 * np.abs(y).max()
        worst = max(worst, float((np.abs(x - y)[big] / np.abs(y)[big]).max()))
    return worst


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
    t_plain, a = timed(torch, lambda: eng.estep())
    t_win, b = timed(torch, lambda: eng.estep(max_window_steps=T // 4))
    return {"case": "20M_x_50_estep", "steps": T, "states": 50, "windows": 4, "ms_unwindowed": t_plain,
            "ms_windowed": t_win, "time_ratio": t_win / t_plain, "max_rel_diff_stats": rel_diff(b, a),
            "logprob_rel_diff": abs(b["logprob"] - a["logprob"]) / abs(a["logprob"])}


def case2():
    import torch
    from run_configs import sample_long
    from tehmm_b200 import synth
    from tehmm_b200.engine import get_engine
    m = synth.make_model(N=50, seed=0)
    T = 250_000_000
    obs = sample_long(synth, m, T, seed=300)
    eng = get_engine(0)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    lp_score = float(eng.score()[0])
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(eng.device)
    t0 = time.perf_counter()
    st = eng.estep()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    return {"case": "c5_estep", "steps": T, "states": 50, "estep_seconds": sec,
            "peak_gb": torch.cuda.max_memory_allocated(eng.device) / 1e9,
            "estep_logprob": st["logprob"], "score_logprob": lp_score,
            "logprob_rel_diff": abs(st["logprob"] - lp_score) / abs(lp_score),
            "score_samples": "not measured"}


if __name__ == "__main__":
    gpu = card()
    for fn in [case1] + ([case2] if "--c5" in sys.argv else []):
        r = fn()
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)
