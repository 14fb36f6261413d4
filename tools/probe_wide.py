#!/usr/bin/env python
"""33..64 states, one sequence: forward pass by the tcgen05 kernel (default) against the one-chunk-per-warp
kernel (option "tile" = 0); log-likelihoods must agree."""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from tehmm_b200 import _lib, synth
from tehmm_b200.engine import Engine

T = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
ctx = _lib.get_context(0); eng = Engine(ctx)
for N in (50, 64, 33):
    m = synth.make_model(N=N, seed=0)
    obs, _ = synth.sample_obs(m, T, seed=1)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    prec, tdt = eng._prec("f32")
    _, blin, rowmax = eng.run_emission(prec, tdt, None, False, True)
    torch.cuda.synchronize()
    ctx.set_option("timing", 1)
    for _ in range(3):
        _, blin, rowmax = eng.run_emission(prec, tdt, None, False, True)
    torch.cuda.synchronize()
    us_em = ctx.stat("us_emission")
    ctx.set_option("timing", 0)
    res = {}
    bres = {}
    for opt in (1, 0):
        ctx.set_option("tile", opt)
        for _ in range(2):
            alpha, lp = ctx.optimistic(lambda: eng.run_forward(prec, tdt, blin, rowmax, None))
        torch.cuda.synchronize()
        ctx.set_option("timing", 1)
        for _ in range(3):
            alpha, lp = ctx.optimistic(lambda: eng.run_forward(prec, tdt, blin, rowmax, None))
        torch.cuda.synchronize()
        res[opt] = (ctx.stat("us_forward"), float(lp[0].item()), ctx.stat("umma_passes"), ctx.stat("repaired_chunks_forward"))
        # backward twin: MAP only, and posteriors + MAP
        for fl in (2, 3):
            for _ in range(3):
                outs = ctx.optimistic(lambda: eng.run_backward(prec, tdt, fl, blin, alpha, None))
            torch.cuda.synchronize()
            bres.setdefault(opt, {})[fl] = (ctx.stat("us_backward"), outs[1].cpu().numpy() if outs[1] is not None else None)
            del outs
        ctx.set_option("timing", 0)
    ctx.set_option("tile", 1)
    elog, _, rm = eng.run_emission(prec, tdt, None, True, False)
    for _ in range(2):
        vs = ctx.optimistic(lambda: eng.run_viterbi(prec, elog, None, None, want64=False, rowmax=rm))
    torch.cuda.synchronize()
    ctx.set_option("timing", 1)
    for _ in range(3):
        vs = ctx.optimistic(lambda: eng.run_viterbi(prec, elog, None, None, want64=False, rowmax=rm))
    torch.cuda.synchronize()
    vit = {"viterbi_dp_us": ctx.stat("us_viterbi_dp"), "traceback_us": ctx.stat("us_traceback"), "rescore_us": ctx.stat("us_rescore"),
           "repaired_traceback": ctx.stat("repaired_chunks_traceback")}
    ctx.set_option("timing", 0)
    del elog, vs
    print(json.dumps(vit), flush=True)
    print(json.dumps({"N": N, "T": T, "emission_us": us_em, "tcgen05_us": res[1][0], "warp_kernel_us": res[0][0], "logprob_tcgen05": res[1][1],
                      "logprob_warp": res[0][1], "rel_diff": abs(res[1][1] - res[0][1]) / abs(res[0][1]),
                      "umma_passes": res[1][2], "repaired": res[1][3],
                      "bwd_map_tcgen05_us": bres[1][2][0], "bwd_map_warp_us": bres[0][2][0],
                      "bwd_post_map_tcgen05_us": bres[1][3][0], "bwd_post_map_warp_us": bres[0][3][0],
                      "map_agreement": float(np.mean(bres[1][2][1] == bres[0][2][1])),
                      "repaired_backward": ctx.stat("repaired_chunks_backward")}), flush=True)
