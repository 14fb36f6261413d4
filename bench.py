#!/usr/bin/env python
"""bench.py -- trellis cells/s of one fwd-bwd + Viterbi sweep (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: emission gather-sum ->
forward -> backward with posterior argmax (MAP) -> Viterbi DP -> traceback +
float64 re-score.  Workload at N=1 = BASELINE.json configs[1]: 10 tracks
(6 multinomial + 4 binary), 30 states, ONE sequence of 10 M observations
(alyrata-like synthetic, sampled from the model).  With N GPUs every rank runs
its own sequence of the same shape (weak scaling, no data-path collective).

value  : cells/s (sum over ranks of T*N, divided by the max-over-ranks device
         time of the K timed steps), observations already resident in HBM.
e2e    : the same metric through the public API with HOST buffers
         (MultitrackHmm.decode_batch for Viterbi and for MAP): H2D of the
         observations and D2H of the int64 state paths inside the timed region.
--impl reference : the reference's own CPU implementation (oracle/_ref when it
         is built, else the oracle port) on the host cores, one process per core
         in the style of teHmmEval --chroms --proc.
--dump-outputs DIR : after the timed steps, what the last one returned on rank 0 (scores
         float64, state paths float32, sampled at fixed positions beyond 2 M steps) as
         DIR/<name>.npy.  Model and observations come from fixed seeds, so two builds run with
         the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the tree may be read-only; bench.py writes nothing into it

METRIC = "hmm_trellis_cells_per_sec_fwd_bwd_viterbi"
UNIT = "cells/s"
N_STATES, T_DEFAULT = 30, 10_000_000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--T", type=int, default=T_DEFAULT, help="observations per GPU")
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--cpu-sample", type=int, default=400_000, help="observations of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-em", action="store_true")
    ap.add_argument("--no-split", action="store_true", help="skip the strong-scaling runs of configs 3 and 4")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def workload_config(T, gpus):
    return {"workload": "c2: alyrata-like synthetic, 10 multinomial/binary tracks, 30 states, one "
                        "sequence of %d observations per GPU, fwd-bwd(MAP)+Viterbi sweep" % T,
            "states": N_STATES, "tracks": 10, "obs_per_gpu": T, "gpus": gpus,
            "l2": "inputs larger than L2 (obs %.0f MB, lattices %.1f GB per GPU), no flush needed" % (
                T * 10 / 1e6, T * N_STATES * 4 * 3 / 1e9)}


# ------------------------------------------------------------------ clocks
class ClockSampler(object):
    """SM clock / throttle reasons DURING the timed region.  The timed region is a
    few tens of milliseconds, far below nvidia-smi's sampling period, so NVML is
    polled directly from a thread (nvidia-smi --query-gpu is the fallback)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None
        self.thread = threading.Thread(target=self._poll if self.nvml else self._poll_smi, daemon=True)
        self.thread.start()

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    reasons = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    reasons = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                try:
                    power = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                except Exception:
                    power = 0.0
                self.samples.append((sm, reasons, power))
            except Exception:
                pass
            time.sleep(0.002)

    def _poll_smi(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                bits = 0
                for bit, v in zip((0x8, 0x40, 0x20, 0x4), f[3:7]):
                    if v.lower().startswith("active"):
                        bits |= bit
                self.max_sm = float(f[1])
                self.samples.append((float(f[0]), bits, float(f[2])))
            except Exception:
                time.sleep(0.05)

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = set()
        for _, bits, _ in self.samples:
            for bit, nm in names.items():
                if bits & bit:
                    reasons.add(nm)
        sm = [x[0] for x in self.samples]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(getattr(self, "max_sm", max(sm))),
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(x[2] for x in self.samples),
                "source": "nvml" if self.nvml else "nvidia-smi"}


# ------------------------------------------------------------------ CPU arms
def cpu_sweep_reference(R, m, obs):
    """the reference's own Cython functions + its NumPy glue (basehmm.py:265-272,357)"""
    T, N = obs.shape[0], m["N"]
    frame = np.zeros((T, N))
    R._emission.fastAllLogProbs(obs, m["table"], frame, 1.0, None)
    fwd = np.zeros((T, N))
    R._hmm._forward(T, N, m["log_start"], m["log_trans"], frame, None, fwd)
    bwd = np.zeros((T, N))
    R._hmm._backward(T, N, m["log_start"], m["log_trans"], frame, None, bwd)
    gamma = fwd + bwd
    post = np.exp(gamma.T - R.basehmm.logsumexp(gamma, axis=1)).T
    post += np.finfo(np.float32).eps
    post /= np.sum(post, axis=1).reshape((-1, 1))
    mp = np.argmax(post, axis=1)
    st, lp = R._hmm._viterbi(T, N, m["log_start"], m["log_trans"], None, frame)
    return lp, st, mp


def cpu_sweep(kind, m, obs):
    if kind == "reference":
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ref_loader
        return cpu_sweep_reference(ref_loader.load(), m, obs)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    r = orc.sweep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"])
    return r["vit_logprob"], r["vit_states"], r["map_states"]


def cpu_kind():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import ref_loader
        if ref_loader.available():
            ref_loader.load()
            return "reference"
    except Exception:
        pass
    import oracle as orc
    orc.build()
    return "port"


def _cpu_worker(args):
    kind, seed, T = args
    from tehmm_b200 import synth
    m = synth.make_model(N=N_STATES, seed=0)
    obs, _ = synth.sample_obs(m, T, seed=seed)
    t0 = time.perf_counter()
    cpu_sweep(kind, m, obs)
    return time.perf_counter() - t0


def run_reference_arm(args):
    """--impl reference: every host core runs the reference sweep on its own slice."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    kind = cpu_kind()
    cores = os.cpu_count() or 1
    per = max(20_000, min(100_000, args.cpu_sample // 4))
    ctx = mp.get_context("fork")
    times = []
    with ctx.Pool(cores) as pool:
        for it in range(args.warmup + args.steps):
            # step time = slowest worker's sweep (data generation is outside the clock)
            dt = max(pool.map(_cpu_worker, [(kind, 1000 + 97 * it + c, per) for c in range(cores)]))
            if it >= args.warmup:
                times.append(dt)
    total = sum(times)
    cells = float(args.steps) * cores * per * N_STATES
    value = cells / total
    line = {"metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": dict(workload_config(args.T, args.gpus),
                           ran="bounded sample of that workload: %d processes x %d observations per step "
                               "(same model, one sequence each); the reference is O(T), cells/s does not depend on T" % (cores, per),
                           obs_per_step=cores * per),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": "%d processes x %d observations per step (one sequence each, "
                                       "teHmmEval --chroms --proc style), N=30, K=10" % (cores, per)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------ strong scaling of configs 3 and 4
def run_split(world, rank):
    """BASELINE.json configs[3] and [2] split over the ranks the way north_star says: the 24
    chromosomes of the hg19-scale decode and the 350 training sequences are dealt to the ranks by
    longest-processing-time bin packing (parallel.shard_indices); decoding needs no collective, an
    EM iteration ends in ONE all-reduce of the packed statistics.  Fixed total work (strong
    scaling); host wall clock between barriers, max over ranks."""
    import torch
    import torch.distributed as dist
    from tehmm_b200 import parallel, synth
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    from tehmm_b200.hmm import MultitrackHmm

    def reduce(x, op):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def make_hmm(m, seg_len=None, **kw):
        em = IndependentMultinomialEmissionModel(m["N"], list(m["syms"]), zeroAsMissingData=True, effectiveSegmentLength=seg_len)
        em.logProbs = m["table"].copy()
        return MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy(), **kw), em

    def sample_long(m, T, seed, piece=4_000_000):
        out = np.empty((T, m["K"]), dtype=np.uint8)
        for i, a in enumerate(range(0, T, piece)):
            n = min(piece, T - a)
            out[a:a + n] = synth.sample_obs(m, n, seed=seed + i)[0]
        return out

    MAX, SUM = (dist.ReduceOp.MAX, dist.ReduceOp.SUM) if world > 1 else (None, None)
    out = {}
    m = synth.make_model(N=N_STATES, seed=0)
    # ---- config 4: hg19-scale decode, chromosomes sharded
    lens = synth.bench_lengths("c4")
    idx = parallel.shard_indices(lens)
    mine = [sample_long(m, lens[i], seed=200 + 7 * i) for i in idx]
    hv, _ = make_hmm(m)
    hm, _ = make_hmm(m, algorithm="map")
    for _ in range(2):
        hv.decode_batch(mine); hm.decode_batch(mine)
    best = None
    for _ in range(3):
        barrier(); t0 = time.perf_counter()
        hv.decode_batch(mine)
        hm.decode_batch(mine)
        torch.cuda.synchronize()
        dt = reduce(time.perf_counter() - t0, MAX)
        best = dt if best is None else min(best, dt)
    # the same two paths from ONE call (one upload, one emission pass): MultitrackHmm.decode_both_batch
    hv.decode_both_batch(mine)
    best_both = None
    for _ in range(3):
        barrier(); t0 = time.perf_counter()
        hv.decode_both_batch(mine)
        torch.cuda.synchronize()
        dt = reduce(time.perf_counter() - t0, MAX)
        best_both = dt if best_both is None else min(best_both, dt)
    out["c4_decode"] = {"what": "hg19-scale decode (24 sequences, %d bins), Viterbi + MAP through decode_batch with host "
                                "buffers, sequences dealt to %d rank(s); no collective" % (sum(lens), world),
                        "seconds": best, "cells_per_s": sum(lens) * N_STATES / best,
                        "seconds_decode_both_batch": best_both, "cells_per_s_decode_both_batch": sum(lens) * N_STATES / best_both,
                        "largest_shard_steps": int(reduce(sum(lens[i] for i in idx), MAX))}
    del mine
    # ---- config 3: Baum-Welch iterations, sequences sharded, one all-reduce per iteration
    lens = synth.bench_lengths("c3")
    own = set(parallel.shard_indices(lens))
    seqs = [synth.sample_obs(m, n, seed=100 + i)[0] if i in own else np.zeros((n, m["K"]), dtype=np.uint8)
            for i, n in enumerate(lens)]
    m0 = synth.make_model(N=N_STATES, seed=7, zero_frac=0.0)
    hmm, _ = make_hmm(m0, n_iter=2, thresh=0.0)
    hmm.fit(seqs)                       # warm-up (allocator, kernels, NCCL)
    n_iter = 50                         # BASELINE.json configs[2]: 50 EM iterations (the one-time upload of the shard is part of the fit)
    hmm, _ = make_hmm(m0, n_iter=n_iter, thresh=0.0)
    barrier(); t0 = time.perf_counter()
    hmm.fit(seqs)
    torch.cuda.synchronize()
    dt = reduce(time.perf_counter() - t0, MAX)
    out["c3_em"] = {"what": "Baum-Welch on 350 sequences (%d steps) through MultitrackHmm.fit, %d iterations, sequences "
                            "dealt to %d rank(s), one all-reduce + host M-step per iteration" % (sum(lens), n_iter, world),
                    "seconds_per_em_iteration": dt / n_iter, "cells_per_s_per_iteration": sum(lens) * N_STATES / (dt / n_iter)}
    # the same with SEGMENT RATIOS (segmentTracks-style tables: one observation per variable-length segment,
    # ratio = length / 100; _hmm.pyx:140-149,187-188): the ratios are folded into the emission lattice once
    # (tehmm_fold_ratios) and the passes run on the tile kernels
    from tehmm_b200.track import IntegerTrackTable
    rng = np.random.RandomState(3)
    tables = []
    for o in seqs:
        seg = np.minimum(rng.geometric(1.0 / 60.0, size=o.shape[0]), 100).astype(np.int64)
        t = IntegerTrackTable(o.shape[1], "chrG", 0, int(seg.sum()))
        t.segOffsets = np.concatenate([[0], np.cumsum(seg)[:-1]]).astype(np.int64)
        t.data = o
        t.shape = (len(t), o.shape[1])
        tables.append(t)
    hmm, _ = make_hmm(m0, seg_len=100, n_iter=2, thresh=0.0)
    hmm.fit(tables)
    hmm, _ = make_hmm(m0, seg_len=100, n_iter=n_iter, thresh=0.0)
    barrier(); t0 = time.perf_counter()
    hmm.fit(tables)
    torch.cuda.synchronize()
    dt_r = reduce(time.perf_counter() - t0, MAX)
    out["c3_em_with_segment_ratios"] = {"seconds_per_em_iteration": dt_r / n_iter,
                                        "relative_to_without_ratios": dt_r / dt}
    return out


# ------------------------------------------------------------------ our arm
DUMP_SAMPLE = 2_000_000      # state-path entries per dumped path: the dump stays near 32 MB at any --T


def dump_outputs(path, out):
    """What one sweep returns to its caller -- log-likelihood, MAP score and Viterbi log-probability
    (float64) and the two state paths (float32) -- as DIR/<name>.npy.  Paths longer than DUMP_SAMPLE
    are sampled at positions drawn with a fixed seed; state_index holds the positions."""
    import torch
    logprob, mscore, vlp, states, mstates = out
    T = states.numel()
    idx = np.arange(T) if T <= DUMP_SAMPLE else np.sort(np.random.RandomState(0).choice(T, DUMP_SAMPLE, replace=False))
    d_idx = torch.from_numpy(idx).to(states.device)
    arrays = {"logprob": logprob.cpu().numpy(), "map_score": mscore.cpu().numpy(), "viterbi_logprob": vlp.cpu().numpy(),
              "viterbi_states": states[d_idx].cpu().numpy().astype(np.float32),
              "map_states": mstates[d_idx].cpu().numpy().astype(np.float32),
              "state_index": idx.astype(np.float64)}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from tehmm_b200 import _lib, synth
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    from tehmm_b200.engine import Engine
    from tehmm_b200.hmm import MultitrackHmm

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    T = args.T
    # one process per GPU shares the host's cores: the host side of the e2e path (widening the
    # state paths to int64) must not oversubscribe them
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // max(1, world)))
    os.environ.setdefault("TEHMM_HOST_THREADS", str(max(1, min(16, (os.cpu_count() or 1) // max(1, world)))))

    m = synth.make_model(N=N_STATES, seed=0)
    obs, _ = synth.sample_obs(m, T, seed=1 + rank)
    obs_pinned = torch.from_numpy(obs).pin_memory()

    ctx = _lib.get_context(local)
    eng = Engine(ctx)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    d_obs = obs_pinned.to(dev, non_blocking=True).reshape(-1)
    eng.use_device_batch(d_obs, 1, np.array([0, T], dtype=np.int64))
    prec, tdt = eng._prec(args.precision)
    stage_names = ["emission", "forward", "backward_map", "viterbi_dp_traceback"]

    def sweep(events=None):
        def mark(i):
            if events is not None:
                events[i].record()
        mark(0)
        elog, blin, rowmax = eng.run_emission(prec, tdt, None, True, True)
        mark(1)
        alpha, logprob = eng.run_forward(prec, tdt, blin, rowmax, None)
        mark(2)
        _, mstates, mscore = eng.run_backward(prec, tdt, _lib.BWD_MAP, blin, alpha, None)
        mark(3)
        states, _, vlp = eng.run_viterbi(prec, elog, None, None, want64=False, rowmax=rowmax)
        mark(4)
        return logprob, mscore, vlp, states, mstates

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # deferred verification (tehmm_ctx_check): the stages of a sweep are queued back to back and the
    # repair counts are read once per sweep, inside the timed region (a failed check re-runs the sweep
    # with the synchronous verify / repair loop; sanity.deferred_bad counts those)
    plain_sweep = sweep

    def sweep(events=None):
        return ctx.optimistic(lambda: plain_sweep(events))

    for _ in range(args.warmup):
        out = sweep()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launches
    ctx.set_option("timing", 1)          # per-kernel CUDA events, read after the timed region
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(args.steps)]
    barrier()
    for k in range(args.steps):
        out = sweep(evs[k])
    barrier()
    launches = ctx.launches - launches0
    stage_ms = np.zeros(4)
    total_ms = 0.0
    for k in range(args.steps):
        for i in range(4):
            stage_ms[i] += evs[k][i].elapsed_time(evs[k][i + 1])
        total_ms += evs[k][0].elapsed_time(evs[k][4])
    # whole timed region incl. gaps between steps
    region_ms = evs[0][0].elapsed_time(evs[-1][4])
    t_max = torch.tensor([region_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
    region_ms = float(t_max.item())
    cells = float(world) * T * N_STATES * args.steps
    value = cells / (region_ms * 1e-3)
    logprob, mscore, vlp, states, mstates = out
    sanity = {"logprob": float(logprob[0].item()), "viterbi_logprob": float(vlp[0].item()),
              "map_score": float(mscore[0].item()),
              "repairs": {k: ctx.stat("repaired_chunks_" + k) for k in ("forward", "backward", "viterbi")},
              "chunks": ctx.stat("chunks"), "deferred_checks": ctx.stat("deferred_checks"),
              "deferred_bad": ctx.stat("deferred_bad")}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)

    # ---- roofline of the dominant KERNEL: its own duration from CUDA events the library records
    # around it on the launching stream during the timed region (mean over the K steps), against
    # its algorithmic bytes (SURVEY.md section 8d per-step figures split per kernel; DESIGN.md section 5)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    K = m["K"]
    kern_us = {k: ctx.stat("us_" + k) for k in ("emission", "forward", "backward", "viterbi_dp", "traceback", "rescore")}
    ctx.set_option("timing", 0)
    # algorithmic bytes per time step of each kernel: symbols in, compulsory fp32 lattice spill, states out
    alg_bytes = {"emission": K, "forward": K + 4 * N_STATES, "backward": K + 4 * N_STATES + 1,
                 "viterbi_dp": K + N_STATES, "traceback": 2, "rescore": 0}
    # DRAM bytes per launch: `ncu --set full` capture of this command (dram__bytes_read.sum +
    # dram__bytes_write.sum per kernel), 10 M x 30 x 10 only; the stamp says which capture
    traffic_src = os.path.join(ROOT, "profiles", "r02_sweep_traffic.json")
    ncu_traffic, traffic_stamp = None, None
    if os.path.exists(traffic_src) and T == T_DEFAULT and args.precision == "f32":
        tj = json.load(open(traffic_src))
        ncu_traffic, traffic_stamp = tj["bytes_per_launch"], {"file": "profiles/r02_sweep_traffic.json", "commit": tj.get("commit"),
                                                              "capture": tj.get("capture")}
    # the dominant kernel is the longest one, whatever it moves; the headline fraction is the whole
    # sweep's (its 303 algorithmic bytes per step over the time of ALL its kernels)
    dom = max(kern_us, key=lambda k: kern_us[k])
    dom_s = kern_us[dom] * 1e-6
    sweep_s = total_ms / args.steps * 1e-3
    sweep_alg = 3 * K + 9 * N_STATES + 3
    sweep_achieved = sweep_alg * T / sweep_s / 1e9
    traffic_total = float(sum(ncu_traffic.get(k, 0.0) for k in kern_us)) if ncu_traffic else None
    traffic_gbs = traffic_total / sweep_s / 1e9 if ncu_traffic else None
    vit_stage_us = kern_us["viterbi_dp"] + kern_us["traceback"] + max(kern_us["rescore"], 0)
    roofline = {"bound": "hbm", "scope": "whole sweep: every kernel of one step", "achieved": sweep_achieved, "peak": peak,
                "unit": "GB/s", "frac": sweep_achieved / peak, "traffic": traffic_total, "traffic_source": traffic_stamp,
                "peak_source": peak_src, "algorithmic_bytes_per_step": sweep_alg,
                "dram_gbs": traffic_gbs, "dram_frac": traffic_gbs / peak if traffic_gbs else None,
                "kernel": dom, "kernel_choice": "longest kernel of the step by its own CUDA-event time, no tie-break",
                "dominant_kernel": {"name": dom, "us": kern_us[dom], "algorithmic_bytes_per_step": alg_bytes[dom],
                                    "achieved": alg_bytes[dom] * T / dom_s / 1e9, "frac": alg_bytes[dom] * T / dom_s / 1e9 / peak,
                                    "traffic": ncu_traffic.get(dom) if ncu_traffic else None},
                "dominant_stage": {"name": "viterbi (DP + traceback + score)", "us": vit_stage_us,
                                   "algorithmic_bytes_per_step": K + N_STATES + 2,
                                   "frac": (K + N_STATES + 2) * T / (vit_stage_us * 1e-6) / 1e9 / peak},
                "kernel_us": kern_us,
                "kernel_frac": {k: (alg_bytes[k] * T / (v * 1e-6) / 1e9 / peak if v > 0 else None) for k, v in kern_us.items()},
                "kernel_dram_frac": ({k: (ncu_traffic.get(k, 0.0) / (v * 1e-6) / 1e9 / peak if v > 0 else None)
                                      for k, v in kern_us.items()} if ncu_traffic else None),
                "issue_bound_note": "the sweep is bound by fp32 instruction issue, not HBM (DESIGN.md section 5, "
                                    "profiles/r02_notes_sidecar.md): exact fp32 (max,+) at 30 states alone needs 0.56 ms per 10 M steps",
                "stage_ms_per_step": {n: float(v / args.steps) for n, v in zip(stage_names, stage_ms)}}

    # ---- end to end through the public API, host buffers in and out
    e2e = None
    if not args.no_e2e:
        em = IndependentMultinomialEmissionModel(N_STATES, list(m["syms"]), zeroAsMissingData=True)
        em.logProbs = m["table"].copy()
        hmm_v = MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy())
        hmm_m = MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy(), algorithm="map")
        host_obs = obs_pinned.numpy()
        n_e2e = max(1, args.steps)
        def timed(fn):
            for _ in range(max(3, args.warmup)):     # results held like in the timed loop (host result pool warm)
                r = fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                r = fn()
            barrier()
            tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()), r
        # the sweep in ONE call (one upload, one emission pass, both decodings): the reference arm shares
        # its frame between the two decodings in the same way (cpu_sweep_reference)
        dt, rb = timed(lambda: hmm_v.decode_both_batch([host_obs]))
        # and as the two calls the reference API spells it with
        dt2, (rv, rm) = timed(lambda: (hmm_v.decode_batch([host_obs]), hmm_m.decode_batch([host_obs])))
        assert np.array_equal(rb[0][1], rv[0][1]) and np.array_equal(rb[0][3], rm[0][1])
        e2e = {"value": float(world) * T * N_STATES * n_e2e / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(host_obs.nbytes), "d2h_bytes_per_step": int(2 * T + 32),
               "steps": n_e2e, "ms_per_step": 1e3 * dt / n_e2e,
               "api": "MultitrackHmm.decode_both_batch -> tehmm_decode_host_both: NumPy uint8 in (pinned), Viterbi and MAP "
                      "int64 paths out (uint8 states over PCIe, widened by %s host threads)" % os.environ["TEHMM_HOST_THREADS"],
               "two_calls": {"value": float(world) * T * N_STATES * n_e2e / dt2, "ms_per_step": 1e3 * dt2 / n_e2e,
                             "h2d_bytes_per_step": int(2 * host_obs.nbytes),
                             "api": "MultitrackHmm.decode_batch (viterbi) + MultitrackHmm(algorithm='map').decode_batch"}}
        assert rv[0][1].dtype == np.int64 and rv[0][1].shape[0] == T
        # where an end-to-end call spends its time: one more pair of calls, traced (a stream synchronisation
        # per phase, so the phases add up to more than a timed call, whose copies overlap the kernels)
        os.environ["TEHMM_HOST_TRACE"] = "2"
        try:
            br = {}
            for name, h in (("viterbi", hmm_v), ("map", hmm_m)):
                h.decode_batch([host_obs])
                br[name] = {k: float(ctx.lib.tehmm_decode_host_phase_ms(ctx.handle, i))
                            for i, k in enumerate(("set_batch", "h2d_and_emission", "trellis", "d2h_and_widen"))}
            e2e["breakdown_ms_traced"] = br
        finally:
            del os.environ["TEHMM_HOST_TRACE"]

    # ---- seconds per EM iteration (second half of the BASELINE metric)
    em_iter = None
    if not args.no_em:
        eng.use_device_batch(d_obs, 1, np.array([0, T], dtype=np.int64))
        eng.estep(device_result=True)
        barrier()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        n_em = 2
        for _ in range(n_em):
            packed = eng.estep(device_result=True)
            if world > 1:
                dist.all_reduce(packed)
        b_.record()
        barrier()
        em_iter = {"seconds": a.elapsed_time(b_) * 1e-3 / n_em, "obs_per_gpu": T,
                   "what": "emission+forward+backward(xi,posteriors)+histograms+allreduce, device resident"}

    # ---- what speculation costs where filters forget slowly (VERDICT r1 item 4): all-missing stretches of
    # 2 000 - 20 000 steps under the bench model and under a near-reducible matrix (diagonal 0.9999)
    if rank == 0 and not args.no_em:
        hard = {}
        Th = 2_000_000
        for name, sticky in (("bench_model_with_gaps", 0.9), ("diag_0.9999_with_gaps", 0.9999)):
            mh = synth.make_model(N=N_STATES, seed=0, sticky=sticky)
            oh, _ = synth.sample_obs(mh, Th, seed=1)
            oh, _ = synth.add_missing_stretches(oh)
            eng.upload_model(mh["log_start"], mh["log_trans"], mh["table"], 1.0, mh["widths"])
            eng.upload_batch([oh])
            keys = ("repair_passes_forward", "repair_passes_backward", "repair_passes_viterbi", "repair_passes_traceback", "fallbacks")
            for _ in range(2):
                s0 = {k: ctx.stat(k) for k in keys}
                torch.cuda.synchronize(); t0 = time.perf_counter()
                eng.posteriors(renorm_eps=True, want_post=False, want_map=True)
                torch.cuda.synchronize(); t1 = time.perf_counter()
                eng.viterbi()
                torch.cuda.synchronize(); t2 = time.perf_counter()
            hard[name] = dict({k: ctx.stat(k) - v for k, v in s0.items()}, obs=Th, warmup=ctx.stat("warmup"),
                              fwd_bwd_map_ms=1e3 * (t1 - t0), viterbi_ms=1e3 * (t2 - t1), mix_rho=ctx.stat("mix_rho_ppm") * 1e-6)
        sanity["slow_mixing"] = hard
        eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])

    split = None
    if not args.no_split:
        split = run_split(world, rank)

    # the sampler ran through the sweep, the end-to-end loop, the EM iterations and the split runs
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "all timed regions of this run (sweep, e2e, em_iter, split)"

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        kind = cpu_kind()
        Ts = args.cpu_sample
        t0 = time.perf_counter()
        lp_cpu, st_cpu, mp_cpu = cpu_sweep(kind, m, obs[:Ts])
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": Ts * N_STATES / dt, "unit": UNIT, "cores": 1, "kind": kind,
                        "sample": "first %d observations of the rank-0 sequence, single thread, %.1f s" % (Ts, dt)}
        # the CPU run doubles as a parity spot check of the production path on the real workload
        eng.upload_batch([obs[:Ts]])
        lps, sts = eng.viterbi(precision=args.precision)
        cpu_baseline["viterbi_path_agreement"] = float(np.mean(sts[0] == st_cpu))
        cpu_baseline["viterbi_logprob_rel_err"] = float(abs(lps[0] - lp_cpu) / abs(lp_cpu))

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": region_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
                "config": workload_config(T, world), "clocks": clocks, "e2e": e2e,
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
                "em_iter": em_iter, "split": split, "sanity": sanity}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
