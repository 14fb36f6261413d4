#!/usr/bin/env python
"""Generate golden input/output vectors from the REAL reference (teHmm).

Run in the build container only (needs oracle/_ref, built from /root/reference
by oracle/build_ref.py):

    python oracle/build_ref.py && python tests/golden/make_golden.py

Every case stores its inputs AND the reference's outputs in one .npz under
tests/golden/, so the tests never need /root/reference.  Outputs come from the
reference's own Cython modules (_hmm, _emission) and its own Python classes
(hmm.MultitrackHmm, basehmm.MultinomialHMM, emission.IndependentMultinomial-
EmissionModel) -- not from the oracle port.
"""
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_loader  # noqa: E402

R = ref_loader.load()
LOGZERO = R.common.LOGZERO


def rand_model(rng, N, syms, zero_frac=0.2, sticky=0.9):
    """Dirichlet transition rows with a sticky diagonal and exact zeros,
    Dirichlet(0.5) emissions per (track, state).  Returns probabilities."""
    A = rng.dirichlet(np.ones(N), size=N)
    A = sticky * np.eye(N) + (1 - sticky) * A
    if N > 2 and zero_frac > 0:
        mask = rng.rand(N, N) < zero_frac
        np.fill_diagonal(mask, False)
        A[mask] = 0.0
    A /= A.sum(axis=1, keepdims=True)
    pi = rng.dirichlet(np.ones(N))
    em = [[rng.dirichlet(0.5 * np.ones(s)).tolist() for _ in range(N)] for s in syms]
    return pi, A, em


def rand_obs(rng, T, syms, dtype, missing=0.05):
    cols = []
    for s in syms:
        c = rng.randint(1, s + 1, size=T)
        # run-length structure
        keep = rng.rand(T) < 0.7
        for t in range(1, T):
            if keep[t]:
                c[t] = c[t - 1]
        c[rng.rand(T) < missing] = 0
        cols.append(c)
    return np.ascontiguousarray(np.stack(cols, axis=1).astype(dtype))


class FakeTable(R.track.IntegerTrackTable):
    """IntegerTrackTable carrying segment offsets without going through bedtools."""
    pass


def make_table(obs, seg_lens=None):
    T, K = obs.shape
    if seg_lens is None:
        tab = R.track.IntegerTrackTable(K, "chrG", 0, T, dtype=obs.dtype)
        tab.data[:] = obs
        return tab
    total = int(np.sum(seg_lens))
    tab = R.track.IntegerTrackTable(K, "chrG", 0, total, dtype=obs.dtype)
    tab.segOffsets = np.concatenate([[0], np.cumsum(seg_lens)[:-1]]).astype(np.int64)
    tab.data = obs.copy()
    tab.shape = (len(tab), K)
    return tab


def low_level_case(name, seed, N, syms, T, dtype, with_ratio, zero_frac=0.2, normalize_fac=0.0):
    rng = np.random.RandomState(seed)
    pi, A, em = rand_model(rng, N, syms, zero_frac)
    K = len(syms)
    emission = R.emission.IndependentMultinomialEmissionModel(
        N, list(syms), em, zeroAsMissingData=True, normalizeFac=normalize_fac)
    table = emission.getLogProbs().copy()
    obs = rand_obs(rng, T, syms, dtype)
    ratios = rng.uniform(0.01, 10.0, size=T) if with_ratio else None
    log_start = R.common.myLog(pi).astype(np.float64)
    log_trans = R.common.myLog(A).astype(np.float64)

    frame = np.zeros((T, N))
    R._emission.fastAllLogProbs(obs, table, frame, emission.normalizeFac, ratios)
    fwd = np.zeros((T, N))
    R._hmm._forward(T, N, log_start, log_trans, frame, ratios, fwd)
    bwd = np.zeros((T, N))
    R._hmm._backward(T, N, log_start, log_trans, frame, ratios, bwd)
    states, vlp = R._hmm._viterbi(T, N, log_start, log_trans, ratios, frame)
    lp = R.basehmm.logsumexp(fwd[-1])
    gamma = fwd + bwd
    post = np.exp(gamma.T - R.basehmm.logsumexp(gamma, axis=1)).T
    lneta = np.zeros((N, N))
    if T > 1:
        R._hmm._log_sum_lneta(T, N, fwd, log_trans, bwd, frame, lp, ratios, lneta)
    stats = emission.initStats()
    R._emission.fastAccumulateStats(obs, stats, post, ratios)
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"),
        N=N, K=K, syms=np.array(syms), normalize=emission.normalizeFac,
        pi=pi, A=A, table=table, obs=obs,
        ratios=np.zeros(0) if ratios is None else ratios,
        log_start=log_start, log_trans=log_trans,
        frame=frame, fwd=fwd, bwd=bwd, vit_states=states, vit_logprob=vlp,
        logprob=lp, post=post, lneta=lneta, obs_stats=stats)
    print("%-28s N=%d K=%d T=%d %s ratios=%s  lp=%.6f vit=%.6f" % (
        name, N, K, T, np.dtype(dtype).name, with_ratio, lp, vlp))


def impossible_rows_case():
    """_emission.pyx:59,73-80 quirk: rows are zeroed only before the first
    feasible row (SURVEY.md 8a3 probe: obs [1,0,1] -> [0, -0.69.., -1e100])."""
    N = 2
    table = np.zeros((1, N, 3))
    table[0, :, 1] = LOGZERO          # symbol 1 impossible in both states
    table[0, :, 2] = np.log(0.5)
    cases = {}
    for key, seq in (("a", [1, 0, 1]), ("b", [1, 1, 2, 1]), ("c", [2, 1, 1]), ("d", [1, 1, 1])):
        obs = np.asarray(seq, dtype=np.uint8).reshape(-1, 1)
        out = np.zeros((len(seq), N))
        R._emission.fastAllLogProbs(obs, table, out, 1.0, None)
        cases["obs_" + key] = obs
        cases["out_" + key] = out
    np.savez_compressed(os.path.join(HERE, "impossible_rows.npz"), table=table, **cases)
    print("impossible_rows: a ->", cases["out_a"][:, 0])


def wikipedia_case():
    """tests/hmmTest.py:48-135 and :138-191."""
    emissionprob = [[0.1, 0.4, 0.5], [0.6, 0.3, 0.1]]
    startprob = [0.6, 0.4]
    transmat = [[0.7, 0.3], [0.4, 0.6]]
    h = R.basehmm.MultinomialHMM(2, startprob=startprob, transmat=transmat)
    h.emissionprob_ = emissionprob
    lp_sk, st_sk = h.decode([0, 1, 2])
    post_sk = h.predict_proba([0, 1, 2])
    out = dict(emissionprob=np.array(emissionprob), startprob=np.array(startprob),
               transmat=np.array(transmat), sk_logprob=lp_sk, sk_states=st_sk,
               sk_post=post_sk)
    variants = {
        "v1": ([3], [emissionprob], [[0], [1], [2]]),
        "v3": ([3, 1, 1], [emissionprob, [[1.], [1.]], [[1.], [1.]]],
               [[0, 0, 0], [1, 0, 0], [2, 0, 0]]),
        "v4": ([3, 1, 1, 10],
               [emissionprob, [[1.], [1.]], [[1.], [1.]], [[.1] * 10, [.1] * 10]],
               [[0, 0, 0, 0], [1, 0, 0, 5], [2, 0, 0, 7]]),
    }
    for key, (syms, params, obs) in variants.items():
        em = R.emission.IndependentMultinomialEmissionModel(
            2, syms, params, zeroAsMissingData=False)
        hmm = R.hmm.MultitrackHmm(em, startprob=startprob, transmat=transmat)
        obs = np.asarray(obs)
        lp, st = hmm.decode(obs)
        sc, post = hmm.score_samples(obs)
        out[key + "_table"] = em.getLogProbs()
        out[key + "_obs"] = obs
        out[key + "_vit_logprob"] = lp
        out[key + "_vit_states"] = st
        out[key + "_score"] = sc
        out[key + "_post"] = post
        out[key + "_frame"] = hmm._compute_log_likelihood(obs)
        flp, ftab = hmm._do_forward_pass(out[key + "_frame"])
        out[key + "_fwd"] = ftab
        out[key + "_bwd"] = hmm._do_backward_pass(out[key + "_frame"])
    np.savez_compressed(os.path.join(HERE, "wikipedia.npz"), **out)
    print("wikipedia: exp(logprob)=%.5f states=%s" % (np.exp(lp_sk), st_sk))


def dpbench_case():
    """tests/dpBenchmark.py:90-98 frame generator and :111-155 fb invariant with
    random.seed(200) segRatios, on the default emission model of :55-56."""
    S, T = 10, 400
    frame = np.zeros((T, S))
    for i in range(T):
        for j in range(S):
            frame[i, j] = R.common.myLog(float(j) / float(S))
            frame[i, j] += R.common.myLog((float(i % 9) + 1.) / 10)
    hmm = R.hmm.MultitrackHmm(
        emissionModel=R.emission.IndependentMultinomialEmissionModel(S, [2]))
    flp, ftab = hmm._do_forward_pass(frame)
    btab = hmm._do_backward_pass(frame)
    vlp, vst = hmm._do_viterbi_pass(frame)
    random.seed(200)
    ratios = np.array([random.uniform(0.01, 10.) for _ in range(T)])
    hmm.emissionModel.getSegmentRatios = lambda x: ratios
    sflp, sftab = hmm._do_forward_pass(frame)
    sbtab = hmm._do_backward_pass(frame)
    svlp, svst = hmm._do_viterbi_pass(frame)
    np.savez_compressed(
        os.path.join(HERE, "dpbench.npz"), frame=frame,
        log_start=hmm._log_startprob, log_trans=hmm._log_transmat,
        fwd=ftab, bwd=btab, logprob=flp, vit_logprob=vlp, vit_states=vst,
        ratios=ratios, seg_fwd=sftab, seg_bwd=sbtab, seg_logprob=sflp,
        seg_vit_logprob=svlp, seg_vit_states=svst)
    print("dpbench: lp=%.6f seg lp=%.6f" % (flp, sflp))


def fit_case(name, seed, N, syms, lens, n_iter, seg=False, dtype=np.uint8):
    """Whole-class parity: MultitrackHmm.fit / decode / score_samples / score."""
    rng = np.random.RandomState(seed)
    pi, A, em = rand_model(rng, N, syms, zero_frac=0.0)
    K = len(syms)
    obs_list = [rand_obs(rng, T, syms, dtype) for T in lens]
    seg_lens = [rng.randint(1, 400, size=T) if seg else None for T in lens]
    tables = [make_table(o, s) for o, s in zip(obs_list, seg_lens)]
    emission = R.emission.IndependentMultinomialEmissionModel(
        N, list(syms), em, zeroAsMissingData=True, fudge=0.0,
        effectiveSegmentLength=100 if seg else None)
    hmm = R.hmm.MultitrackHmm(emission, startprob=pi.copy(), transmat=A.copy(),
                              n_iter=n_iter, thresh=0.0, fixStart=False,
                              transMatEpsilons=True)
    init_table = emission.getLogProbs().copy()
    init_log_start = hmm._log_startprob.copy()
    init_log_trans = hmm._log_transmat.copy()
    hmm.fit(tables)
    out = dict(N=N, K=K, syms=np.array(syms), n_iter=n_iter, seg=int(seg),
               init_pi=pi, init_A=A, init_table=init_table,
               init_log_start=init_log_start, init_log_trans=init_log_trans,
               fit_startprob=hmm.startprob_, fit_transmat=hmm.transmat_,
               fit_log_start=hmm._log_startprob, fit_log_trans=hmm._log_transmat,
               fit_table=emission.getLogProbs(),
               fit_last_logprob=hmm.getLastLogProb(),
               fit_iterations=hmm.current_iteration)
    for i, (o, s, tab) in enumerate(zip(obs_list, seg_lens, tables)):
        out["obs_%d" % i] = o
        if seg:
            out["seglens_%d" % i] = s
        lp, st = hmm.decode(tab)
        out["vit_logprob_%d" % i] = lp
        out["vit_states_%d" % i] = st
        sc, post = hmm.score_samples(tab)
        out["score_%d" % i] = sc
        out["post_%d" % i] = post
    out["nseq"] = len(lens)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print("%-28s N=%d K=%d lens=%s iters=%d last lp=%.6f" % (
        name, N, K, lens, n_iter, hmm.getLastLogProb()))


def hmmtest_fit_case():
    """tests/hmmTest.py:195-250: fit over the 7 params subsets, MultitrackHmm
    (fast _hmm path) against MultinomialHMM (_basehmm path)."""
    prng = np.random.RandomState(9)
    emissionprob = [[0.1, 0.4, 0.5], [0.6, 0.3, 0.1]]
    h = R.basehmm.MultinomialHMM(2, startprob=[0.6, 0.4],
                                 transmat=[[0.7, 0.3], [0.4, 0.6]], random_state=prng)
    h.emissionprob_ = emissionprob
    train_obs = [h.sample(n=10)[0] for _ in range(10)]
    out = dict(nseq=10)
    for i, o in enumerate(train_obs):
        out["obs_%d" % i] = np.asarray(o)
    for params in ["s", "t", "e", "st", "se", "te", "ste"]:
        init_params = params.replace("e", "")
        em3 = R.emission.IndependentMultinomialEmissionModel(
            2, [3, 1, 1], zeroAsMissingData=False)
        hmm3 = R.hmm.MultitrackHmm(em3, params=params, init_params=init_params)
        hmm3.transmat_ = [[0.5, 0.5], [0.5, 0.5]]
        hmm3.startprob_ = [0.5, 0.5]
        train3 = []
        for o in train_obs:
            o3 = np.zeros((len(o), 3), dtype=np.float64)
            o3[:, 0] = o
            train3.append(o3)
        hmm3.fit(train3)
        out[params + "_transmat"] = hmm3.transmat_
        out[params + "_startprob"] = hmm3.startprob_
        out[params + "_table"] = em3.getLogProbs()
        lp, st = hmm3.decode(train3[0])
        out[params + "_vit_logprob"] = lp
        out[params + "_vit_states"] = st
    np.savez_compressed(os.path.join(HERE, "hmmtest_fit.npz"), **out)
    print("hmmtest_fit: ste transmat =", out["ste_transmat"].round(6).tolist())


def counts_case():
    """_emission.pyx:236-332 supervised counts, incl. ratios."""
    rng = np.random.RandomState(77)
    syms = [3, 7, 2]
    N, T = 4, 200
    obs = rand_obs(rng, T, syms, np.uint8)
    tab = make_table(obs)
    em = R.emission.IndependentMultinomialEmissionModel(N, syms, fudge=1.0)
    stats = em.initStats()
    intervals = [("chrG", 0, 50, 0), ("chrG", 50, 60, 1), ("chrG", 60, 150, 2),
                 ("chrG", 150, 151, 3), ("chrG", 151, 200, 0)]
    for iv in intervals:
        R._emission.fastUpdateCounts(iv, tab, stats, None)
    ratios = rng.uniform(0.5, 3.0, size=T)
    stats_r = em.initStats()
    for iv in intervals:
        R._emission.fastUpdateCounts(iv, tab, stats_r, ratios)
    np.savez_compressed(os.path.join(HERE, "counts.npz"), obs=obs, N=N, syms=np.array(syms),
                        intervals=np.array([[a, b, c] for _, a, b, c in intervals]),
                        stats=stats, ratios=ratios, stats_ratio=stats_r)
    print("counts: total=%.1f" % stats.sum())


def gaussian_case():
    """emission.py:483-615: IndependentMultinomialAndGaussianEmissionModel -- constructor
    (makeGaussian on the initial table), maximize() on posterior-weighted counts, and a user
    `STATE TRACK MEAN STDEV` line.  Track 1 is gaussian over the values 0..11 (scaled category
    map, track.py:668-760), tracks 0 and 2 stay multinomial."""
    rng = np.random.RandomState(31)
    N, syms = 3, [4, 12, 2]
    tracks = []
    for k, ns in enumerate(syms):
        t = R.track.Track(number=k)
        t.name = "t%d" % k
        t.dist = "gaussian" if k == 1 else "multinomial"
        t.valMap = R.track.CategoryMap(reserved=1)
        for v in range(ns):
            t.valMap.update(str(v) if k != 1 else str(float(3 * v)))     # values 0, 3, 6, ... for the gaussian track
        tracks.append(t)
    _, _, params = rand_model(rng, N, syms, zero_frac=0.0)
    em = R.emission.IndependentMultinomialAndGaussianEmissionModel(
        N, list(syms), tracks, params, zeroAsMissingData=True, fudge=0.0)
    out = dict(N=N, syms=np.array(syms), init_params_0=np.array(params[0]), init_params_1=np.array(params[1]),
               init_params_2=np.array(params[2]),
               values_1=np.array([float(tracks[1].valMap.getMapBack(s)) for s in range(1, syms[1] + 1)]),
               table0=em.getLogProbs().copy(), gauss0=em.gaussParams.copy())
    stats = em.initStats()
    T = 500
    obs = rand_obs(rng, T, syms, np.uint8)
    post = rng.dirichlet(np.ones(N), size=T)
    em.accumulateStats(obs, stats, post)
    out["obs"] = obs
    out["post"] = post
    out["stats"] = np.array(stats)
    em.maximize(stats, tracks)
    out["table1"] = em.getLogProbs().copy()
    out["gauss1"] = em.gaussParams.copy()
    logProbs = em.getLogProbs().copy()
    mask = np.zeros(logProbs.shape, dtype=np.int8)
    em.applyUserEmissionLine(tracks[1], 2, ["2", "t1", "7.5", "2.25"], logProbs, mask)
    out["table_user"] = logProbs
    out["mask_user"] = mask
    out["gauss_user"] = em.gaussParams.copy()
    np.savez_compressed(os.path.join(HERE, "gaussian.npz"), **out)
    print("gaussian: mu/sigma state 0 = %s -> %s" % (out["gauss0"][1, 0], out["gauss1"][1, 0]))


def runsum_case():
    """_track.pyx:13-25 on the masks of tests/test_gpu_tracks.py:test_runSum_matches_reference, stored
    as the step from the previous entry (int8, compresses to a few hundred kB at n = 1 000 003).

    The committed runsum.npz was recorded from tehmm_b200._track.runSum at the code of commit edcc791,
    whose test run compared that function bit for bit with this one on these masks and passed."""
    import importlib
    track = importlib.import_module("teHmm._track")
    rng = np.random.RandomState(5)
    out = {}
    for n in (1, 31, 1000, 1_000_003):
        mask = (rng.rand(n) < 0.3).astype(np.uint8)
        s = np.zeros(n, dtype=np.int32)
        track.runSum(mask, s)
        out["steps_%d" % n] = np.diff(s, prepend=0).astype(np.int8)
    np.savez_compressed(os.path.join(HERE, "runsum.npz"), **out)
    print("runsum: last entry %d" % s[-1])


def readbed_case():
    """trackIO.py:67-212 (readBedData, no bedtools call) on the three seeded BED files of
    tests/test_gpu_tracks.py:test_readBedData_matches_reference, with the reference's own CategoryMap /
    BinaryMap: the filled buffer and the size of the value map per case.

    The committed readbed.npz was recorded from tehmm_b200.trackIO.readBedData, with the value maps the
    test restates, at the code of commit edcc791, whose test run compared that function bit for bit
    with this one (the reference's maps on both sides) on these files and passed."""
    import importlib
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_tracks import READBED_CASES, readbed_inputs
    trackIO = importlib.import_module("teHmm.trackIO")
    out = {}
    for case in READBED_CASES:
        tmp = tempfile.mkdtemp()
        path, maps, kw, lo, hi = readbed_inputs(tmp, case, lambda: R.track.CategoryMap(reserved=1), R.track.BinaryMap)
        m = maps()
        buf = np.full(hi - lo, m.getMissingVal(), dtype=np.uint8)
        out["out_" + case] = trackIO.readBedData(path, "chr1", lo, hi, valMap=m, updateValMap=True,
                                                 needIntersect=False, outputBuf=buf, **kw)
        out["nvals_" + case] = len(m)
    np.savez_compressed(os.path.join(HERE, "readbed.npz"), **out)
    print("readbed: value maps of sizes %s" % [int(out["nvals_" + c]) for c in READBED_CASES])


def main():
    if "--only-gaussian" in sys.argv:
        return gaussian_case()
    if "--only-runsum" in sys.argv:
        return runsum_case()
    if "--only-readbed" in sys.argv:
        return readbed_case()
    wikipedia_case()
    impossible_rows_case()
    dpbench_case()
    counts_case()
    hmmtest_fit_case()
    low_level_case("ll_n2_k1_t1", 1, 2, [2], 1, np.uint8, False, zero_frac=0.0)
    low_level_case("ll_n2_k1_t2", 2, 2, [2], 2, np.uint8, False, zero_frac=0.0)
    low_level_case("ll_n3_k2_t17", 3, 3, [2, 3], 17, np.uint8, False)
    low_level_case("ll_n5_k3_t300_u16", 4, 5, [4, 2, 300], 300, np.uint16, False)
    low_level_case("ll_n5_k3_t300_i32", 5, 5, [4, 2, 9], 300, np.int32, False)
    low_level_case("ll_n30_k10_t500", 6, 30, [4, 8, 16, 32, 64, 250, 2, 2, 2, 2], 500,
                   np.uint8, False)
    low_level_case("ll_n30_k10_t500_seg", 7, 30, [4, 8, 16, 32, 64, 250, 2, 2, 2, 2], 500,
                   np.uint8, True)
    low_level_case("ll_n4_k2_t64_seg", 8, 4, [3, 5], 64, np.uint8, True)
    low_level_case("ll_n50_k4_t200", 9, 50, [4, 8, 2, 2], 200, np.uint8, False)
    low_level_case("ll_n33_k2_t90_norm", 10, 33, [6, 3], 90, np.uint8, False, normalize_fac=1.0)
    fit_case("fit_n4_k3", 21, 4, [3, 5, 2], [120, 1, 77, 300], 4)
    fit_case("fit_n30_k10", 22, 30, [4, 8, 16, 32, 64, 250, 2, 2, 2, 2], [400, 250, 90], 3)
    fit_case("fit_n5_k2_seg", 23, 5, [4, 6], [150, 80], 3, seg=True)
    gaussian_case()
    runsum_case()
    readbed_case()


if __name__ == "__main__":
    main()
