"""-m gpu: the drop-in claim (INTEGRATION.md Level 0), proven on the reference's OWN classes.

The unmodified reference built under oracle/_ref (oracle/build_ref.py) imports its kernels at
/root/reference/hmm.py:57 (`from . import _hmm`) and /root/reference/emission.py:19
(`from ._emission import canFast, fastAllLogProbs, fastAccumulateStats, fastUpdateCounts`).
These tests rebind exactly those names to tehmm_b200._hmm / tehmm_b200._emission and run the
reference's own MultitrackHmm.fit / decode / score / score_samples / supervisedTrain /
viterbi / posteriorDecode and the statesToBed loop of bin/teHmmEval.py:238-262 -- first on the
untouched reference (Cython on the CPU), then with our CUDA kernels underneath -- and compare:
bit-exact where the strict kernels are bit-exact (emission frames, Viterbi paths and scores,
supervised counts, emission histograms given the same posteriors), <= 1e-10 otherwise
(forward / backward / lneta use libdevice exp / log instead of glibc's).
"""
import contextlib
import io
import os
import sys
import types

import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from conftest import ROOT, golden

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "oracle"))


@pytest.fixture(scope="module")
def R():
    import ref_loader
    if not ref_loader.available():
        pytest.skip("needs the original teHmm's own classes, which the repository does not ship: build them "
                    "into oracle/_ref with oracle/build_ref.py (TEHMM_REFERENCE = the teHmm source directory)")
    return ref_loader.load()


@contextlib.contextmanager
def cuda_kernels(R):
    """what a maintainer's two-line patch does (INTEGRATION.md): the reference's classes on our kernels"""
    from tehmm_b200 import _emission as our_em
    from tehmm_b200 import _hmm as our_hmm
    names = ("canFast", "fastAllLogProbs", "fastAccumulateStats", "fastUpdateCounts")
    saved = (R.hmm._hmm, {n: getattr(R.emission, n) for n in names})
    calls = {"n": 0}

    def counted(fn):
        def wrapper(*a, **k):
            calls["n"] += 1
            return fn(*a, **k)
        wrapper.__name__ = fn.__name__
        return wrapper

    shim = types.SimpleNamespace(**{n: counted(getattr(our_hmm, n))
                                    for n in ("_forward", "_backward", "_viterbi", "_log_sum_lneta")})
    R.hmm._hmm = shim
    for n in names:
        setattr(R.emission, n, getattr(our_em, n) if n == "canFast" else counted(getattr(our_em, n)))
    try:
        yield calls
    finally:
        R.hmm._hmm = saved[0]
        for n, f in saved[1].items():
            setattr(R.emission, n, f)


def ref_table(R, obs, seg_lens=None):
    T, K = obs.shape
    if seg_lens is None:
        tab = R.track.IntegerTrackTable(K, "chrG", 0, T, dtype=obs.dtype)
        tab.data[:] = obs
        return tab
    tab = R.track.IntegerTrackTable(K, "chrG", 0, int(np.sum(seg_lens)), dtype=obs.dtype)
    tab.segOffsets = np.concatenate([[0], np.cumsum(seg_lens)[:-1]]).astype(np.int64)
    tab.data = obs.copy()
    tab.shape = (len(tab), K)
    return tab


def build_fit_model(R, g):
    N, syms = int(g["N"]), [int(s) for s in g["syms"]]
    seg = int(g["seg"]) == 1
    em = R.emission.IndependentMultinomialEmissionModel(
        N, syms, zeroAsMissingData=True, fudge=0.0, effectiveSegmentLength=100 if seg else None)
    em.logProbs = g["init_table"].copy()
    hmm = R.hmm.MultitrackHmm(em, startprob=g["init_pi"].copy(), transmat=g["init_A"].copy(),
                              n_iter=int(g["n_iter"]), thresh=0.0, fixStart=False, transMatEpsilons=True)
    tables = [ref_table(R, g["obs_%d" % i], g["seglens_%d" % i] if seg else None)
              for i in range(int(g["nseq"]))]
    return hmm, em, tables


def run_flow(R, g):
    hmm, em, tables = build_fit_model(R, g)
    hmm.fit(tables)
    out = dict(transmat=hmm.transmat_.copy(), startprob=hmm.startprob_.copy(), table=em.getLogProbs().copy(),
               last=hmm.getLastLogProb(), iters=hmm.current_iteration, dec=[], ss=[], score=[], frames=[])
    # decode with the golden (untouched-reference) parameters so that both runs decode the same model
    hmm._log_transmat = g["fit_log_trans"].copy()
    hmm._log_startprob = g["fit_log_start"].copy()
    em.logProbs = g["fit_table"].copy()
    for tab in tables:
        out["dec"].append(hmm.decode(tab))
        out["ss"].append(hmm.score_samples(tab))
        out["score"].append(hmm.score(tab))
        out["frames"].append(hmm._compute_log_likelihood(tab))
    td = types.SimpleNamespace(getTrackTableList=lambda: tables, getTrackList=lambda: None)
    out["viterbi"] = hmm.viterbi(td)
    out["postdecode"] = hmm.posteriorDecode(td)
    return out


@pytest.mark.parametrize("name", ["fit_n4_k3", "fit_n30_k10", "fit_n5_k2_seg"])
def test_reference_classes_run_on_our_kernels(R, name):
    g = golden(name)
    cpu = run_flow(R, g)                          # untouched reference, Cython on the CPU
    with cuda_kernels(R) as calls:
        gpu = run_flow(R, g)                      # the same classes, tehmm_b200 kernels underneath
    assert calls["n"] > 10 * int(g["nseq"])       # the rebinding really carried the work
    # the untouched run reproduces the committed golden vectors (generated by the same code)
    assert_array_equal(cpu["transmat"], g["fit_transmat"])
    assert gpu["iters"] == cpu["iters"] == int(g["fit_iterations"])
    assert gpu["last"] == pytest.approx(cpu["last"], rel=1e-10)
    assert_allclose(gpu["transmat"], cpu["transmat"], rtol=1e-10, atol=1e-300)
    assert_allclose(gpu["startprob"], cpu["startprob"], rtol=1e-10, atol=1e-300)
    assert_allclose(np.exp(gpu["table"]), np.exp(cpu["table"]), rtol=1e-10, atol=1e-300)
    for i in range(int(g["nseq"])):
        assert_array_equal(gpu["frames"][i], cpu["frames"][i])                 # bit-exact gather-sum
        assert gpu["dec"][i][0] == cpu["dec"][i][0] == float(g["vit_logprob_%d" % i])   # bit-exact Viterbi
        assert_array_equal(gpu["dec"][i][1], cpu["dec"][i][1])
        assert gpu["dec"][i][1].dtype == cpu["dec"][i][1].dtype
        assert gpu["score"][i] == pytest.approx(cpu["score"][i], rel=1e-10)
        assert gpu["ss"][i][0] == pytest.approx(cpu["ss"][i][0], rel=1e-10)
        assert_allclose(gpu["ss"][i][1], cpu["ss"][i][1], rtol=1e-9, atol=1e-12)
        for key in ("viterbi", "postdecode"):
            assert gpu[key][i][0] == cpu[key][i][0]
            assert_array_equal(np.asarray(list(gpu[key][i][1])), np.asarray(list(cpu[key][i][1])))


def test_hmmtest_vectors_on_reference_classes(R):
    """tests/hmmTest.py:48-135,147-151 (Wikipedia rainy/sunny) through the reference's classes
    with our kernels rebound: exp(logprob) = 0.01344, path [1,0,0], the posterior KAT."""
    g = golden("wikipedia")
    with cuda_kernels(R) as calls:
        em = R.emission.IndependentMultinomialEmissionModel(
            2, [3], [[[0.1, 0.4, 0.5], [0.6, 0.3, 0.1]]], zeroAsMissingData=False)
        hmm = R.hmm.MultitrackHmm(em, startprob=[0.6, 0.4], transmat=[[0.7, 0.3], [0.4, 0.6]])
        obs = np.asarray([[0], [1], [2]], dtype=np.uint8)
        lp, st = hmm.decode(obs)
        sc, post = hmm.score_samples(obs)
        assert calls["n"] >= 5
    assert np.exp(lp) == pytest.approx(0.01344, rel=1e-12)
    assert_array_equal(st, [1, 0, 0])
    assert sc == pytest.approx(float(g["v1_score"]), rel=1e-12)
    assert_allclose(post, g["v1_post"], rtol=1e-10)
    assert_allclose(post, [[0.23170303, 0.76829697], [0.62406281, 0.37593719], [0.86397706, 0.13602294]],
                    atol=5e-9)


def test_supervised_train_on_reference_classes(R):
    """hmm.py:174-210 + emission.py:293-331 (-> fastUpdateCounts per interval): integer counts,
    so transition / start / emission parameters must be BIT-identical with our kernel."""
    rng = np.random.RandomState(5)
    N, syms, T = 4, [3, 7, 2], 600
    obs = np.stack([rng.randint(0, s + 1, size=T) for s in syms], axis=1).astype(np.uint8)
    cuts = [0, 50, 60, 150, 151, 300, 420, 600]
    states = [0, 1, 2, 3, 0, 2, 1]
    intervals = [("chrG", cuts[i], cuts[i + 1], states[i]) for i in range(len(states))]

    def flow():
        tabs = [ref_table(R, obs)]
        td = types.SimpleNamespace(getTrackTableList=lambda: tabs, getTrackList=lambda: None)
        em = R.emission.IndependentMultinomialEmissionModel(N, syms, zeroAsMissingData=True)
        hmm = R.hmm.MultitrackHmm(em)
        hmm.supervisedTrain(td, intervals)
        lp, st = hmm.decode(tabs[0])
        return hmm.transmat_.copy(), hmm.startprob_.copy(), em.getLogProbs().copy(), lp, st

    cpu = flow()
    with cuda_kernels(R) as calls:
        gpu = flow()
        assert calls["n"] >= len(intervals)
    for a, b in zip(gpu[:3], cpu[:3]):
        assert_array_equal(a, b)
    assert gpu[3] == cpu[3]
    assert_array_equal(gpu[4], cpu[4])


def reference_states_to_bed(trackTable, states):
    """the bedFile branch of /root/reference/bin/teHmmEval.py:238-262, statement for statement, on the
    reference's own TrackTable methods (the script itself is Python 2 -- `print` statements at :206 --
    and cannot be imported)"""
    buf = io.StringIO()
    chrom = trackTable.getChrom()
    start = trackTable.getStart()
    end = trackTable.getEnd()
    segOffsets = trackTable.getSegmentOffsets()
    maskOffsets = trackTable.getMaskRunningOffsets()
    if segOffsets is None:
        assert len(states) == end - start
    segDist = 0
    for i in range(len(states)):
        curStart = start + segDist
        intLen = 1
        if segOffsets is not None:
            intLen = trackTable.getSegmentLength(i)
        segDist += intLen
        if maskOffsets is not None:
            curStart += maskOffsets[curStart - trackTable.getStart()]
        curEnd = curStart + intLen
        buf.write("%s\t%d\t%d\t%s\n" % (chrom, curStart, curEnd, states[i]))
    return buf.getvalue()


def test_states_to_bed_on_real_decode_output(R, tmp_path):
    """teHmmEval.py:193-204: model.viterbi(trackData) then statesToBed per table, with the decode
    coming from the reference's class on our kernels and the writer being tehmm_b200.output."""
    from tehmm_b200 import output
    g = golden("fit_n5_k2_seg")
    hmm, em, tables = build_fit_model(R, g)
    hmm._log_transmat = g["fit_log_trans"].copy()
    hmm._log_startprob = g["fit_log_start"].copy()
    em.logProbs = g["fit_table"].copy()
    td = types.SimpleNamespace(getTrackTableList=lambda: tables, getTrackList=lambda: None)
    with cuda_kernels(R):
        vit = hmm.viterbi(td)
    path = tmp_path / "out.bed"
    with open(path, "w") as f:
        for (prob, states), tab in zip(vit, tables):
            output.statesToBed(tab, np.asarray(list(states)), f)
    want = "".join(reference_states_to_bed(tab, np.asarray(list(states))) for (prob, states), tab in zip(vit, tables))
    assert open(path).read() == want
    assert want.count("\n") == sum(len(t) for t in tables)
