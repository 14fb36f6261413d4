"""-m gpu: tehmm_decode_host_ratios / tehmm_decode_host_both_ratios -- the host-buffer decode of
segmented tables (segmentTracks.py, teHmmEval.py --segment).  Reference call being replaced:
basehmm.py:361-396 decode -> hmm.py:668-676, whose Viterbi DP sees the table's segment ratios
(_hmm.pyx:201-259) while the emission (basehmm.py:327) and the MAP decoding (basehmm.py:261-264)
do not.  Each sequence is decoded with its own ratios, or with none.
"""
import ctypes

import numpy as np
import pytest
from numpy.testing import assert_array_equal

from parity import assert_near_ties_only, oracle_all, oracle_frame

pytestmark = pytest.mark.gpu


def _setup(ctx):
    for k in ("chunk_tiles", "warmup", "fine_len"):
        ctx.set_option(k, 0)
    ctx.set_option("tile", 1)


def _engine():
    from tehmm_b200.engine import get_engine
    eng = get_engine(0)
    _setup(eng.ctx)
    return eng


def _ratios(rng, n, cap=300):
    """segment length / 100 with segments of up to `cap` bins: many ratios > 1, most < 1"""
    return np.minimum(rng.geometric(1.0 / 60.0, size=n), cap) / 100.0


def _model(N, seed):
    from tehmm_b200 import synth
    return synth.make_model(N=N, seed=seed)


def _oracle_viterbi(oracle, m, obs, r):
    frame = oracle_frame(oracle, obs, m["table"], 1.0, None)
    st, lp = oracle._viterbi(obs.shape[0], m["N"], m["log_start"], m["log_trans"], r, frame)
    return frame, st, lp


def _segmented_table(obs, seg_lens):
    """an IntegerTrackTable as bin/segmentTracks.py + TrackTable.segment leave it (track.py:449-513)"""
    from tehmm_b200.track import IntegerTrackTable
    t = IntegerTrackTable(obs.shape[1], "chrG", 0, int(seg_lens.sum()))
    t.segOffsets = np.concatenate([[0], np.cumsum(seg_lens)[:-1]]).astype(np.int64)
    t.data = obs.copy()
    t.shape = (len(t), obs.shape[1])
    return t


def _hmm(m, seg_len=100, **kw):
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    from tehmm_b200.hmm import MultitrackHmm
    em = IndependentMultinomialEmissionModel(m["N"], list(m["syms"]), zeroAsMissingData=True, fudge=0.0,
                                             effectiveSegmentLength=seg_len)
    em.logProbs = m["table"].copy()
    return MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy(), **kw), em


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int32])
@pytest.mark.parametrize("N", [2, 30, 50, 64])
def test_float64_matches_the_oracle_with_ratios(oracle, N, dtype):
    """float64 (generic kernels): states identical to the reference's, log-probability to 1e-10"""
    from tehmm_b200 import _lib, synth
    m = _model(N, seed=5)
    lens = [1, 2, 5003, 20000, 777]
    rng = np.random.RandomState(N)
    seqs = [synth.sample_obs(m, n, seed=10 + i)[0].astype(dtype) for i, n in enumerate(lens)]
    ratios = [_ratios(rng, n) for n in lens]
    assert max(r.max() for r in ratios) > 1.5
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    lp, _, states = eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f64", ratios=ratios)
    assert eng.h2d_bytes == sum(lens) * (m["K"] * np.dtype(dtype).itemsize + 8)
    for i, (obs, r) in enumerate(zip(seqs, ratios)):
        _, want, wlp = _oracle_viterbi(oracle, m, obs, r)
        assert states[i].dtype == np.int64 and states[i].shape == (lens[i],)
        assert_array_equal(states[i], want)
        assert lp[i] == pytest.approx(wlp, rel=1e-10)


@pytest.mark.parametrize("N", [30, 50])
def test_float32_near_ties_only(oracle, N):
    from tehmm_b200 import _lib, synth
    m = _model(N, seed=7)
    lens = [1, 2, 40001, 3, 150000]
    rng = np.random.RandomState(11)
    seqs = [synth.sample_obs(m, n, seed=30 + i)[0] for i, n in enumerate(lens)]
    ratios = [_ratios(rng, n) for n in lens]
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    lp, _, states = eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f32", ratios=ratios)
    for i, (obs, r) in enumerate(zip(seqs, ratios)):
        frame, want, wlp = _oracle_viterbi(oracle, m, obs, r)
        assert_near_ties_only(states[i], want, frame, m["log_start"], m["log_trans"], r, label="N%d seq %d" % (N, i))
        assert lp[i] == pytest.approx(wlp, rel=1e-6)


def test_float32_50_states_long_sequence_without_repairs(oracle):
    """the two-warps-per-chunk DP with ratios on one 2 M-step sequence of a bench-like model
    (segments of up to 100 bins, effective length 100): near-ties only, and no chunk needs a repair"""
    from tehmm_b200 import _lib, synth
    m = _model(50, seed=0)
    T = 2_000_000
    obs = synth.sample_obs(m, T, seed=300)[0]
    r = _ratios(np.random.RandomState(3), T, cap=100)
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    rep0, bad0 = eng.ctx.stat("repaired_chunks_viterbi"), eng.ctx.stat("deferred_bad")
    lp, _, states = eng.decode_host([obs], _lib.DECODE_VITERBI, precision="f32", ratios=[r])
    assert eng.ctx.stat("repaired_chunks_viterbi") == rep0 and eng.ctx.stat("deferred_bad") == bad0
    frame, want, wlp = _oracle_viterbi(oracle, m, obs, r)
    assert_near_ties_only(states[0], want, frame, m["log_start"], m["log_trans"], r, label="50 states, 2 M steps")
    assert lp[0] == pytest.approx(wlp, rel=1e-6)


@pytest.mark.parametrize("prec", ["f32", "f64"])
@pytest.mark.parametrize("N", [30, 50])
def test_same_answer_as_the_device_pointer_route(N, prec):
    """every sequence with ratios: bit-identical to upload_batch + Engine.viterbi(ratios_dp=...)"""
    from tehmm_b200 import _lib, synth
    m = _model(N, seed=2)
    lens = [700_001, 5, 90_000]
    rng = np.random.RandomState(5)
    seqs = [synth.sample_obs(m, n, seed=50 + i)[0] for i, n in enumerate(lens)]
    ratios = [_ratios(rng, n) for n in lens]
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(seqs)
    lp_d, st_d = eng.viterbi(ratios_em=None, ratios_dp=ratios, precision=prec)
    lp, _, st = eng.decode_host(seqs, _lib.DECODE_VITERBI, precision=prec, ratios=ratios)
    assert_array_equal(lp, lp_d)
    for a, b in zip(st, st_d):
        assert_array_equal(a, b)


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("N", [30, 50])
def test_mixed_batch_each_sequence_as_the_reference(oracle, N, prec):
    """a segmented table next to a plain array: the plain one gets the reference's segRatios=None
    recursion (not the one at ratio 1.0, which differs through _hmm.pyx:234-237) -- the same states as
    decoding it alone -- and the segmented ones their own ratios"""
    from tehmm_b200 import _lib, engine, synth
    m = _model(N, seed=5)
    rng = np.random.RandomState(9)
    lens = [30000, 20000, 4001]
    obs = [synth.sample_obs(m, n, seed=70 + i)[0] for i, n in enumerate(lens)]
    segs = [np.minimum(rng.geometric(1.0 / 60.0, size=n), 300).astype(np.int64) for n in lens]
    batch = [_segmented_table(obs[0], segs[0]), obs[1], _segmented_table(obs[2], segs[2])]
    # the test means something: for the plain sequence, ratio 1.0 and no ratios differ in the reference
    _, st_none, lp_none = _oracle_viterbi(oracle, m, obs[1], None)
    _, st_one, lp_one = _oracle_viterbi(oracle, m, obs[1], np.ones(lens[1]))
    assert lp_one != pytest.approx(lp_none, rel=1e-10)
    engine.set_precision(prec)
    try:
        hmm, em = _hmm(m)
        out = hmm.decode_batch(batch)
        eng = _engine()
        lp1, _, st1 = eng.decode_host([obs[1]], _lib.DECODE_VITERBI, precision=prec)
    finally:
        engine.set_precision("f32")
    assert_array_equal(out[1][1], st1[0])
    # fp32 at <= 32 states: alone, the log-probability is the DP's own sum; in a batch with ratios it is the
    # float64 re-score of the same path
    assert out[1][0] == pytest.approx(lp1[0], rel=1e-12 if prec == "f64" or N > 32 else 1e-9)
    for i in range(3):
        r = em.getSegmentRatios(batch[i])
        assert (r is None) == (i == 1)
        frame, want, wlp = _oracle_viterbi(oracle, m, obs[i], r)
        lp, st = out[i]
        if prec == "f64":
            assert_array_equal(st, want)
            assert lp == pytest.approx(wlp, rel=1e-10)
        else:
            assert_near_ties_only(st, want, frame, m["log_start"], m["log_trans"], r, label="mixed seq %d" % i)
            assert lp == pytest.approx(wlp, rel=1e-6)


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_decode_both_with_segment_ratios_is_the_two_calls(oracle, prec):
    """one upload (observations and ratios once), one emission pass: bit-identical to
    decode_batch(viterbi) then decode_batch(map); the forward log-likelihood bookkeeping is the same"""
    from tehmm_b200 import engine, synth
    m = _model(30, seed=0)
    rng = np.random.RandomState(1)
    lens = [1_200_003, 17, 300_000, 1]
    tables = []
    for i, n in enumerate(lens):
        o = synth.sample_obs(m, n, seed=20 + i)[0]
        tables.append(_segmented_table(o, np.minimum(rng.geometric(1.0 / 60.0, size=n), 100).astype(np.int64)))
    engine.set_precision(prec)
    try:
        hv, em = _hmm(m)
        hm, _ = _hmm(m, algorithm="map")
        hb, _ = _hmm(m)
        assert all(em.getSegmentRatios(t) is not None for t in tables)
        v, mp = hv.decode_batch(tables), hm.decode_batch(tables)
        both = hb.decode_both_batch(tables)
        eng = hb._engine()
        assert eng.h2d_bytes == sum(lens) * (m["K"] + 8)
    finally:
        engine.set_precision("f32")
    assert len(both) == len(tables)
    for (vlp, vst, msc, mst), (lp, st), (sc, ms) in zip(both, v, mp):
        assert vlp == lp and msc == sc
        assert_array_equal(vst, st)
        assert_array_equal(mst, ms)
    assert hb.getLastLogProb() == hm.getLastLogProb() and hb.getLastLogProb() is not None
    if prec == "f64":                      # and the MAP half ignores the ratios, as the reference's
        i = 2
        ref = oracle_all(oracle, tables[i].data, m["table"], 1.0, m["log_start"], m["log_trans"])
        assert_array_equal(both[i][3], np.argmax(ref["post"], axis=1))
        _, want, _ = _oracle_viterbi(oracle, m, tables[i].data, em.getSegmentRatios(tables[i]))
        assert_array_equal(both[i][1], want)


def test_refused_deferred_check_still_gives_the_reference_answers(oracle):
    """a warm-up of ONE step: the optimistic attempt of both entry points is refused and the synchronous
    verify / repair loop (which has no exact-resolution fallback with ratios) gives the oracle's answers"""
    from tehmm_b200 import _lib, synth
    from tehmm_b200.engine import Engine
    m = _model(30, seed=5)
    lens = [9000, 3, 26000]
    rng = np.random.RandomState(2)
    seqs = [synth.sample_obs(m, n, seed=40 + i)[0] for i, n in enumerate(lens)]
    ratios = [_ratios(rng, n) for n in lens]
    ratios[1] = None
    for both in (False, True):
        ctx = _lib.Context(0)                  # a fresh context: no back-off from an earlier refusal
        try:
            _setup(ctx)
            ctx.set_option("chunk_tiles", 2)
            ctx.set_option("fine_len", 48)
            ctx.set_option("warmup", 1)
            eng = Engine(ctx)
            eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
            bad0 = ctx.stat("deferred_bad")
            if both:
                lp, states, _, mstates, flp = eng.decode_host_both(seqs, precision="f64", ratios=ratios)
            else:
                lp, _, states = eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f64", ratios=ratios)
            assert ctx.stat("deferred_bad") > bad0
            assert ctx.check() == 0
            for i, obs in enumerate(seqs):
                _, want, wlp = _oracle_viterbi(oracle, m, obs, ratios[i])
                assert_array_equal(states[i], want)
                assert lp[i] == pytest.approx(wlp, rel=1e-10)
                if both:
                    ref = oracle.sweep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"])
                    assert_array_equal(mstates[i], ref["map_states"])
                    assert flp[i] == pytest.approx(ref["logprob"], rel=1e-10)
        finally:
            ctx.close()


def _raw_call(eng, both, seqs, ratios, obs_null=None):
    """the C entry point itself on sentinel-filled outputs; returns (rc, outputs)"""
    arrays, dt, offsets, ptrs = eng._host_arrays(seqs)
    if obs_null is not None:
        ptrs[obs_null] = None
    keep, rptrs = eng._host_ratios(ratios, offsets)
    total, n = int(offsets[-1]), len(seqs)
    outs = [np.full(total, -7, dtype=np.int64), np.full(n, 3.5), np.full(total, -7, dtype=np.int64),
            np.full(n, 3.5), np.full(n, 3.5)]
    p = [ctypes.c_void_p(a.ctypes.data) for a in outs]
    if both:
        rc = eng.lib.tehmm_decode_host_both_ratios(eng.ctx.handle, ptrs, n, dt.itemsize, n, _ptr(offsets), rptrs,
                                                   0, p[0], p[1], p[2], p[3], p[4])
    else:
        rc = eng.lib.tehmm_decode_host_ratios(eng.ctx.handle, ptrs, n, dt.itemsize, n, _ptr(offsets), rptrs,
                                              0, 0, p[0], p[1], p[3])
    del keep
    return rc, outs


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


@pytest.mark.parametrize("bad", [np.nan, np.inf, 0.0, -1.0])
def test_rejects_bad_ratios_and_leaves_outputs_alone(bad):
    from tehmm_b200 import _lib, synth
    m = _model(30, seed=1)
    lens = [3_000_000, 40]                 # the bad value lies in the last staging slice
    seqs = [synth.sample_obs(m, n, seed=90 + i)[0] for i, n in enumerate(lens)]
    ratios = [np.full(lens[0], 0.5), None]
    ratios[0][-3] = bad
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    for both in (False, True):
        rc, outs = _raw_call(eng, both, seqs, ratios)
        assert rc == _lib.TEHMM_EINVAL
        assert b"segment ratio" in eng.lib.tehmm_last_error()
        for o in outs:
            assert np.all(o == (-7 if o.dtype == np.int64 else 3.5))
    with pytest.raises(AssertionError):
        eng.decode_host(seqs, _lib.DECODE_VITERBI, ratios=ratios)
    with pytest.raises(AssertionError):
        eng.decode_host_both(seqs, ratios=ratios)
    # a NULL observation pointer
    good = [np.full(lens[0], 0.5), None]
    for both in (False, True):
        rc, outs = _raw_call(eng, both, seqs, good, obs_null=0)
        assert rc == _lib.TEHMM_EINVAL
        for o in outs:
            assert np.all(o == (-7 if o.dtype == np.int64 else 3.5))
    # and the context still decodes afterwards
    lp, _, st = eng.decode_host(seqs, _lib.DECODE_VITERBI, ratios=good)
    assert st[0].shape == (lens[0],) and np.isfinite(lp).all()


def test_wider_than_64_states_takes_the_strict_path(oracle):
    """more than 64 states: segmented tables are decoded by the strict float64 kernels, with the ratios"""
    from tehmm_b200 import engine, synth
    m = _model(70, seed=4)
    rng = np.random.RandomState(6)
    lens = [1500, 2]
    tables = [_segmented_table(synth.sample_obs(m, n, seed=80 + i)[0],
                               np.minimum(rng.geometric(1.0 / 60.0, size=n), 300).astype(np.int64))
              for i, n in enumerate(lens)]
    engine.set_precision("f64")
    try:
        hmm, em = _hmm(m)
        assert hmm._wide()
        out = hmm.decode_batch(tables)
        both = hmm.decode_both_batch(tables)
    finally:
        engine.set_precision("f32")
    for i, t in enumerate(tables):
        r = em.getSegmentRatios(t)
        _, want, wlp = _oracle_viterbi(oracle, m, t.data, r)
        assert_array_equal(out[i][1], want)
        assert out[i][0] == pytest.approx(wlp, rel=1e-10)
        assert_array_equal(both[i][1], want)
