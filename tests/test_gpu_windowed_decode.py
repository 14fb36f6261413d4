"""-m gpu: Viterbi and MAP decoding in time windows (Engine.viterbi / Engine.posteriors(want_map=True) /
Engine.decode_host* with max_window_steps, DESIGN.md section 11).  Each window's Viterbi DP starts from
the delta row the window to its left ends on and its traceback from the state the window to its right
chose (tehmm_set_viterbi_boundary); MAP runs through the windowed forward-backward.  So windowed paths
equal the unwindowed ones on the same GPU, and the float64 ones equal the oracle's."""
import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from parity import assert_map_near_ties_only, assert_near_ties_only, oracle_frame

pytestmark = pytest.mark.gpu

# ragged batch of test_gpu_windowed.py: one-step sequences, cuts one step after a start and one before an end
LENS = [9001, 5000, 1, 7, 12345]
CAPS = (sum(LENS) // 2 + 3, 9002, 7000, 4999, 26353)      # 2 .. 7 windows, none a multiple of a chunk or tile


def _engine():
    from tehmm_b200.engine import get_engine
    eng = get_engine(0)
    for k in ("chunk_tiles", "warmup", "fine_len"):
        eng.ctx.set_option(k, 0)
    eng.ctx.set_option("tile", 1)
    return eng


def _setup(N, lens, dtype=np.uint8, seed=3, ratios=False):
    from tehmm_b200 import synth
    m = synth.make_model(N=N, seed=seed)
    seqs = [synth.sample_obs(m, n, seed=seed * 100 + i)[0].astype(dtype) for i, n in enumerate(lens)]
    rr = None
    if ratios:
        rng = np.random.default_rng(seed)
        rr = [None if i == 1 else rng.choice([0.4, 1.0, 1.0, 2.5, 7.0], size=n) for i, n in enumerate(lens)]
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(seqs)
    return m, seqs, rr, eng


def _oracle_viterbi(oracle, m, obs, r):
    frame = oracle_frame(oracle, obs, m["table"], 1.0, None)
    st, lp = oracle._viterbi(obs.shape[0], m["N"], m["log_start"], m["log_trans"], r, frame)
    return frame, st, lp


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("N", [2, 30, 50, 64])
@pytest.mark.parametrize("ratios", [False, True])
def test_windowed_viterbi_equals_unwindowed(N, prec, ratios, oracle):
    m, seqs, rr, eng = _setup(N, LENS, ratios=ratios)
    ref_lp, ref_st = eng.viterbi(ratios_dp=rr, precision=prec)
    # Engine.viterbi gives a sequence without ratios 1.0 in a batch that has some (upload_ratios)
    r_or = [None if rr is None else (np.ones(len(o)) if rr[i] is None else rr[i]) for i, o in enumerate(seqs)]
    refs = [_oracle_viterbi(oracle, m, o, r) for o, r in zip(seqs, r_or)] if prec == "f32" else None
    for cap in CAPS:
        total = sum(LENS)
        assert 2 <= -(-total // cap) <= 7 and total % cap != 0
        lp, st = eng.viterbi(ratios_dp=rr, precision=prec, max_window_steps=cap)
        if prec == "f64":
            for a, b in zip(st, ref_st):
                assert_array_equal(a, b)
            assert_allclose(lp, ref_lp, rtol=1e-12)
        else:
            assert_allclose(lp, ref_lp, rtol=1e-5)
            for i, (a, (frame, ost, _)) in enumerate(zip(st, refs)):
                assert_near_ties_only(a, ost, frame, m["log_start"], m["log_trans"], r_or[i],
                                      label="N=%d cap=%d seq %d" % (N, cap, i))


def test_one_step_viterbi_windows_against_the_oracle(oracle):
    """windows of ONE step (every row a window) on a short batch: f64 against the oracle's Viterbi"""
    m, seqs, rr, eng = _setup(30, [40, 1, 25], dtype=np.uint16)
    lp, st = eng.viterbi(precision="f64", max_window_steps=1)
    for i, o in enumerate(seqs):
        _, ost, olp = _oracle_viterbi(oracle, m, o, None)
        assert_array_equal(st[i], ost)
        assert lp[i] == pytest.approx(olp, rel=1e-10)


def test_cut_where_the_path_stays_in_state_0_with_a_ratio(oracle):
    """the first row of a window has ratio 7.0 and the best path goes 0 -> 0 across the cut: the
    reference's from-state-0 term (_hmm.pyx:234-237) at the continued first row, f64 against the oracle"""
    from tehmm_b200 import synth
    m = synth.make_model(N=8, seed=5, sticky=0.97)
    obs = synth.sample_obs(m, 6000, seed=51)[0]
    r = np.ones(obs.shape[0])
    frame = oracle_frame(oracle, obs, m["table"], 1.0, None)
    st, _ = oracle._viterbi(obs.shape[0], m["N"], m["log_start"], m["log_trans"], r, frame)
    cut = None
    for t in range(1500, 4500):
        if st[t - 1] == 0 and st[t] == 0:
            r2 = r.copy()
            r2[t] = 7.0
            st2, _ = oracle._viterbi(obs.shape[0], m["N"], m["log_start"], m["log_trans"], r2, frame)
            if st2[t - 1] == 0 and st2[t] == 0:
                cut, r, st = t, r2, st2
                break
    assert cut is not None, "no 0 -> 0 step in the sampled path"
    _, lp_ref = oracle._viterbi(obs.shape[0], m["N"], m["log_start"], m["log_trans"], r, frame)
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    lp, got = eng.viterbi(ratios_dp=[r], precision="f64", max_window_steps=cut)
    assert_array_equal(got[0], st)
    assert lp[0] == pytest.approx(lp_ref, rel=1e-10)


def test_all_missing_stretch_across_a_cut(oracle):
    """a stretch of missing data (symbol 0 on every track) across the cut: the DP's and the traceback's
    exact fallback run next to the boundary conditions; Viterbi and MAP, f64 against the oracle"""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=8)
    obs = synth.sample_obs(m, 6000, seed=81)[0]
    obs[2500:3700] = 0
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    ref = oracle.sweep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"])
    lp, st = eng.viterbi(precision="f64", max_window_steps=3001)
    assert_array_equal(st[0], ref["vit_states"])
    assert lp[0] == pytest.approx(ref["vit_logprob"], rel=1e-10)
    out = eng.posteriors(renorm_eps=True, want_post=False, want_map=True, precision="f64", max_window_steps=3001)
    assert_array_equal(out["map_states"][0], ref["map_states"])
    assert out["map_score"][0] == pytest.approx(ref["map_score"], rel=1e-9)
    assert out["logprob"][0] == pytest.approx(ref["logprob"], rel=1e-10)


def test_deferred_check_refused_inside_a_windowed_viterbi():
    """warm-up of one step: the optimistic attempt of a window is refused and redone synchronously"""
    m, seqs, rr, eng = _setup(30, [9000, 3, 26000])
    ref_lp, ref_st = eng.viterbi(precision="f64")
    eng.ctx.set_option("chunk_tiles", 2)
    eng.ctx.set_option("fine_len", 48)
    eng.ctx.set_option("warmup", 1)
    try:
        eng.upload_batch(seqs)
        eng.ctx.set_option("defer_skip", 0)
        bad = eng.ctx.stat("deferred_bad")
        lp, st = eng.viterbi(precision="f64", max_window_steps=12000)
        assert eng.ctx.stat("deferred_bad") > bad
        assert eng.ctx.check() == 0
    finally:
        for k in ("chunk_tiles", "warmup", "fine_len"):
            eng.ctx.set_option(k, 0)
    for a, b in zip(st, ref_st):
        assert_array_equal(a, b)
    assert_allclose(lp, ref_lp, rtol=1e-12)


def test_viterbi_boundary_is_checked_and_no_boundary_changes_nothing():
    from tehmm_b200 import _lib
    m, seqs, rr, eng = _setup(30, [10, 20])
    h = eng.ctx.handle
    f = eng.lib.tehmm_set_viterbi_boundary
    d = np.zeros(30)
    s0, s2, s10 = (np.array([k], dtype=np.int64) for k in (0, 2, 1))
    two = np.array([1, 0], dtype=np.int64)
    st0, st_bad, st_neg = (np.array([k], dtype=np.int32) for k in (0, 30, -1))
    for seq, vec in ((s2, d), (two, np.zeros(60)), (s0, np.full(30, np.nan)), (s0, np.full(30, np.inf)),
                     (s0, np.full(30, -np.inf))):
        assert f(h, len(seq), _lib.ptr(seq), _lib.ptr(np.ascontiguousarray(vec)), 0, None, None, None) == _lib.TEHMM_EINVAL
    for st, ratio in ((st_bad, None), (st_neg, None), (st0, np.array([np.inf])), (st0, np.array([np.nan])),
                      (st0, np.array([0.0]))):
        assert f(h, 0, None, None, 1, _lib.ptr(s0), _lib.ptr(st), _lib.ptr(ratio)) == _lib.TEHMM_EINVAL
    assert f(h, 0, None, None, 1, _lib.ptr(s2), _lib.ptr(st0), None) == _lib.TEHMM_EINVAL
    # accepted: -inf components with a finite one, no ratio or a negative one (none)
    v = np.full(30, -np.inf)
    v[3] = -2.0
    _lib.check(f(h, 1, _lib.ptr(s10), _lib.ptr(v), 1, _lib.ptr(s0), _lib.ptr(st0), _lib.ptr(np.array([-1.0]))))
    # no boundary (cleared by a call without entries, and by tehmm_set_batch): bit-identical passes
    _lib.check(f(h, 0, None, None, 0, None, None, None))
    m, seqs, rr, eng = _setup(30, LENS, ratios=True)
    for prec in ("f32", "f64"):
        a_lp, a_st = eng.viterbi(ratios_dp=rr, precision=prec)
        _lib.check(f(h, 0, None, None, 0, None, None, None))
        b_lp, b_st = eng.viterbi(ratios_dp=rr, precision=prec)
        assert np.array_equal(a_lp, b_lp)
        assert all(np.array_equal(x, y) for x, y in zip(a_st, b_st))


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("N", [2, 30, 50, 64])
def test_windowed_map_equals_unwindowed(N, prec):
    m, seqs, rr, eng = _setup(N, LENS)
    ref = eng.posteriors(renorm_eps=True, want_post=True, want_map=True, precision=prec)
    ref64 = eng.posteriors(renorm_eps=True, want_post=True, precision="f64") if prec == "f32" else ref
    t = dict(rtol=1e-10) if prec == "f64" else dict(rtol=1e-5)
    for cap in CAPS[:3]:
        for want_post in (False, True):
            got = eng.posteriors(renorm_eps=True, want_post=want_post, want_map=True, precision=prec,
                                 max_window_steps=cap)
            assert_allclose(got["logprob"], ref["logprob"], **t)
            assert_allclose(got["map_score"], ref["map_score"], **t)
            for i, (a, b) in enumerate(zip(got["map_states"], ref["map_states"])):
                if prec == "f64":
                    assert_array_equal(a, b)
                else:
                    assert_map_near_ties_only(a, ref64["post"][i], label="N=%d cap=%d seq %d" % (N, cap, i))
            if want_post:
                for a, b in zip(got["post"], ref["post"]):
                    assert_allclose(a, b, **(dict(rtol=1e-10, atol=1e-12) if prec == "f64" else dict(rtol=1e-5, atol=2e-6)))


def _decode_inputs(N, ratios):
    from tehmm_b200 import synth
    m = synth.make_model(N=N, seed=11)
    seqs = [synth.sample_obs(m, n, seed=110 + i)[0] for i, n in enumerate(LENS)]
    rr = None
    if ratios:
        rng = np.random.default_rng(11)
        rr = [None if i == 1 else rng.choice([0.4, 1.0, 2.5, 7.0], size=n) for i, n in enumerate(LENS)]
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    return m, seqs, rr, eng


def _same_decode(a, b, map_score=True):
    lp_a, sc_a, st_a = a
    lp_b, sc_b, st_b = b
    assert_allclose(lp_a, lp_b, rtol=1e-10)
    if map_score:
        assert_allclose(sc_a, sc_b, rtol=1e-10)
    assert len(st_a) == len(st_b)
    for x, y in zip(st_a, st_b):
        assert x.dtype == np.int64
        assert_array_equal(x, y)


@pytest.mark.parametrize("N", [30, 50])
@pytest.mark.parametrize("ratios", [False, True])
def test_decode_host_in_windows_equals_the_one_call(N, ratios):
    """float64, one array per sequence: VITERBI, MAP and BOTH through the windows equal the host call"""
    from tehmm_b200 import _lib
    m, seqs, rr, eng = _decode_inputs(N, ratios)
    for cap in (9002, 4999):
        _same_decode(eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f64", ratios=rr, max_window_steps=cap),
                     eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f64", ratios=rr), map_score=False)
        _same_decode(eng.decode_host(seqs, _lib.DECODE_MAP, precision="f64", ratios=rr, max_window_steps=cap),
                     eng.decode_host(seqs, _lib.DECODE_MAP, precision="f64", ratios=rr))
        got = eng.decode_host_both(seqs, precision="f64", ratios=rr, max_window_steps=cap)
        ref = eng.decode_host_both(seqs, precision="f64", ratios=rr)
        _same_decode((got[0], None, got[1]), (ref[0], None, ref[1]), map_score=False)
        _same_decode((got[4], got[2], got[3]), (ref[4], ref[2], ref[3]))


def test_multitrack_hmm_decodes_in_windows(monkeypatch):
    """MultitrackHmm.decode_both / decode (viterbi, map) with every host decode in windows, float64"""
    from tehmm_b200 import engine
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    from tehmm_b200.engine import Engine
    from tehmm_b200.hmm import MultitrackHmm
    m, seqs, rr, eng = _decode_inputs(30, False)

    def run():
        em = IndependentMultinomialEmissionModel(30, list(m["syms"]), zeroAsMissingData=True)
        em.logProbs = m["table"].copy()
        h = MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy())
        return h.decode_both_batch(seqs), h.decode_batch(seqs, "viterbi"), h.decode_batch(seqs, "map")
    old = engine.get_precision()
    engine.set_precision("f64")
    try:
        a = run()
        one, both = Engine.decode_host, Engine.decode_host_both
        monkeypatch.setattr(Engine, "decode_host", lambda self, *args, **kw: one(self, *args, max_window_steps=7000, **kw))
        monkeypatch.setattr(Engine, "decode_host_both",
                            lambda self, *args, **kw: both(self, *args, max_window_steps=7000, **kw))
        b = run()
    finally:
        engine.set_precision(old)
    for x, y in zip(a[0], b[0]):
        assert x[0] == pytest.approx(y[0], rel=1e-10) and x[2] == pytest.approx(y[2], rel=1e-10)
        assert_array_equal(x[1], y[1])
        assert_array_equal(x[3], y[3])
    for ra, rb in zip(a[1:], b[1:]):
        for x, y in zip(ra, rb):
            assert x[0] == pytest.approx(y[0], rel=1e-10)
            assert_array_equal(x[1], y[1])


class _FakeLib(object):
    """the library with the host decodes returning `code` (as when the arena does not fit)"""

    def __init__(self, lib, code):
        self._lib, self._code = lib, code

    def __getattr__(self, name):
        if name.startswith("tehmm_decode_host") and name != "tehmm_decode_host_bytes":
            return lambda *args: self._code
        return getattr(self._lib, name)


def test_out_of_memory_route_decodes_in_windows(monkeypatch):
    """TEHMM_ENOMEM from the host decode: the batch is decoded through the engine instead (here unwindowed
    or in windows as free memory allows: the batch is small), with the host call's results; other codes raise"""
    from tehmm_b200 import _lib
    m, seqs, rr, eng = _decode_inputs(30, True)
    ref_v = eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f64", ratios=rr)
    ref_b = eng.decode_host_both(seqs, precision="f64", ratios=rr)
    real = eng.lib
    monkeypatch.setattr(eng, "lib", _FakeLib(real, _lib.TEHMM_ENOMEM))
    _same_decode(eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f64", ratios=rr), ref_v, map_score=False)
    got = eng.decode_host_both(seqs, precision="f64", ratios=rr)
    _same_decode((got[0], None, got[1]), (ref_b[0], None, ref_b[1]), map_score=False)
    _same_decode((got[4], got[2], got[3]), (ref_b[4], ref_b[2], ref_b[3]))
    monkeypatch.setattr(eng, "lib", _FakeLib(real, _lib.TEHMM_ECUDA))
    with pytest.raises(_lib.TehmmError):
        eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f64")
    with pytest.raises(_lib.TehmmError):
        eng.decode_host_both(seqs, precision="f64")
