"""-m gpu: forward-backward in time windows (Engine.estep / Engine.posteriors with
max_window_steps, DESIGN.md section 11).  Every window runs exactly from the boundary
vectors of its neighbours, so windowed statistics, log-likelihoods and posteriors equal
the unwindowed ones on the same GPU, and the float64 ones equal the oracle's."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

pytestmark = pytest.mark.gpu


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
        rr = [None if i == 1 else rng.choice([1.0, 1.0, 2.5, 7.0], size=n) for i, n in enumerate(lens)]
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(seqs)
    return m, seqs, rr, eng


def _tol(prec):
    return dict(rtol=1e-10, atol=1e-12) if prec == "f64" else dict(rtol=1e-5, atol=2e-6)


def _same_stats(a, b, prec):
    t = _tol(prec)
    assert a["nobs"] == b["nobs"]
    assert a["logprob"] == pytest.approx(b["logprob"], rel=t["rtol"])
    assert_allclose(a["logprobs"], b["logprobs"], rtol=t["rtol"])
    assert_allclose(a["start"], b["start"], **t)
    assert_allclose(a["trans"], b["trans"], **t)
    assert_allclose(a["obs"], b["obs"], **t)


# ragged batches: one-step sequences, cuts one step after a start and one before an end
# (sequence 1 covers rows 9001 .. 14000: windows of 9002 rows cut one step after its start, windows
# of 7000 rows one step before its end; windows of 26353 rows leave a last window of one step)
LENS = [9001, 5000, 1, 7, 12345]


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("N", [2, 30, 50, 64])
@pytest.mark.parametrize("ratios", [False, True])
def test_windowed_estep_equals_unwindowed(N, prec, ratios):
    m, seqs, rr, eng = _setup(N, LENS, ratios=ratios)
    total = sum(LENS)
    ref = eng.estep(ratios=rr, precision=prec)
    for cap in (total // 2 + 3, 9002, 7000, 4999, 26353):   # 2 .. 6 windows, none a multiple of a chunk or tile
        n_win = -(-total // cap)
        assert 2 <= n_win <= 7 and total % cap != 0
        got = eng.estep(ratios=rr, precision=prec, max_window_steps=cap)
        _same_stats(got, ref, prec)


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int32])
@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("N", [2, 30, 50, 64])
def test_windowed_posteriors_equal_unwindowed(N, dtype, prec):
    m, seqs, rr, eng = _setup(N, LENS, dtype=dtype, ratios=True)
    for renorm in (True, False):
        ref = eng.posteriors(ratios_dp=rr, renorm_eps=renorm, precision=prec)
        for cap in (sum(LENS) // 3 + 1, 9002, 5001):
            got = eng.posteriors(ratios_dp=rr, renorm_eps=renorm, precision=prec, max_window_steps=cap)
            assert_allclose(got["logprob"], ref["logprob"], rtol=_tol(prec)["rtol"])
            for a, b in zip(got["post"], ref["post"]):
                assert a.shape == b.shape
                assert_allclose(a, b, **_tol(prec))


@pytest.mark.parametrize("N", [50, 64])
def test_tcgen05_backward_takes_windows_with_exit_vectors(N):
    """33..64 states, fp32: every window of one long sequence is a single-sequence batch, so the
    tcgen05 forward and backward kernels take its first passes -- the backward of every window but the
    last one ending on an exit vector.  umma_passes counts them: 3 forward passes of the forward sweep,
    then a forward and a backward pass per window (11 in all) can only be reached if all 4 backward
    passes took the tcgen05 kernel."""
    m, seqs, rr, eng = _setup(N, [40000])
    ref = eng.posteriors(renorm_eps=True, precision="f32")
    before = eng.ctx.stat("umma_passes")
    got = eng.posteriors(renorm_eps=True, precision="f32", max_window_steps=10001)
    assert eng.ctx.stat("umma_passes") - before >= 11
    assert_allclose(got["logprob"], ref["logprob"], rtol=1e-5)
    assert_allclose(got["post"][0], ref["post"][0], **_tol("f32"))


def test_one_step_windows_against_the_oracle(oracle):
    """windows of ONE step (every row a window) and a short batch: f64 against the oracle's E-step"""
    m, seqs, rr, eng = _setup(30, [40, 1, 25], dtype=np.uint16)
    got = eng.estep(precision="f64", max_window_steps=1)
    K, N, S = m["table"].shape
    s0, tr, ob = np.zeros(N), np.zeros((N, N)), np.zeros((K, N, S))
    lps = [oracle.estep_sequence(o, m["table"], 1.0, m["log_start"], m["log_trans"], None, s0, tr, ob) for o in seqs]
    assert_allclose(got["logprobs"], lps, rtol=1e-10)
    assert_allclose(got["start"], s0, rtol=1e-10, atol=1e-14)
    assert_allclose(got["trans"], tr, rtol=1e-10, atol=1e-14)
    assert_allclose(got["obs"], ob, rtol=1e-10, atol=1e-14)


def test_all_missing_gap_across_a_cut(oracle):
    """a stretch of missing data (symbol 0 on every track) across the cut: f64 against the oracle"""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=8)
    obs = synth.sample_obs(m, 6000, seed=81)[0]
    obs[2500:3700] = 0
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    got = eng.estep(precision="f64", max_window_steps=3001)
    plain = eng.estep(precision="f64")
    _same_stats(got, plain, "f64")
    K, N, S = m["table"].shape
    s0, tr, ob = np.zeros(N), np.zeros((N, N)), np.zeros((K, N, S))
    lp = oracle.estep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"], None, s0, tr, ob)
    # the gap leaves the float64 chunk boundaries to the exact fallback, accepted at its own tolerance
    # (api.cu, tolerance_after_fallback): windowed or not, the counts are within ~1e-9 of the oracle's
    assert got["logprob"] == pytest.approx(lp, rel=1e-10)
    assert_allclose(got["start"], s0, rtol=1e-8, atol=1e-14)
    assert_allclose(got["trans"], tr, rtol=1e-8, atol=1e-14)
    assert_allclose(got["obs"], ob, rtol=1e-8, atol=1e-14)
    post = eng.posteriors(renorm_eps=False, precision="f64", max_window_steps=3001)
    ref = oracle.sweep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"])
    assert post["logprob"][0] == pytest.approx(ref["logprob"], rel=1e-10)


def test_no_boundary_vectors_change_nothing():
    """tehmm_set_boundary with no vectors leaves every pass bit-identical"""
    from tehmm_b200 import _lib
    m, seqs, rr, eng = _setup(30, LENS)
    a = eng.estep(precision="f32")
    _lib.check(eng.lib.tehmm_set_boundary(eng.ctx.handle, 0, None, None, 0, None, None))
    b = eng.estep(precision="f32")
    for k in ("start", "trans", "obs", "logprobs"):
        assert np.array_equal(a[k], b[k]), k
    pa = eng.posteriors(precision="f32")
    _lib.check(eng.lib.tehmm_set_boundary(eng.ctx.handle, 0, None, None, 0, None, None))
    pb = eng.posteriors(precision="f32")
    assert np.array_equal(pa["logprob"], pb["logprob"])
    assert all(np.array_equal(x, y) for x, y in zip(pa["post"], pb["post"]))


def test_boundary_vectors_are_checked():
    from tehmm_b200 import _lib
    m, seqs, rr, eng = _setup(30, [10, 20])
    v = np.full(30, 1.0 / 30)
    for seq, vec in (([2], v), ([0], -v), ([0], np.zeros(30)), ([0], np.full(30, np.nan))):
        s = np.array(seq, dtype=np.int64)
        vec = np.ascontiguousarray(vec)
        assert eng.lib.tehmm_set_boundary(eng.ctx.handle, 1, _lib.ptr(s), _lib.ptr(vec), 0, None, None) == _lib.TEHMM_EINVAL
    # unfolded ratios in the backward pass's own transition counts would count a continued first row as a start
    s, vec = np.zeros(1, dtype=np.int64), np.ascontiguousarray(v)
    _lib.check(eng.lib.tehmm_set_boundary(eng.ctx.handle, 1, _lib.ptr(s), _lib.ptr(vec), 0, None, None))
    prec, tdt = eng._prec("f32")
    d_r = eng.upload_ratios([np.full(10, 2.0), None])
    _, blin, rowmax = eng.run_emission(prec, tdt, None, False, True)
    alpha, _ = eng.run_forward(prec, tdt, blin, rowmax, d_r)
    st = eng.empty(30 + 900, eng.torch.float64).zero_()
    with pytest.raises(AssertionError, match="fold the ratios"):
        eng.run_backward(prec, tdt, _lib.BWD_TRANS, blin, alpha, d_r, start_trans=st)


def test_deferred_check_refused_inside_a_windowed_estep():
    """warm-up of one step: the optimistic attempt of a window is refused and redone synchronously"""
    m, seqs, rr, eng = _setup(30, [9000, 3, 26000])
    ref = eng.estep(precision="f32")
    eng.ctx.set_option("chunk_tiles", 2)
    eng.ctx.set_option("fine_len", 48)
    eng.ctx.set_option("warmup", 1)
    try:
        eng.upload_batch(seqs)
        eng.ctx.set_option("defer_skip", 0)
        bad = eng.ctx.stat("deferred_bad")
        got = eng.estep(precision="f32", max_window_steps=12000)
        assert eng.ctx.stat("deferred_bad") > bad
        assert eng.ctx.check() == 0
    finally:
        for k in ("chunk_tiles", "warmup", "fine_len"):
            eng.ctx.set_option(k, 0)
    _same_stats(got, ref, "f32")


def test_fit_windowed_equals_unwindowed(monkeypatch):
    """three EM iterations of MultitrackHmm.fit in float64 with every E-step in windows, at the
    tolerances of the strict-kernel fit test"""
    from tehmm_b200 import engine, synth
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    from tehmm_b200.engine import Engine
    from tehmm_b200.hmm import MultitrackHmm
    syms = (5, 3, 9)
    m = synth.make_model(N=50, syms=syms, seed=13)
    seqs = [synth.sample_obs(m, T, seed=20 + i)[0] for i, T in enumerate([4000, 1, 2570])]

    def fitted():
        em = IndependentMultinomialEmissionModel(50, list(syms), zeroAsMissingData=True)
        em.logProbs = m["table"].copy()
        h = MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy(), n_iter=3, thresh=0.0)
        h.fit(seqs)
        return h, em
    old = engine.get_precision()
    engine.set_precision("f64")
    try:
        a, ema = fitted()
        plain = Engine.estep
        monkeypatch.setattr(Engine, "estep", lambda self, *args, **kw: plain(self, *args, max_window_steps=1777, **kw))
        b, emb = fitted()
    finally:
        engine.set_precision(old)
    assert_allclose(a.transmat_, b.transmat_, rtol=1e-9, atol=1e-300)
    assert_allclose(a.startprob_, b.startprob_, rtol=1e-9, atol=1e-300)
    assert_allclose(ema.getLogProbs(), emb.getLogProbs(), rtol=1e-9, atol=1e-300)
    assert a.getLastLogProb() == pytest.approx(b.getLastLogProb(), rel=1e-10)
