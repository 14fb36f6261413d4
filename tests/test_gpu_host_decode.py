"""-m gpu: tehmm_decode_host -- the whole decode call with HOST buffers on both
sides (pinned staging + worker threads in, uint8 states over PCIe widened to the
reference's int64 out) -- against the oracle and against the device-pointer path
it is built on.  Reference call being replaced: basehmm.py:361-396 decode ->
hmm.py:668-676 / basehmm.py:332-359.
"""
import numpy as np
import pytest
from numpy.testing import assert_array_equal

from parity import assert_map_near_ties_only, assert_near_ties_only, oracle_all, oracle_frame

pytestmark = pytest.mark.gpu


def _engine():
    from tehmm_b200.engine import get_engine
    eng = get_engine(0)
    for k in ("chunk_tiles", "warmup", "fine_len"):
        eng.ctx.set_option(k, 0)
    eng.ctx.set_option("tile", 1)
    return eng


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int32])
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_decode_host_matches_oracle(oracle, dtype, prec):
    from tehmm_b200 import _lib, synth
    m = synth.make_model(N=30, seed=5)
    lens = [1, 7, 4099, 20000, 333]                       # ragged, incl. a one-step sequence
    seqs = [synth.sample_obs(m, n, seed=10 + i)[0].astype(dtype) for i, n in enumerate(lens)]
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    lp, _, states = eng.decode_host(seqs, _lib.DECODE_VITERBI, precision=prec)
    flp, score, mstates = eng.decode_host(seqs, _lib.DECODE_MAP, precision=prec)
    for i, obs in enumerate(seqs):
        ref = oracle.sweep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"])
        assert states[i].dtype == np.int64 and states[i].shape == (lens[i],)
        if prec == "f64":
            assert_array_equal(states[i], ref["vit_states"])
            assert_array_equal(mstates[i], ref["map_states"])
        else:
            full = oracle_all(oracle, obs, m["table"], 1.0, m["log_start"], m["log_trans"])
            assert_near_ties_only(states[i], ref["vit_states"], full["frame"], m["log_start"], m["log_trans"])
            assert_map_near_ties_only(mstates[i], full["post"])
        tol = 1e-10 if prec == "f64" else 1e-5
        assert lp[i] == pytest.approx(ref["vit_logprob"], rel=1e-6 if prec == "f32" else 1e-10)
        assert flp[i] == pytest.approx(ref["logprob"], rel=tol)


def test_decode_host_equals_device_path_large():
    """1.5 M steps (several staging slices and D2H slices), pageable and pinned input:
    bit-identical to the torch-plumbed device-pointer path."""
    import torch
    from tehmm_b200 import _lib, synth
    m = synth.make_model(N=30, seed=0)
    T = 1_500_000
    obs, _ = synth.sample_obs(m, T, seed=2)
    obs2, _ = synth.sample_obs(m, 200_003, seed=3)
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs, obs2])
    lp_d, st_d = eng.viterbi()
    out = eng.posteriors(renorm_eps=True, want_post=False, want_map=True)
    pinned = torch.from_numpy(obs).pin_memory().numpy()
    for first in (obs, pinned):
        lp, _, st = eng.decode_host([first, obs2], _lib.DECODE_VITERBI)
        assert eng.d2h_bytes == T + 200_003 + 32
        assert_array_equal(lp, lp_d)
        assert_array_equal(st[0], st_d[0])
        assert_array_equal(st[1], st_d[1])
        flp, sc, ms = eng.decode_host([first, obs2], _lib.DECODE_MAP)
        assert_array_equal(flp, out["logprob"])
        assert_array_equal(sc, out["map_score"])
        assert_array_equal(ms[0], out["map_states"][0])
        assert_array_equal(ms[1], out["map_states"][1])
    assert eng.h2d_bytes == (T + 200_003) * 10 and eng.d2h_bytes == T + 200_003 + 32


@pytest.mark.parametrize("nseq", [1, 2])
def test_decode_host_wide_model_equals_device_path(nseq):
    """50 states (lattice rows of 64 floats): the host-buffer call streams the observations through the wide
    four-states-per-lane emission kernel in pieces and runs the tcgen05 forward / backward kernels (one sequence)
    or the generic ones (two), the two-warps-per-chunk Viterbi DP and the two-chunks-per-warp traceback:
    bit-identical to the torch-plumbed device-pointer path."""
    from tehmm_b200 import _lib, synth
    m = synth.make_model(N=50, seed=3)
    lens = [700_001] if nseq == 1 else [400_000, 300_001]
    seqs = [synth.sample_obs(m, n, seed=20 + i)[0] for i, n in enumerate(lens)]
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(seqs)
    lp_d, st_d = eng.viterbi()
    out = eng.posteriors(renorm_eps=True, want_post=False, want_map=True)
    before = eng.ctx.stat("umma_passes")
    lp, _, st = eng.decode_host(seqs, _lib.DECODE_VITERBI)
    flp, sc, ms = eng.decode_host(seqs, _lib.DECODE_MAP)
    assert eng.ctx.stat("umma_passes") == before + (2 if nseq == 1 else 0)
    assert_array_equal(lp, lp_d)
    assert_array_equal(flp, out["logprob"])
    assert_array_equal(sc, out["map_score"])
    for i in range(nseq):
        assert_array_equal(st[i], st_d[i])
        assert_array_equal(ms[i], out["map_states"][i])


def test_decode_both_equals_the_two_calls():
    """one upload, one emission pass, both decodings: bit-identical to decode(viterbi) and decode(map)"""
    from tehmm_b200 import synth
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    from tehmm_b200.engine import get_engine
    from tehmm_b200.hmm import MultitrackHmm
    m = synth.make_model(N=30, seed=0)
    obs = [synth.sample_obs(m, T, seed=20 + i)[0] for i, T in enumerate([1_200_003, 17, 300_000, 1])]
    em = IndependentMultinomialEmissionModel(30, list(m["syms"]), zeroAsMissingData=True)
    em.logProbs = m["table"].copy()
    hv = MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy())
    hm = MultitrackHmm(em, startprob=m["pi"].copy(), transmat=m["A"].copy(), algorithm="map")
    v, mp = hv.decode_batch(obs), hm.decode_batch(obs)
    both = hv.decode_both_batch(obs)
    assert len(both) == len(obs)
    for (vlp, vst, msc, mst), (lp, st), (sc, ms) in zip(both, v, mp):
        assert vlp == lp and msc == sc
        assert_array_equal(vst, st)
        assert_array_equal(mst, ms)
        assert vst.dtype == np.int64 and mst.dtype == np.int64
    assert get_engine(0).d2h_bytes == 2 * sum(len(o) for o in obs) + 32 * len(obs)
    assert hv.getLastLogProb() is not None


def test_decode_api_uses_host_path_and_keeps_reference_answers():
    """hmmTest.py:48-135 known answer through MultitrackHmm.decode (now tehmm_decode_host)."""
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    from tehmm_b200.hmm import MultitrackHmm
    em = IndependentMultinomialEmissionModel(2, [3], [[[0.1, 0.4, 0.5], [0.6, 0.3, 0.1]]], zeroAsMissingData=False)
    hmm = MultitrackHmm(em, startprob=[0.6, 0.4], transmat=[[0.7, 0.3], [0.4, 0.6]])
    lp, st = hmm.decode(np.array([[0], [1], [2]], dtype=np.int64))   # non-fast dtype: cast on host
    assert np.exp(lp) == pytest.approx(0.01344, rel=1e-6)
    assert_array_equal(st, [1, 0, 0])
    assert st.dtype == np.int64


@pytest.mark.parametrize("nranks", [2, 5])
def test_time_sharded_single_sequence_virtual_ranks(nranks):
    """SURVEY 8e / config 5: one long sequence split in time over `nranks` (virtual) ranks --
    every rank's window decoded on this GPU in turn, the boundary vectors exchanged through
    the same verdict the all-gather feeds -- equals the single-GPU decode of the whole
    sequence: Viterbi path and float64 score, MAP path, forward log-likelihood."""
    from tehmm_b200 import parallel, synth
    m = synth.make_model(N=30, seed=4)
    T = 400_000
    obs, _ = synth.sample_obs(m, T, seed=9)
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    lp_full, st_full = eng.viterbi()
    out = eng.posteriors(renorm_eps=True, want_post=False, want_map=True)
    shards = parallel.time_shards(T, nranks)
    H = 2048
    for fn, kind in ((eng.viterbi_window, "viterbi"), (eng.map_window, "map"), (eng.score_window, "score")):
        res = [fn(obs, c, (max(0, c[0] - H), min(T, c[1] + H))) for c in shards]
        allv = [parallel.boundary_vector(r) for r in res]
        assert parallel.boundaries_agree(allv, shards, res[0]["mode"], res[0]["tol"]), kind
        if kind == "viterbi":
            path = np.concatenate([r["result"][1] for r in res])
            assert_array_equal(path, st_full[0])
            # the shards return float64 path scores, the single-GPU decode the fp32 DP's own value
            assert sum(r["result"][0] for r in res) == pytest.approx(lp_full[0], rel=1e-8)
        elif kind == "map":
            assert_array_equal(np.concatenate([r["result"] for r in res]), out["map_states"][0])
        else:
            assert sum(r["result"] for r in res) == pytest.approx(out["logprob"][0], rel=1e-9)
    # a halo of 2 steps must be caught at the boundaries
    res = [eng.viterbi_window(obs, c, (max(0, c[0] - 2), min(T, c[1] + 2))) for c in shards]
    assert not parallel.boundaries_agree([parallel.boundary_vector(r) for r in res], shards, "diff", 1e-5)


def test_decode_host_list_of_sequences_without_concatenation():
    """nptr = nseq: one host matrix per sequence (the reference's list of TrackTables)"""
    from tehmm_b200 import _lib, synth
    m = synth.make_model(N=30, seed=6)
    lens = [3_000_001, 17, 1_200_000, 5]                 # slices of the staging ring span sequences
    seqs = [synth.sample_obs(m, n, seed=40 + i)[0] for i, n in enumerate(lens)]
    eng = _engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    lp, _, st = eng.decode_host(seqs, _lib.DECODE_VITERBI)
    for i, s in enumerate(seqs):
        lp1, _, st1 = eng.decode_host([s], _lib.DECODE_VITERBI)
        assert_array_equal(st[i], st1[0])
        assert lp[i] == pytest.approx(lp1[0], rel=1e-12)


def test_deferred_verification_falls_back_to_the_repair_loop(oracle):
    """tehmm_ctx_check / option "defer": the stages are queued without waiting for their
    verification counts; with a warm-up of ONE step almost every speculated chunk boundary
    is wrong, so the check must fail and the synchronous verify / repair loop must produce
    the reference's answers (_hmm.pyx:120-259) all the same -- through the host-buffer decode
    and through the engine passes."""
    from tehmm_b200 import _lib, synth
    m = synth.make_model(N=30, seed=5)
    lens = [9000, 3, 26000]
    seqs = [synth.sample_obs(m, n, seed=40 + i)[0] for i, n in enumerate(lens)]
    eng = _engine()
    eng.ctx.set_option("chunk_tiles", 2)
    eng.ctx.set_option("fine_len", 48)
    eng.ctx.set_option("warmup", 1)
    try:
        eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
        eng.ctx.set_option("defer_skip", 0)
        bad0 = eng.ctx.stat("deferred_bad")
        lp, _, states = eng.decode_host(seqs, _lib.DECODE_VITERBI, precision="f64")
        flp, score, mstates = eng.decode_host(seqs, _lib.DECODE_MAP, precision="f64")
        assert eng.ctx.stat("deferred_bad") > bad0               # the optimistic attempt was refused
        assert eng.ctx.check() == 0                              # and nothing is left pending
        for i, obs in enumerate(seqs):
            ref = oracle.sweep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"])
            assert_array_equal(states[i], ref["vit_states"])
            assert_array_equal(mstates[i], ref["map_states"])
            assert lp[i] == pytest.approx(ref["vit_logprob"], rel=1e-10)
            assert flp[i] == pytest.approx(ref["logprob"], rel=1e-10)
        # engine passes (fp32 production kernels): optimistic attempt, refused, repaired
        eng.upload_batch(seqs)
        eng.ctx.set_option("defer_skip", 0)
        bad1 = eng.ctx.stat("deferred_bad")
        out = eng.posteriors(renorm_eps=False, want_map=True, want_post=False, precision="f32")
        vlp, vst = eng.viterbi(precision="f32")
        st = eng.estep(precision="f32")
        assert eng.ctx.stat("deferred_bad") > bad1
        for i, obs in enumerate(seqs):
            ref = oracle.sweep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"])
            assert out["logprob"][i] == pytest.approx(ref["logprob"], rel=1e-5)
            assert vlp[i] == pytest.approx(ref["vit_logprob"], rel=1e-6)
            assert_near_ties_only(vst[i], ref["vit_states"], oracle_frame(oracle, obs, m["table"]),
                                  m["log_start"], m["log_trans"])
        assert st["obs"].sum() == pytest.approx(sum(lens) * m["K"], rel=1e-5)
        # a healthy warm-up: the optimistic attempt stands (once the back-off after a refusal is over)
        assert eng.ctx.stat("defer_skip") > 0
        eng.ctx.set_option("defer_skip", 0)
        eng.ctx.set_option("warmup", 0)
        eng.upload_batch(seqs)
        bad2 = eng.ctx.stat("deferred_bad")
        checks2 = eng.ctx.stat("deferred_checks")
        vlp2, vst2 = eng.viterbi(precision="f32")
        assert eng.ctx.stat("deferred_bad") == bad2 and eng.ctx.stat("deferred_checks") > checks2
        for i in range(len(seqs)):
            assert_array_equal(vst2[i], vst[i])
    finally:
        for k in ("chunk_tiles", "warmup", "fine_len"):
            eng.ctx.set_option(k, 0)
