"""-m gpu: the batched chunked-parallel kernels (C ABI tehmm_run_*) against the
oracle and the reference's golden vectors.

Tolerances (north_star): float32 path <= 1e-5 relative on log-likelihood,
posteriors and expected counts; float64 verification mode <= 1e-10.  Viterbi
paths must be identical except at documented near-ties: wherever the path
differs, the float64 score of our path must equal the reference's score to the
same tolerance.
"""
import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

from conftest import golden, golden_names, ratios_of
from parity import (ATOL, TOL, assert_map_near_ties_only, assert_near_ties_only, min_rtol, oracle_all,
                    oracle_frame, trans_counts_extended)

pytestmark = pytest.mark.gpu


def engine(chunk_tiles=0, warmup=0, fine_len=0, tile=1):
    """chunk_tiles / warmup: the one-chunk-per-warp partition; fine_len / tile: the
    sixteen-chunks-per-warp tensor-core kernels (csrc/tile.cu), on by default"""
    from tehmm_b200.engine import get_engine
    eng = get_engine(0)
    eng.ctx.set_option("chunk_tiles", chunk_tiles)
    eng.ctx.set_option("warmup", warmup)
    eng.ctx.set_option("fine_len", fine_len)
    eng.ctx.set_option("tile", tile)
    return eng


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("name", golden_names("ll_"))
def test_golden_batched(name, prec):
    g = golden(name)
    if int(g["N"]) > 64:
        pytest.skip("batched path supports N <= 64")
    eng = engine(chunk_tiles=1, warmup=8)          # T is small: force several chunks
    r = ratios_of(g)
    widths = [int(s) + 1 for s in g["syms"]]
    eng.upload_model(g["log_start"], g["log_trans"], g["table"], float(g["normalize"]), widths)
    eng.upload_batch([g["obs"]])
    rl = None if r is None else [r]
    frames = eng.emission_frames(rl)
    assert_array_equal(frames[0], g["frame"])                   # float64 gather-sum is bit-exact
    out = eng.posteriors(ratios_em=rl, ratios_dp=rl, renorm_eps=False, want_map=True, precision=prec)
    assert out["logprob"][0] == pytest.approx(float(g["logprob"]), rel=TOL[prec])
    assert_allclose(out["post"][0], g["post"], rtol=TOL[prec], atol=ATOL[prec])
    lps, states = eng.viterbi(ratios_em=rl, ratios_dp=rl, precision=prec)
    if prec == "f64":
        assert_array_equal(states[0], g["vit_states"])
    else:
        assert_near_ties_only(states[0], g["vit_states"], g["frame"], g["log_start"], g["log_trans"], r, label=name)
    assert lps[0] == pytest.approx(float(g["vit_logprob"]), rel=1e-6 if prec == "f32" else 1e-10)
    st = eng.estep(ratios=rl, precision=prec)
    T = g["obs"].shape[0]
    assert st["logprob"] == pytest.approx(float(g["logprob"]), rel=TOL[prec])
    assert_allclose(st["start"], g["post"][0], rtol=TOL[prec], atol=ATOL[prec])
    if T > 1:
        assert_allclose(st["trans"], np.exp(g["lneta"]), rtol=TOL[prec], atol=ATOL[prec])
    assert_allclose(st["obs"], g["obs_stats"], rtol=TOL[prec], atol=ATOL[prec])


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("warmup", [1, 64])
def test_multi_sequence_ragged(oracle, prec, warmup):
    """ragged batch incl. T=1 and T=2 sequences; warmup=1 forces the repair path."""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=21)
    lens = [1, 2, 700, 65, 64, 1300, 129]
    obs = [synth.sample_obs(m, T, seed=30 + i)[0] for i, T in enumerate(lens)]
    eng = engine(chunk_tiles=2, warmup=warmup)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(obs)
    out = eng.posteriors(renorm_eps=True, want_map=True, precision=prec)
    lps, states = eng.viterbi(precision=prec)
    for i, o in enumerate(obs):
        ref = oracle_all(oracle, o, m["table"], 1.0, m["log_start"], m["log_trans"])
        assert out["logprob"][i] == pytest.approx(ref["logprob"], rel=TOL[prec])
        post = oracle.posteriors(ref["fwd"], ref["bwd"], renorm_eps=True)
        assert_allclose(out["post"][i], post, rtol=TOL[prec], atol=ATOL[prec])
        if prec == "f64":
            assert_array_equal(out["map_states"][i], np.argmax(post, axis=1))
        else:
            assert_map_near_ties_only(out["map_states"][i], post)
        assert out["map_score"][i] == pytest.approx(np.max(post, axis=1).sum(), rel=TOL[prec])
        if prec == "f64":
            assert_array_equal(states[i], ref["vit_states"])
        else:
            assert_near_ties_only(states[i], ref["vit_states"], ref["frame"], m["log_start"], m["log_trans"])
        assert lps[i] == pytest.approx(ref["vit_logprob"], rel=1e-6 if prec == "f32" else 1e-10)
    if warmup == 1:
        assert eng.ctx.stat("repair_passes_forward") > 0      # the repair path really ran


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_estep_matches_oracle(oracle, prec):
    """Device E-step == sum over sequences of the reference's per-sequence E-step."""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=41)
    lens = [3000, 500, 1, 2500]
    obs = [synth.sample_obs(m, T, seed=50 + i)[0] for i, T in enumerate(lens)]
    eng = engine(chunk_tiles=4, warmup=64)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(obs)
    st = eng.estep(precision=prec)
    K, N, S = m["table"].shape
    s0, tr, ob = np.zeros(N), np.zeros((N, N)), np.zeros((K, N, S))
    lp = 0.0
    for o in obs:
        lp += oracle.estep_sequence(o, m["table"], 1.0, m["log_start"], m["log_trans"], None, s0, tr, ob)
    assert st["logprob"] == pytest.approx(lp, rel=TOL[prec])
    assert st["nobs"] == len(obs)
    assert_allclose(st["start"], s0, rtol=TOL[prec], atol=ATOL[prec])
    if prec == "f32":
        assert_allclose(st["trans"], tr, rtol=TOL[prec], atol=ATOL[prec])
    else:
        # Documented divergence (DESIGN section 6): at T = 3000 the REFERENCE's float64 log-space lattices
        # carry ulp(|log alpha|) absolute rounding, 4.0e-10 relative on these counts against an
        # extended-precision (64-bit mantissa) evaluation; our scaled-space float64 kernels meet the 1e-10
        # contract against that arbiter and are within the reference's own error of the reference.
        truth = trans_counts_extended([oracle_frame(oracle, o, m["table"]) for o in obs],
                                      m["log_start"], m["log_trans"])
        assert_allclose(st["trans"], truth, rtol=TOL[prec], atol=ATOL[prec])
        assert min_rtol(tr, truth, ATOL[prec]) > TOL[prec]         # the reference itself is outside 1e-10 here
        assert_allclose(st["trans"], tr, rtol=1e-9, atol=ATOL[prec])
    assert_allclose(st["obs"], ob, rtol=TOL[prec], atol=ATOL[prec])
    # size-independent properties: posterior mass is conserved
    assert st["obs"].sum() == pytest.approx(sum(lens) * K, rel=1e-6)
    assert st["trans"].sum() * N == pytest.approx(sum(lens) - len(lens), rel=1e-6)


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("N", [12, 40])
def test_segment_ratios(oracle, prec, N):
    """ratios in the emission and in the DP, including the Viterbi from-state-0 quirk; N = 40: the
    two-states-per-lane kernels and the two-chunks-per-warp traceback with the quirk's correction."""
    from tehmm_b200 import synth
    m = synth.make_model(N=N, syms=(4, 8, 2), seed=61, zero_frac=0.0)
    T = 900
    obs = synth.sample_obs(m, T, seed=62)[0]
    r = np.random.RandomState(63).uniform(0.05, 6.0, size=T)
    eng = engine(chunk_tiles=2, warmup=64)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    ref = oracle_all(oracle, obs, m["table"], 1.0, m["log_start"], m["log_trans"], r_em=r, r_dp=r)
    out = eng.posteriors(ratios_em=[r], ratios_dp=[r], renorm_eps=False, precision=prec)
    assert out["logprob"][0] == pytest.approx(ref["logprob"], rel=TOL[prec])
    assert_allclose(out["post"][0], ref["post"], rtol=TOL[prec], atol=ATOL[prec])
    # decode(): emission WITHOUT ratios, DP with ratios (basehmm.py:327, hmm.py:674)
    ref2 = oracle_all(oracle, obs, m["table"], 1.0, m["log_start"], m["log_trans"], r_em=None, r_dp=r)
    lps, states = eng.viterbi(ratios_em=None, ratios_dp=[r], precision=prec)
    assert lps[0] == pytest.approx(ref2["vit_logprob"], rel=1e-6 if prec == "f32" else 1e-10)
    if prec == "f64":
        assert_array_equal(states[0], ref2["vit_states"])
    else:
        assert_near_ties_only(states[0], ref2["vit_states"], ref2["frame"], m["log_start"], m["log_trans"], r)
    # E-step with ratios
    K, N, S = m["table"].shape
    s0, tr, ob = np.zeros(N), np.zeros((N, N)), np.zeros((K, N, S))
    oracle.estep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"], r, s0, tr, ob)
    st = eng.estep(ratios=[r], precision=prec)
    assert_allclose(st["trans"], tr, rtol=TOL[prec], atol=ATOL[prec])
    assert_allclose(st["obs"], ob, rtol=TOL[prec], atol=ATOL[prec])


def test_wide_model_50_states(oracle):
    """N = 50 (two states per lane), int32 symbols."""
    from tehmm_b200 import synth
    m = synth.make_model(N=50, syms=(4, 8, 2, 2), seed=71)
    obs = synth.sample_obs(m, 1500, seed=72, dtype=np.int32)[0]
    eng = engine(chunk_tiles=4, warmup=64)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    ref = oracle_all(oracle, obs, m["table"], 1.0, m["log_start"], m["log_trans"])
    for prec in ("f64", "f32"):
        out = eng.posteriors(renorm_eps=False, precision=prec)
        assert out["logprob"][0] == pytest.approx(ref["logprob"], rel=TOL[prec])
        assert_allclose(out["post"][0], ref["post"], rtol=TOL[prec], atol=ATOL[prec])
        lps, states = eng.viterbi(precision=prec)
        assert lps[0] == pytest.approx(ref["vit_logprob"], rel=1e-6)
        if prec == "f64":
            assert_array_equal(states[0], ref["vit_states"])
        else:
            assert_near_ties_only(states[0], ref["vit_states"], ref["frame"], m["log_start"], m["log_trans"])
    st = eng.estep(precision="f32")
    K, N, S = m["table"].shape
    s0, tr, ob = np.zeros(N), np.zeros((N, N)), np.zeros((K, N, S))
    oracle.estep_sequence(obs, m["table"], 1.0, m["log_start"], m["log_trans"], None, s0, tr, ob)
    assert_allclose(st["trans"], tr, rtol=TOL["f32"], atol=ATOL["f32"])
    assert_allclose(st["obs"], ob, rtol=TOL["f32"], atol=ATOL["f32"])


@pytest.mark.parametrize("N", [33, 64])
@pytest.mark.parametrize("warmup", [1, 64])
def test_wide_viterbi_two_warps_per_chunk_ragged(oracle, N, warmup):
    """33..64 states, float32: viterbi_wide_kernel (two warps per chunk, lazily normalised rows) and the
    two-chunks-per-warp traceback on a ragged multi-sequence batch incl. T = 1 and T = 2; warmup = 1 forces
    the repair passes (mode 1 of both kernels).  Paths equal the oracle's except at float32 near-ties."""
    from tehmm_b200 import synth
    m = synth.make_model(N=N, seed=500 + N)
    lens = [1, 2, 900, 65, 64, 1700, 131]
    obs = [synth.sample_obs(m, T, seed=510 + i)[0] for i, T in enumerate(lens)]
    eng = engine(chunk_tiles=2, warmup=warmup, fine_len=96)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(obs)
    before = eng.ctx.stat("repair_passes_viterbi") + eng.ctx.stat("repair_passes_traceback")
    lps, states = eng.viterbi(precision="f32")
    for i, o in enumerate(obs):
        ref = oracle_all(oracle, o, m["table"], 1.0, m["log_start"], m["log_trans"])
        assert_near_ties_only(states[i], ref["vit_states"], ref["frame"], m["log_start"], m["log_trans"])
        assert lps[i] == pytest.approx(ref["vit_logprob"], rel=1e-6)
    if warmup == 1:
        assert eng.ctx.stat("repair_passes_viterbi") + eng.ctx.stat("repair_passes_traceback") > before


@pytest.mark.parametrize("N", [33, 50, 64])
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16])
def test_wide_emission_merged_tables(oracle, N, dtype):
    """33..64 states, float32: the merged-table emission kernel with 64-float rows
    (emission_merged_kernel<.., NS = 2>) against _emission.pyx:20-144 -- elog + rowmax must
    give the reference frame, blin = exp(elog); also with an out-of-table symbol in the
    batch (dense float64 table fallback) and with segment ratios."""
    from tehmm_b200 import synth
    m = synth.make_model(N=N, seed=300 + N)
    lens = [700, 1, 37, 1200]
    obs = [synth.sample_obs(m, T, seed=310 + i, dtype=dtype)[0] for i, T in enumerate(lens)]
    # a symbol beyond its track's table but inside the dense table's width (log-prob LOGZERO rows exist there)
    k_small = int(np.argmin(m["syms"]))
    if m["syms"][k_small] + 1 < m["table"].shape[2]:
        obs[3][600, k_small] = m["syms"][k_small] + 1
    rng = np.random.RandomState(5)
    ratios = [np.where(rng.rand(T) < 0.3, rng.uniform(1.0, 3.0, size=T), 1.0) for T in lens]
    eng = engine(chunk_tiles=4, warmup=64)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(obs)
    prec, tdt = eng._prec("f32")
    LD = eng.LD
    for use_ratios in (False, True):
        d_r = eng.upload_ratios(ratios) if use_ratios else None
        elog, blin, rowmax = eng.run_emission(prec, tdt, d_r, True, True)
        elog = elog.cpu().numpy().reshape(-1, LD)[:, :N].astype(np.float64)
        blin = blin.cpu().numpy().reshape(-1, LD)[:, :N].astype(np.float64)
        rowmax = rowmax.cpu().numpy()
        a = 0
        for o, r in zip(obs, ratios):
            T = o.shape[0]
            frame = np.zeros((T, N))
            oracle.fastAllLogProbs(o, m["table"], frame, 1.0, r if use_ratios else None)
            got = elog[a:a + T] + rowmax[a:a + T, None]
            live = frame > -1e50                     # LOGZERO entries: only "far below the maximum" matters
            assert_allclose(got[live], frame[live], rtol=2e-6, atol=2e-5)
            assert np.all(got[~live] < -1e30) or np.all(elog[a:a + T][~live] < -80)
            # the maximum taken out: float32 merged-table rounding (6e-8 relative) on top of the float64 common part
            assert_allclose(rowmax[a:a + T], frame.max(axis=1), rtol=1e-6, atol=2e-5)
            # ex2.approx of a float32 argument: ~1e-7 near the maximum, a few 1e-6 relative 60 units below it
            assert_allclose(blin[a:a + T], np.exp(elog[a:a + T]), rtol=1e-5, atol=1e-12)
            a += T


def test_f32_vs_f64_at_scale():
    """T = 2e6 (oracle would take minutes): float32 production path against the
    float64 verification path on the GPU, plus size-independent invariants."""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=81)
    T = 2_000_000
    obs = synth.sample_obs(m, T, seed=82)[0]
    eng = engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    a = eng.posteriors(renorm_eps=False, want_map=True, want_post=False, precision="f64")
    before = {k: eng.ctx.stat("repaired_chunks_" + k) for k in ("forward", "backward", "viterbi")}
    b = eng.posteriors(renorm_eps=False, want_map=True, want_post=False, precision="f32")
    assert b["logprob"][0] == pytest.approx(a["logprob"][0], rel=1e-7)
    assert np.mean(a["map_states"][0] == b["map_states"][0]) > 0.9995
    lp64, s64 = eng.viterbi(precision="f64")
    lp32, s32 = eng.viterbi(precision="f32")
    assert lp32[0] == pytest.approx(lp64[0], rel=1e-7)          # near-ties only
    assert np.mean(s64[0] == s32[0]) > 0.995
    assert lp64[0] <= a["logprob"][0]                            # best path <= total probability
    st = eng.estep(precision="f32")
    assert st["obs"].sum() == pytest.approx(T * m["K"], rel=1e-6)
    assert st["trans"].sum() * m["N"] == pytest.approx(T - 1, rel=1e-6)
    assert st["start"].sum() == pytest.approx(1.0, rel=1e-6)
    # the speculative warm-up must be good enough that (almost) nothing is repaired
    nchunks = eng.ctx.stat("chunks")
    for k in before:
        assert eng.ctx.stat("repaired_chunks_" + k) - before[k] <= 0.02 * nchunks, k


# ---------------------------------------------------------------- tensor-core tile kernels
@pytest.mark.parametrize("N", [2, 5, 30, 32])
@pytest.mark.parametrize("warmup,fine_len", [(8, 16), (1, 24), (64, 0)])
def test_tile_kernels_ragged(oracle, N, warmup, fine_len):
    """csrc/tile.cu (fp32, 16 chunks per warp on the tensor cores) against the oracle:
    ragged batch, chunks shorter / longer than the warm-up, sequence starts and ends
    inside the warm-up window, partial tiles, the repair path (warmup=1)."""
    from tehmm_b200 import synth
    syms = (4, 8, 2) if N < 30 else synth.BENCH_SYMS
    m = synth.make_model(N=N, syms=syms, seed=100 + N)
    lens = [1, 2, 700, 65, 17, 1300, 129, 3, 40]
    obs = [synth.sample_obs(m, T, seed=130 + i)[0] for i, T in enumerate(lens)]
    eng = engine(chunk_tiles=2, warmup=warmup, fine_len=fine_len, tile=1)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(obs)
    before = eng.ctx.stat("tile_passes")
    out = eng.posteriors(renorm_eps=True, want_map=True, precision="f32")
    assert eng.ctx.stat("tile_passes") >= before + 2          # the tile kernels really ran
    for i, o in enumerate(obs):
        ref = oracle_all(oracle, o, m["table"], 1.0, m["log_start"], m["log_trans"])
        assert out["logprob"][i] == pytest.approx(ref["logprob"], rel=TOL["f32"])
        post = oracle.posteriors(ref["fwd"], ref["bwd"], renorm_eps=True)
        assert_allclose(out["post"][i], post, rtol=TOL["f32"], atol=ATOL["f32"])
        assert_map_near_ties_only(out["map_states"][i], post)
        assert out["map_score"][i] == pytest.approx(np.max(post, axis=1).sum(), rel=TOL["f32"])
    if warmup == 1 and N >= 5:
        assert eng.ctx.stat("repair_passes_forward") > 0
    # score-only (no alpha lattice) and MAP-only variants
    lp = eng.score(precision="f32")
    assert_allclose(lp, out["logprob"], rtol=1e-12)
    mo = eng.posteriors(renorm_eps=False, want_map=True, want_post=False, precision="f32")
    for i in range(len(obs)):
        assert np.mean(mo["map_states"][i] == out["map_states"][i]) >= 0.995


def test_tile_and_warp_kernels_interoperate(oracle):
    """forward by one implementation, backward by the other: same alpha lattice
    conventions (canonical power-of-two scaling), same posteriors."""
    from tehmm_b200 import _lib, synth
    m = synth.make_model(N=30, seed=151)
    obs = [synth.sample_obs(m, T, seed=160 + i)[0] for i, T in enumerate([900, 2100, 77])]
    res = {}
    for fwd_tile in (0, 1):
        for bwd_tile in (0, 1):
            eng = engine(chunk_tiles=2, warmup=32, fine_len=48, tile=fwd_tile)
            eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
            eng.upload_batch(obs)
            prec, tdt = eng._prec("f32")
            _, blin, rowmax = eng.run_emission(prec, tdt, None, False, True)
            alpha, logprob = eng.run_forward(prec, tdt, blin, rowmax, None)
            eng.ctx.set_option("tile", bwd_tile)
            post, _, _ = eng.run_backward(prec, tdt, _lib.BWD_POSTERIORS, blin, alpha, None)
            res[(fwd_tile, bwd_tile)] = (logprob.cpu().numpy(), post.cpu().numpy())
    eng.ctx.set_option("tile", 1)
    base = res[(0, 0)]
    for key, (lp, post) in res.items():
        assert_allclose(lp, base[0], rtol=1e-7)
        assert_allclose(post, base[1], rtol=TOL["f32"], atol=ATOL["f32"])


def test_xi_tensor_core_kernel_vs_cuda_core_and_f64():
    """Expected transition counts: the tensor-core xi kernel (two dense products per 16 steps,
    csrc/tile.cu) against the one-chunk-per-warp accumulation it replaces and against the
    float64 verification mode, at a size where per-entry counts span six decades; and the
    size-independent conservation law sum(xi) * N == (steps - sequences)  (1/N: _hmm.pyx:179)."""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=8)
    lens = [250_000, 17, 64_001, 5]
    obs = [synth.sample_obs(m, T, seed=70 + i)[0] for i, T in enumerate(lens)]
    eng = engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch(obs)
    ref = eng.estep(precision="f64")
    eng.ctx.set_option("tile", 0)
    scan = eng.estep(precision="f32")
    eng.ctx.set_option("tile", 1)
    before = eng.ctx.stat("launches")
    tile = eng.estep(precision="f32")
    assert eng.ctx.stat("launches") > before
    N = 30
    for st in (scan, tile):
        assert_allclose(st["trans"], ref["trans"], rtol=1e-5, atol=2e-6)
        assert_allclose(st["start"], ref["start"], rtol=1e-5, atol=2e-6)
        assert st["trans"].sum() * N == pytest.approx(sum(lens) - len(lens), rel=1e-6)
    assert_allclose(tile["obs"], scan["obs"], rtol=1e-5, atol=2e-6)
    # zero transitions of the model stay exactly zero
    assert np.all(tile["trans"][m["A"] == 0] == 0)


@pytest.mark.parametrize("fine_len,warmup", [(0, 0), (64, 64), (96, 64), (64, 128), (200, 32)])
def test_forward_tensor_map_blocks_single_sequence(oracle, fine_len, warmup):
    """fwd_tile_kernel moves whole blocks with one 3-D tensor-map copy when the batch is ONE
    regularly chunked sequence (warm-up clocks read the box one chunk up; the last, ragged tile
    and warm-ups longer than a chunk take the per-row copies): log-likelihood, posteriors and
    MAP path against the oracle and against the one-chunk-per-warp kernels."""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=21)
    T = 40_003                                      # not a multiple of any chunk length
    obs, _ = synth.sample_obs(m, T, seed=22)
    ref = oracle_all(oracle, obs, m["table"], 1.0, m["log_start"], m["log_trans"])
    eng = engine(fine_len=fine_len, warmup=warmup, tile=1)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    before = eng.ctx.stat("tile_passes")
    out = eng.posteriors(renorm_eps=False, want_map=True, precision="f32")
    assert eng.ctx.stat("tile_passes") > before
    assert out["logprob"][0] == pytest.approx(ref["logprob"], rel=TOL["f32"])
    assert_allclose(out["post"][0], ref["post"], rtol=TOL["f32"], atol=ATOL["f32"])
    eng2 = engine(fine_len=fine_len, warmup=warmup, tile=0)
    eng2.upload_batch([obs])
    scan = eng2.posteriors(renorm_eps=False, want_map=True, precision="f32")
    assert scan["logprob"][0] == pytest.approx(out["logprob"][0], rel=1e-6)
    assert np.mean(scan["map_states"][0] == out["map_states"][0]) > 0.999


@pytest.mark.parametrize("fine_len,warmup", [(0, 0), (96, 64), (200, 32), (64, 64), (66, 2), (128, 126)])
def test_backward_tile_kernel_single_sequence(oracle, fine_len, warmup):
    """bwd_tile_kernel on ONE regularly chunked sequence whose forward pass took the tensor-map
    blocks: regular and ragged tiles, the sequence end and warm-ups that do not fit a chunk.
    Posteriors against the oracle (basehmm.py:265-272,332-359)."""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=23)
    T = 70_011
    obs, _ = synth.sample_obs(m, T, seed=24)
    ref = oracle_all(oracle, obs, m["table"], 1.0, m["log_start"], m["log_trans"])
    eng = engine(fine_len=fine_len, warmup=warmup, tile=1)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    before = eng.ctx.stat("tile_passes")
    out = eng.posteriors(renorm_eps=False, want_map=True, precision="f32")
    assert eng.ctx.stat("tile_passes") > before
    assert_allclose(out["post"][0], ref["post"], rtol=TOL["f32"], atol=ATOL["f32"])


def test_full_size_c2_properties(oracle):
    """BASELINE.json configs[1] at FULL size (one sequence of 10 M steps, 30 states, 10 tracks):
    the oracle cannot run this in seconds, so the checks are the size-independent ones --
    conservation laws of the E-step, Viterbi score <= log-likelihood, the float64 score of
    the returned path recomputed on the host, prefix consistency (paths coalesce), no repairs
    -- plus the oracle on a 200 k prefix."""
    from tehmm_b200 import synth
    m = synth.make_model(N=30, seed=0)
    T = 10_000_000
    obs, _ = synth.sample_obs(m, T, seed=1)
    eng = engine()
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    kinds = ("forward", "backward", "viterbi", "traceback")
    before = {k: eng.ctx.stat("repaired_chunks_" + k) for k in kinds}     # counters are per context, cumulative
    lps, states = eng.viterbi()
    out = eng.posteriors(renorm_eps=True, want_post=False, want_map=True)
    st = eng.estep()
    K, N = m["K"], m["N"]
    path = states[0]
    assert path.shape == (T,) and path.dtype == np.int64 and path.min() >= 0 and path.max() < N
    assert lps[0] <= out["logprob"][0] < 0
    assert 0.9 * T < out["map_score"][0] <= T * (1 + 1e-6)
    assert st["logprob"] == pytest.approx(out["logprob"][0], rel=1e-9)
    assert st["obs"].sum() == pytest.approx(T * K, rel=1e-6)          # every step adds one unit per track
    assert st["trans"].sum() * N == pytest.approx(T - 1, rel=1e-6)    # (1/N: _hmm.pyx:179)
    assert st["start"].sum() * 1.0 == pytest.approx(1.0, rel=1e-5)
    assert np.all(st["trans"][m["A"] == 0] == 0)
    for k in kinds:
        assert eng.ctx.stat("repaired_chunks_" + k) == before[k]
    # float64 score of the returned path, recomputed on the host from the reference-layout tables
    idx = np.arange(T)
    e = np.zeros(T)
    for k in range(K):
        e += m["table"][k, path, obs[:, k]]
    score = m["log_start"][path[0]] + e.sum() + m["log_trans"][path[:-1], path[1:]].sum()
    # the returned log-probability is the fp32 DP's own value (row maxima summed in float64): the
    # reference's viterbi_lattice[T-1, argmax] up to the DP's rounding, ~1e-10 relative at this size;
    # option "rescore" returns the float64 score of the returned path instead (exact to summation order)
    assert lps[0] == pytest.approx(score, rel=1e-8)
    eng.ctx.set_option("rescore", 1)
    try:
        lps_x, states_x = eng.viterbi()
    finally:
        eng.ctx.set_option("rescore", 0)
    assert_array_equal(states_x[0], path)
    assert lps_x[0] == pytest.approx(score, rel=1e-11)
    print("viterbi log-prob: DP %.6f, float64 re-score %.6f, rel. diff %.2e" % (
        lps[0], lps_x[0], abs(lps[0] - lps_x[0]) / abs(lps_x[0])))
    # prefix: the first 150 k states of the 10 M decode == those of a stand-alone 200 k decode == the oracle's
    n0 = 200_000
    ref = oracle.sweep_sequence(obs[:n0], m["table"], 1.0, m["log_start"], m["log_trans"])
    assert_array_equal(path[:150_000], ref["vit_states"][:150_000])
    assert np.mean(out["map_states"][0][:150_000] == ref["map_states"][:150_000]) > 0.9999


@pytest.mark.parametrize("N,T", [(33, 60_011), (50, 60_000), (50, 60_100), (64, 45_020)])
def test_tcgen05_kernels_vs_cuda_core_for_33_to_64_states(oracle, N, T):
    """fwd_umma_kernel and its backward twin bwd_umma_kernel (csrc/umma.cu; default unless option "tile" is 0):
    the forward pass and the backward / posterior / MAP pass of a single-sequence batch of 33..64 states on
    tcgen05.mma M128 N64 K8 with two threads per chunk.  Same log-likelihood, posteriors and MAP path as the
    oracle and as the one-chunk-per-warp kernels -- with no ragged last chunk (60 000 = 400 x 150), one shorter
    than the warm-up (11, 20 steps) and one longer (100); multi-sequence batches stay on the generic kernels."""
    from tehmm_b200 import synth
    m = synth.make_model(N=N, seed=41)
    obs, _ = synth.sample_obs(m, T, seed=42)
    ref = oracle_all(oracle, obs, m["table"], 1.0, m["log_start"], m["log_trans"])
    eng = engine(fine_len=150)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    before, repairs = eng.ctx.stat("umma_passes"), eng.ctx.stat("repair_passes_backward")
    out = eng.posteriors(renorm_eps=False, want_map=True, precision="f32")
    assert eng.ctx.stat("umma_passes") == before + 2             # forward and backward
    only_map = eng.posteriors(renorm_eps=False, want_post=False, want_map=True, precision="f32")
    assert eng.ctx.stat("umma_passes") == before + 4
    eps = eng.posteriors(renorm_eps=True, want_map=True, precision="f32")
    eng.ctx.set_option("tile", 0)
    try:
        base = eng.posteriors(renorm_eps=False, want_map=True, precision="f32")
        base_eps = eng.posteriors(renorm_eps=True, want_map=True, precision="f32")
    finally:
        eng.ctx.set_option("tile", 1)
    assert eng.ctx.stat("umma_passes") == before + 6
    assert eng.ctx.stat("repair_passes_backward") == repairs
    assert out["logprob"][0] == pytest.approx(ref["logprob"], rel=TOL["f32"])
    assert_allclose(out["post"][0], ref["post"], rtol=TOL["f32"], atol=ATOL["f32"])
    assert out["logprob"][0] == pytest.approx(base["logprob"][0], rel=1e-7)
    assert_map_near_ties_only(out["map_states"][0], ref["post"], label="tcgen05 N=%d" % N)
    assert np.array_equal(only_map["map_states"][0], out["map_states"][0])
    assert_allclose(eps["post"][0], base_eps["post"][0], rtol=TOL["f32"], atol=ATOL["f32"])
    for key in ("map_score", "map_logprob"):
        if key in out:
            assert_allclose(np.asarray(out[key]), np.asarray(base[key]), rtol=1e-6)
            assert_allclose(np.asarray(eps[key]), np.asarray(base_eps[key]), rtol=1e-6)
    # two sequences: not a regular [chunk][step][64] array, the tcgen05 kernels do not apply
    eng.upload_batch([obs[:20_000], obs[20_000:]])
    eng.posteriors(renorm_eps=False, want_post=False, want_map=True, precision="f32")
    assert eng.ctx.stat("umma_passes") == before + 6


def test_tcgen05_kernels_several_tiles_per_cta_vs_cuda_core():
    """More tiles of 128 chunks than SMs (1.3 M steps in chunks of 64: 159 tiles): a CTA of fwd_umma_kernel /
    bwd_umma_kernel walks a second tile with the same barriers, tensor-memory columns and shared-memory rings.
    Against the one-chunk-per-warp kernels on the same partition."""
    from tehmm_b200 import synth
    m = synth.make_model(N=50, seed=43)
    T = 1_300_000
    obs, _ = synth.sample_obs(m, T, seed=44)
    eng = engine(fine_len=64)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.upload_batch([obs])
    before = eng.ctx.stat("umma_passes")
    out = eng.posteriors(renorm_eps=False, want_post=True, want_map=True, precision="f32")
    assert eng.ctx.stat("umma_passes") == before + 2
    eng.ctx.set_option("tile", 0)
    try:
        base = eng.posteriors(renorm_eps=False, want_post=True, want_map=True, precision="f32")
    finally:
        eng.ctx.set_option("tile", 1)
    assert out["logprob"][0] == pytest.approx(base["logprob"][0], rel=1e-7)
    assert np.mean(out["map_states"][0] == base["map_states"][0]) > 0.99999
    assert_allclose(out["map_score"], base["map_score"], rtol=1e-6)
    # float32 against float32: a few ulp of the posterior's own magnitude
    assert_allclose(out["post"][0], base["post"][0], rtol=2e-4, atol=1e-6)
