"""Supervised training in one device pass (tehmm_supervised_counts, Engine.supervised_counts,
IndependentMultinomialEmissionModel / MultitrackHmm.supervisedTrain) against the per-interval path:
a restatement of the reference's loops over _emission.fastUpdateCounts (emission.py:293-331,
hmm.py:174-210) and the CPU oracle's fastUpdateCounts.  Counts are compared bit for bit.  The host
mapping of intervals to table rows is checked without a GPU."""
import types

import numpy as np
import pytest
from numpy.testing import assert_array_equal

from conftest import golden

gpu = pytest.mark.gpu


# ------------------------------------------------------------------ fixtures
def make_tables(rng, dtype, layout, segmented=(), nsym=(3, 5, 2)):
    """IntegerTrackTables of the (chrom, start, end) layout; those listed in `segmented` are cut
    into segments on the host (setSegments)"""
    from tehmm_b200.track import IntegerTrackTable
    tables = []
    for i, (chrom, start, end) in enumerate(layout):
        t = IntegerTrackTable(len(nsym), chrom, start, end, dtype=dtype)
        for k, s in enumerate(nsym):
            t.data[:, k] = rng.randint(0, s + 1, size=end - start)
        if i in segmented:
            offs = np.unique(np.concatenate([[0], rng.randint(1, end - start, size=(end - start) // 7)]))
            t.setSegments(offs)
        tables.append(t)
    return tables


LAYOUT = [("chr2", 0, 300), ("chr2", 300, 700), ("chr2", 900, 1000), ("chr1", 50, 450), ("chr1", 450, 460),
          ("chr3", 0, 2000)]


def random_intervals(rng, n, N, layout=LAYOUT, sort=True):
    """labelled intervals: inside tables, across two tables, in gaps, outside every table, empty"""
    out = []
    chroms = sorted(set(c for c, _, _ in layout)) + ["chrX"]
    for _ in range(n):
        c = chroms[rng.randint(len(chroms))]
        s = int(rng.randint(0, 2100))
        e = s + int(rng.choice([0, 1, 3, 40, 250, 700]))
        if e == s:          # an empty interval at a segment start is an assertion in the reference's scan
            c, s, e = layout[0][0], layout[0][1] + s % 50, layout[0][1] + s % 50
        out.append((c, s, e, int(rng.randint(N))))
    if sort:
        out.sort(key=lambda iv: (iv[0], iv[1]))
    return out


def reference_emission_counts(model, tables, intervals, update):
    """emission.py:293-331 statement for statement, `update` standing for fastUpdateCounts"""
    obsStats = model.initStats()
    lastTable, lastRatios = None, None
    lastHit = 0
    lastOverlapEnd = -1
    for interval in intervals:
        hit = False
        for tableIdx in range(lastHit, len(tables)):
            table = tables[tableIdx]
            overlap = table.getOverlapInTableCoords(interval, lastOverlapEnd)
            if overlap is not None:
                lastHit = tableIdx
                hit = True
                lastOverlapEnd = max(0, overlap[2] - 1)
                if table is not lastTable:
                    lastRatios = model.getSegmentRatios(table)
                    lastTable = table
                update(overlap, table, obsStats, lastRatios)
            elif hit is True:
                break
    return obsStats


def batched_emission_counts(model, tables, intervals):
    """the obsStats supervisedTrain hands to maximize"""
    seen = {}
    model.maximize = lambda obsStats, trackList=None: seen.setdefault("stats", obsStats.copy())
    model.validate = lambda: None
    model.supervisedTrain(types.SimpleNamespace(getTrackTableList=lambda: tables, getTrackList=lambda: None),
                          intervals)
    return seen["stats"]


def make_model(N, nsym, fudge, eff=None):
    from tehmm_b200.emission import IndependentMultinomialEmissionModel
    return IndependentMultinomialEmissionModel(N, list(nsym), fudge=fudge, effectiveSegmentLength=eff)


# ------------------------------------------------------------------ host mapping (no GPU)
@pytest.mark.parametrize("seed", range(6))
def test_interval_triples_match_the_scan(seed):
    from tehmm_b200 import supervised
    rng = np.random.RandomState(seed)
    tables = make_tables(rng, np.uint8, LAYOUT, segmented=(1, 3, 5))
    for sort in (True, False):
        intervals = random_intervals(rng, 300, 4, sort=sort)
        fast = supervised.interval_triples(tables, intervals)
        slow = supervised._scan(tables, intervals)
        for a, b in zip(fast, slow):
            assert_array_equal(a, b)


def test_interval_triples_chromosome_order_quirk():
    """tables chr2 then chr1, intervals chr1 then chr2: lastHit has passed the chr2 tables when the
    chr2 intervals come, so they count nothing"""
    from tehmm_b200 import supervised
    rng = np.random.RandomState(1)
    tables = make_tables(rng, np.uint8, [("chr2", 0, 100), ("chr1", 0, 100)])
    intervals = [("chr1", 10, 20, 0), ("chr2", 10, 20, 1)]
    tix, lo, hi, st = supervised.interval_triples(tables, intervals)
    assert_array_equal(tix, [1])
    assert_array_equal(np.stack([lo, hi, st]), [[10], [20], [0]])
    for a, b in zip(supervised.interval_triples(tables, intervals), supervised._scan(tables, intervals)):
        assert_array_equal(a, b)


def test_interval_triples_other_layouts_use_the_scan():
    """overlapping tables of one chromosome are outside the vectorised layout: same triples"""
    from tehmm_b200 import supervised
    rng = np.random.RandomState(2)
    tables = make_tables(rng, np.uint8, [("chr1", 0, 100), ("chr1", 50, 150), ("chr2", 0, 10), ("chr1", 200, 300)])
    intervals = random_intervals(rng, 100, 3, layout=[("chr1", 0, 300), ("chr2", 0, 10)])
    assert supervised._chrom_blocks(tables)[0] is None
    for a, b in zip(supervised.interval_triples(tables, intervals), supervised._scan(tables, intervals)):
        assert_array_equal(a, b)


def reference_hmm_counts(N, fudge, intervals):
    """hmm.py:174-210's counting loop"""
    transitionCount = fudge + np.zeros((N, N), np.float64)
    freqCount = fudge + np.zeros((N,), np.float64)
    prev = None
    for interval in intervals:
        state = int(interval[3])
        assert state < N
        transitionCount[state, state] += interval[2] - interval[1] - 1
        freqCount[state] += interval[2] - interval[1]
        if prev is not None and prev[0] == interval[0]:
            if interval[1] < prev[2]:
                raise RuntimeError("Overlapping or out of order training intervals detected: "
                                   "%s and %s." % (str(prev), str(interval)))
            elif interval[1] == prev[2]:
                transitionCount[prev[3], state] += 1
        prev = interval
    return transitionCount, freqCount


def tiling(rng, N, n, chroms=("chr1", "chr2")):
    """sorted, disjoint intervals, many of them abutting"""
    out = []
    for c in chroms:
        pos = 0
        for _ in range(n):
            e = pos + int(rng.randint(1, 60))
            out.append((c, pos, e, int(rng.randint(N))))
            pos = e + (int(rng.randint(0, 5)) if rng.rand() < 0.3 else 0)
    return out


# ------------------------------------------------------------------ GPU
@gpu
def test_golden_counts_batched():
    from tehmm_b200.engine import get_engine
    g = golden("counts")
    N = int(g["N"])
    syms = g["syms"]
    S = int(syms.max()) + 1
    eng = get_engine(0)
    eng.upload_batch([g["obs"]])
    iv = g["intervals"]
    for key, r in (("stats", None), ("stats_ratio", g["ratios"])):
        stats = np.zeros((len(syms), N, S))
        for k, s in enumerate(syms):
            stats[k, :, :s + 1] += 1.0
        eng.supervised_counts(iv[:, 0], iv[:, 1], iv[:, 2], stats, r)
        assert_array_equal(stats, g[key])


@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int32])
@pytest.mark.parametrize("fudge", [0.0, 0.1])
def test_emission_supervised_train_matches_per_interval(dtype, fudge, oracle):
    from tehmm_b200 import _emission
    rng = np.random.RandomState(7 + int(fudge * 10))
    N, nsym = 5, (3, 5, 2)
    tables = make_tables(rng, dtype, LAYOUT, segmented=(1, 3))
    for eff, sort in ((None, True), (4, True), (4, False)):
        intervals = random_intervals(rng, 400, N, sort=sort)
        model = make_model(N, nsym, fudge, eff)
        new = batched_emission_counts(model, tables, intervals)
        old = reference_emission_counts(model, tables, intervals, _emission.fastUpdateCounts)

        def orc(overlap, table, stats, ratios):
            oracle.fastUpdateCounts(overlap, table.getNumPyArray(), stats, ratios)
        cpu = reference_emission_counts(model, tables, intervals, orc)
        assert_array_equal(new, old)
        assert_array_equal(new, cpu)


@gpu
def test_emission_supervised_train_chromosome_order_quirk():
    from tehmm_b200 import _emission
    rng = np.random.RandomState(3)
    tables = make_tables(rng, np.uint8, [("chr2", 0, 500), ("chr2", 500, 900), ("chr1", 0, 800)], segmented=(1,))
    intervals = random_intervals(rng, 60, 3, layout=[("chr1", 0, 800)], sort=True)
    intervals = [iv for iv in intervals if iv[0] == "chr1"] + [("chr2", 100, 800, 2), ("chr2", 10, 20, 1)]
    model = make_model(3, (3, 5, 2), 0.1, 3)
    assert_array_equal(batched_emission_counts(model, tables, intervals),
                       reference_emission_counts(model, tables, intervals, _emission.fastUpdateCounts))


@gpu
@pytest.mark.parametrize("fudge", [0.0, 0.1])
def test_one_interval_of_ten_million_rows(fudge):
    from tehmm_b200 import _emission
    rng = np.random.RandomState(11)
    T = 10_000_000
    tables = make_tables(rng, np.uint8, [("chr1", 0, T)], nsym=(3, 6))
    intervals = [("chr1", 0, T, 2)]
    model = make_model(4, (3, 6), fudge)
    assert_array_equal(batched_emission_counts(model, tables, intervals),
                       reference_emission_counts(model, tables, intervals, _emission.fastUpdateCounts))


@gpu
@pytest.mark.parametrize("fudge", [0.0, 0.25])
def test_hmm_supervised_train_matches_loops(fudge):
    from tehmm_b200 import _emission
    from tehmm_b200.common import myLog
    from tehmm_b200.hmm import MultitrackHmm
    rng = np.random.RandomState(4)
    N, nsym = 4, (3, 5, 2)
    tables = make_tables(rng, np.uint8, [("chr1", 0, 3000), ("chr2", 0, 3000)])
    intervals = tiling(rng, N, 60)
    td = types.SimpleNamespace(getTrackTableList=lambda: tables, getTrackList=lambda: None)
    model = make_model(N, nsym, fudge)
    hmm = MultitrackHmm(model, fudge=fudge)
    hmm.supervisedTrain(td, intervals)
    trans, freq = reference_hmm_counts(N, fudge, intervals)
    for row in range(N):
        trans[row] /= np.sum(trans[row])
    freq /= np.sum(freq)
    want = MultitrackHmm(make_model(N, nsym, fudge), fudge=fudge)
    want.transmat_ = np.copy(trans)         # the property setters store logs; the getters exponentiate
    want._log_transmat = myLog(trans)
    want.startprob_ = freq
    assert_array_equal(hmm._log_transmat, want._log_transmat)
    assert_array_equal(hmm.transmat_, want.transmat_)
    assert_array_equal(hmm.startprob_, want.startprob_)
    ref = make_model(N, nsym, fudge)
    ref.maximize(reference_emission_counts(ref, tables, intervals, _emission.fastUpdateCounts))
    assert_array_equal(model.getLogProbs(), ref.getLogProbs())


@gpu
def test_hmm_supervised_train_errors():
    from tehmm_b200.hmm import MultitrackHmm
    rng = np.random.RandomState(5)
    tables = make_tables(rng, np.uint8, [("chr1", 0, 1000)])
    td = types.SimpleNamespace(getTrackTableList=lambda: tables, getTrackList=lambda: None)
    cases = [
        [("chr1", 0, 10, 0), ("chr1", 20, 30, 1), ("chr1", 25, 40, 1), ("chr1", 5, 8, 0)],   # overlap first
        [("chr1", 0, 10, 0), ("chr1", 20, 30, 9), ("chr1", 25, 40, 1)],                     # bad state first
        [("chr1", 0, 10, 0), ("chr1", 20, 30, 1), ("chr1", 25, 40, 9)],                     # same interval: assert
        [("chr1", 50, 60, 0), ("chr2", 0, 10, 1), ("chr1", 0, 10, 2), ("chr1", 5, 9, 1)],
    ]
    for ivs in cases:
        with pytest.raises((RuntimeError, AssertionError)) as want:
            reference_hmm_counts(3, 0.0, ivs)
        with pytest.raises(want.type) as got:
            MultitrackHmm(make_model(3, (3, 5, 2), 0.0)).supervisedTrain(td, ivs)
        assert type(got.value) is want.type
        if want.type is RuntimeError:       # (pytest rewrites the restatement's bare assert with a message)
            assert str(got.value) == str(want.value)


@gpu
def test_level3_pipeline_supervised_counts(tmp_path):
    """BED -> device table -> segments -> compressed table -> supervised_counts, no table on the host
    side of the counting; equals the host path on the same tables"""
    from tehmm_b200 import trackIO, tracks_device
    from tehmm_b200.engine import get_engine
    from tehmm_b200.track import IntegerTrackTable
    rng = np.random.RandomState(9)
    hi, K, N, eff = 40_000, 3, 4, 20

    class Map(object):
        def __init__(self):
            self.m = {}

        def getMissingVal(self):
            return 0

        def getMap(self, v, update=False):
            if v not in self.m and update:
                self.m[v] = len(self.m) + 1
            return self.m.get(v, 0)
    d = tracks_device.new_table(hi, K)
    for k in range(K):
        p = str(tmp_path / ("t%d.bed" % k))
        with open(p, "w") as f:
            for s in np.sort(rng.randint(0, hi - 1, size=800)):
                f.write("chr1\t%d\t%d\t%s\n" % (s, min(hi, s + int(rng.choice([1, 5, 80]))), "abc"[rng.randint(3)]))
        tracks_device.fill_column(d, k, 0)
        trackIO.rasterizeBedData(d, k, p, "chr1", 0, hi, valCol=3, valMap=Map(), updateValMap=True)
    _, d_off, _ = tracks_device.segment(d, [0, hi], [0] * K, [0] * K, 0, 40, 0)
    d_small = tracks_device.compress(d, d_off, np.ones(K, dtype=np.uint8))
    d_ratios = tracks_device.segment_ratios(d_off, [0, hi], eff)
    # labelled intervals in segment rows
    nseg = int(d_small.shape[0])
    cuts = np.unique(np.concatenate([[0, nseg], rng.randint(0, nseg, size=300)]))
    rs, re_, st = cuts[:-1], cuts[1:], rng.randint(0, N, size=len(cuts) - 1)
    S = 4
    eng = get_engine(0)
    eng.use_device_batch(d_small.reshape(-1), 1, np.array([0, nseg], dtype=np.int64))
    dev = np.full((K, N, S), 0.1)
    eng.supervised_counts(rs, re_, st, dev, d_ratios)
    # host path: the same table through the per-interval fastUpdateCounts
    from tehmm_b200 import _emission
    host = IntegerTrackTable(K, "chr1", 0, hi)
    host.setSegments(d_off.cpu().numpy())
    host.data = d_small.cpu().numpy()
    ref = np.full((K, N, S), 0.1)
    r = d_ratios.cpu().numpy()
    for a, b, s in zip(rs, re_, st):
        _emission.fastUpdateCounts(("chr1", int(a), int(b), int(s)), host, ref, r)
    assert_array_equal(dev, ref)


@gpu
def test_launches_do_not_grow_with_intervals():
    from tehmm_b200.engine import get_engine
    rng = np.random.RandomState(12)
    T, K, N, S = 200_000, 2, 5, 4
    obs = rng.randint(0, S, size=(T, K)).astype(np.uint8)
    eng = get_engine(0)
    eng.upload_batch([obs])
    for init, ratios in ((0.0, None), (0.1, None), (0.0, rng.rand(T))):
        used = []
        for n in (10, 100_000):
            rs = np.sort(rng.randint(0, T - 1, size=n))
            stats = np.full((K, N, S), init)
            before = eng.ctx.stat("launches")
            eng.supervised_counts(rs, rs + 1, rng.randint(0, N, size=n), stats, ratios)
            used.append(eng.ctx.stat("launches") - before)
        assert used[0] == used[1] and used[0] <= 2, used


@gpu
def test_rejections_write_nothing():
    from tehmm_b200._lib import TehmmError
    from tehmm_b200.engine import get_engine
    rng = np.random.RandomState(13)
    T, K, N, S = 1000, 2, 3, 4
    obs = rng.randint(0, S, size=(T, K)).astype(np.uint8)
    obs[500, 1] = S                                        # a symbol >= S
    eng = get_engine(0)
    eng.upload_batch([obs])
    for init, ratios in ((0.0, None), (0.5, None), (0.0, np.ones(T))):
        for rs, re_, st in (([0, 490], [10, 510], [0, 1]),       # counts row 500
                            ([0], [10], [N]),                     # bad state
                            ([0], [T + 1], [0]),                  # row past the table
                            ([-1], [3], [0])):                    # negative row
            stats = np.full((K, N, S), init)
            with pytest.raises(TehmmError):
                eng.supervised_counts(rs, re_, st, stats, ratios)
            assert_array_equal(stats, np.full((K, N, S), init))
    stats = np.zeros((K, N, S))
    eng.supervised_counts([0, 600], [10, 700], [0, 2], stats)   # rows without the bad symbol still count
    assert stats.sum() == 110 * K
