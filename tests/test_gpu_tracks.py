"""-m gpu: the data formats either side of the trellis (SURVEY.md section 8f ranks 2-3) built on the
device -- interval rasterisation, segmentation, segment compression, runSum -- against the
reference: stored outputs of its trackIO.readBedData and _track.runSum (tests/golden/readbed.npz,
runsum.npz), restatements of bin/segmentTracks.py:200-277 (a Python-2 script) and of
TrackTable.segment (track.py:449-533; its binSearch divides with `/`).  Byte / index work: everything
is compared bit for bit."""
import os
import types

import numpy as np
import pytest
from numpy.testing import assert_array_equal

from conftest import golden

pytestmark = pytest.mark.gpu


def write_bed(path, rng, n, lo, hi, names, chrom="chr1", scores=False):
    """n intervals inside [lo, hi), overlapping, sorted by start like sortBed leaves them"""
    starts = np.sort(rng.randint(lo, hi - 1, size=n))
    rows = []
    for s in starts:
        e = min(hi, int(s) + int(rng.choice([1, 1, 2, 5, 30, 400])))
        rows.append((chrom, int(s), e, names[rng.randint(len(names))], "%d" % rng.randint(0, 50)))
    if scores:   # abutting intervals, so that the delta branch (trackIO.py:187-193) is taken
        rows, pos = [], lo
        while pos < hi:
            e = min(hi, pos + int(rng.choice([1, 3, 10, 100])))
            rows.append((chrom, pos, e, names[rng.randint(len(names))], "%d" % rng.randint(0, 9)))
            pos = e + (int(rng.randint(0, 3)) if rng.rand() < 0.3 else 0)
    with open(path, "w") as f:
        for r in rows:
            f.write("%s\t%d\t%d\t%s\t%s\n" % r)
    return rows


class CategoryMap(object):
    """the reference's CategoryMap(reserved=1) (track.py:668-815) as readBedData uses it: values are
    numbered 1, 2, ... in the order they are first added (keyed by the value itself), 0 is missing"""

    def __init__(self):
        self.catMap = {}

    def getMissingVal(self):
        return 0

    def getMap(self, inVal, update=False):
        if update and inVal not in self.catMap:
            self.catMap[inVal] = len(self.catMap) + 1
        return self.catMap.get(inVal, self.getMissingVal())

    def __len__(self):
        return len(self.catMap)


class BinaryMap(CategoryMap):
    """the reference's BinaryMap (track.py:816-832) as readBedData uses it: every interval value is the
    same symbol, bases outside the intervals keep the missing value"""

    def getMap(self, inVal, update=False):
        return CategoryMap.getMap(self, inVal is not None, update)


READBED_CASES = ["category", "binary", "delta"]


def readbed_inputs(tmp_path, case, category_map, binary_map):
    """the BED file, value-map factory and readBedData keywords of one case of
    test_readBedData_matches_reference (tests/golden/make_golden.py:readbed_case runs them through the
    reference's readBedData with its own map classes)"""
    rng = np.random.RandomState({"category": 1, "binary": 2, "delta": 3}[case])
    lo, hi = 1_000, 41_000
    path = os.path.join(str(tmp_path), "t.bed")
    write_bed(path, rng, 3_000, lo, hi, ["LTR", "SINE", "LINE", "DNA", "Simple_repeat"], scores=(case == "delta"))

    def maps():
        return binary_map() if case == "binary" else category_map()
    kw = {"category": dict(valCol=3), "binary": dict(valCol=0), "delta": dict(valCol=4, useDelta=True)}[case]
    return path, maps, kw, lo, hi


@pytest.mark.parametrize("case", READBED_CASES)
def test_readBedData_matches_reference(tmp_path, case):
    """the reference's readBedData output and value-map size, stored per case
    (tests/golden/make_golden.py:readbed_case)"""
    from tehmm_b200 import trackIO
    g = golden("readbed")
    path, maps, kw, lo, hi = readbed_inputs(tmp_path, case, CategoryMap, BinaryMap)
    out_ref = g["out_" + case]
    m_our = maps()
    missing = m_our.getMissingVal()
    buf_our = np.full(hi - lo, missing, dtype=np.uint8)
    out_our = trackIO.readBedData(path, "chr1", lo, hi, valMap=m_our, updateValMap=True, needIntersect=False,
                                  outputBuf=buf_our, **kw)
    assert out_our is buf_our
    assert_array_equal(out_our, out_ref)
    assert len(m_our) == int(g["nvals_" + case])
    assert (out_ref != missing).sum() > 1000
    # the list form (no outputBuf) and our own intersection (bedtools' job in the reference) on a
    # file that also holds another chromosome and intervals sticking out of the query
    lst = trackIO.readBedData(path, "chr1", lo, hi, valMap=maps(), updateValMap=True, needIntersect=False, **kw)
    assert_array_equal(np.asarray(lst, dtype=np.int64), out_ref.astype(np.int64))
    if case != "delta":
        path2 = str(tmp_path / "t2.bed")
        with open(path2, "w") as f:
            f.write("chr2\t%d\t%d\tLTR\t1\n" % (lo + 5, lo + 500))
            f.write(open(path).read())
        sub = trackIO.readBedData(path2, "chr1", lo + 1000, hi - 1000, valMap=maps(), updateValMap=True,
                                  outputBuf=np.full(hi - lo - 2000, missing, dtype=np.uint8), **kw)
        # (category numbers are assigned in order of appearance inside the query: compare through the names)
        if case == "binary":
            assert_array_equal(sub, out_ref[1000:-1000])


def test_rasterize_long_and_overlapping_intervals():
    """later intervals win where they overlap (trackIO.py:198-202), including intervals long enough
    for the block kernel and intervals that stick out of the region"""
    from tehmm_b200 import tracks_device
    lo, hi = 0, 300_000
    s = np.array([-50, 10, 1000, 1500, 100_000, 299_990], dtype=np.int64)
    e = np.array([20, 200_000, 1200, 1501, 250_000, 400_000], dtype=np.int64)
    v = np.array([1, 2, 3, 4, 5, 6], dtype=np.int32)
    v0 = np.array([11, 12, 13, 14, 15, 16], dtype=np.int32)
    want = np.zeros(hi - lo, dtype=np.uint8)
    for i in range(len(s)):
        a, b = max(lo, s[i]), min(hi, e[i])
        want[a] = v0[i]
        want[a + 1:b] = v[i]
    d = tracks_device.new_table(hi - lo, 3)
    tracks_device.fill_column(d, 1, 0)
    tracks_device.rasterize(d, 1, s, e, v, v0, lo, hi)
    got = d.cpu().numpy()
    assert_array_equal(got[:, 1], want)
    assert not got[:, 0].any() and not got[:, 2].any()


def test_runSum_matches_reference():
    """the reference's _track.runSum on the same masks, stored per position as the step from the
    previous entry (tests/golden/make_golden.py:runsum_case)"""
    from tehmm_b200 import _track
    g = golden("runsum")
    rng = np.random.RandomState(5)
    for n in (1, 31, 1000, 1_000_003):
        mask = (rng.rand(n) < 0.3).astype(np.uint8)
        b = np.zeros(n, dtype=np.int32)
        _track.runSum(mask, b)
        assert_array_equal(b, np.cumsum(g["steps_%d" % n], dtype=np.int64))


def reference_segment_scan(data, args):
    """bin/segmentTracks.py:214-239 (the per-table loop of segmentTracks) with isNewSegment
    (segmentTracks.py:241-277) inlined; returns the rows where a segment starts"""
    starts = [0]
    prevMode = args.comp == "prev"
    pi, curLen = 0, 0
    for i in range(1, len(data)):
        curLen += 1
        if args.fixLen > 0:
            new = curLen >= args.fixLen
        elif args.maxLen > 0 and curLen >= args.maxLen:
            new = True
        else:
            difCount, cutTrackFound = 0, False
            for j in range(data.shape[1]):
                if args.ignoreList[j] == 0 and data[i][j] != data[pi][j]:
                    difCount += 1
                    if args.cutList[j] == 1:
                        cutTrackFound = True
            new = cutTrackFound is True or difCount > args.thresh
        if new:
            starts.append(i)
            pi = i
            curLen = 0
        if prevMode:
            pi = i
    return np.asarray(starts, dtype=np.int64)


def runny_table(rng, T, K, p_change):
    """K columns of run-length data: every track changes value with its own probability"""
    data = np.zeros((T, K), dtype=np.uint8)
    for k in range(K):
        ch = rng.rand(T) < p_change[k]
        ch[0] = True
        vals = rng.randint(0, 4, size=int(ch.sum()))
        data[:, k] = vals[np.cumsum(ch) - 1]
    return data


SEG_CASES = [
    dict(comp="first", thresh=1, maxLen=0, fixLen=0, cut=[], ignore=[]),
    dict(comp="prev", thresh=1, maxLen=0, fixLen=0, cut=[], ignore=[]),
    dict(comp="first", thresh=0, maxLen=100, fixLen=0, cut=[2], ignore=[0]),
    dict(comp="prev", thresh=2, maxLen=37, fixLen=0, cut=[1, 3], ignore=[5]),
    dict(comp="first", thresh=3, maxLen=0, fixLen=0, cut=[4], ignore=[]),
    dict(comp="first", thresh=1, maxLen=0, fixLen=250, cut=[], ignore=[]),
    dict(comp="first", thresh=5, maxLen=1000, fixLen=0, cut=[], ignore=[]),          # segments longer than a scan chunk
]


@pytest.mark.parametrize("case", range(len(SEG_CASES)))
def test_segmentation_matches_reference_scan(case, tmp_path):
    from tehmm_b200 import segmentTracks
    from tehmm_b200.track import IntegerTrackTable
    cfg = SEG_CASES[case]
    rng = np.random.RandomState(10 + case)
    K = 6
    lens = [1, 2, 5_000, 257, 30_000]
    tables = []
    for r, T in enumerate(lens):
        t = IntegerTrackTable(K, "chr%d" % (r + 1), 1000 * r, 1000 * r + T)
        t.data[:] = runny_table(rng, T, K, [0.01, 0.02, 0.005, 0.05, 0.002, 0.3])
        tables.append(t)
    args = types.SimpleNamespace(comp=cfg["comp"], thresh=cfg["thresh"], maxLen=cfg["maxLen"], fixLen=cfg["fixLen"],
                                 ignoreList=[1 if j in cfg["ignore"] else 0 for j in range(K)],
                                 cutList=[1 if j in cfg["cut"] else 0 for j in range(K)], stats=None, co=7,
                                 outBed=str(tmp_path / "seg.bed"))
    per_table, _, _, _ = segmentTracks.segment_tables(tables, args)
    total = 0
    for (t, starts), T in zip(per_table, lens):
        want = reference_segment_scan(t.data, args)
        assert_array_equal(starts, want)
        total += len(want)
    assert total > len(lens)
    # the BED the script writes (segmentTracks.py:224-238): names are the hexadecimal running count from --co
    td = types.SimpleNamespace(getTrackTableList=lambda: tables)
    segmentTracks.segmentTracks(td, args, {})
    lines = open(args.outBed).read().splitlines()
    assert len(lines) == total
    first = lines[0].split("\t")
    assert first[0] == "chr1" and int(first[1]) == 0 and first[3] == hex(7)[2:]
    assert lines[-1].split("\t")[3] == hex(7 + total - 1)[2:]
    ends = {}
    for ln in lines:
        c, a, b, _ = ln.split("\t")
        assert int(b) > int(a)
        assert ends.get(c, int(a)) == int(a)          # segments tile each table without gaps
        ends[c] = int(b)
    for r, T in enumerate(lens):
        assert ends["chr%d" % (r + 1)] == 1000 * r + T


def test_segment_compress_matches_reference_logic():
    """TrackTable.segment with interpolate (track.py:449-495,515-533,603-620): per-track mode of every
    segment (scipy.stats.mode: the smallest of the most frequent values), one row per segment; and the
    segment-length ratios (track.py:504-513)"""
    from tehmm_b200.track import IntegerTrackTable
    rng = np.random.RandomState(3)
    T, K = 50_000, 5
    t = IntegerTrackTable(K, "chrX", 500, 500 + T)
    t.data[:] = runny_table(rng, T, K, [0.2, 0.5, 0.05, 0.9, 0.01])
    orig = t.data.copy()
    cuts = np.unique(np.concatenate([[0], rng.randint(1, T, size=4_000)]))
    lens = np.diff(np.append(cuts, T))
    assert lens.max() > 64 and lens.min() == 1
    segs = [("chrX", 500 + int(a), 500 + int(a + n)) for a, n in zip(cuts, lens)]
    t.segment(segs, None, interpolate=True)
    assert t.data.shape == (len(cuts), K) and len(t) == len(cuts)
    want = np.empty((len(cuts), K), dtype=np.uint8)
    for s, (a, n) in enumerate(zip(cuts, lens)):
        for k in range(K):
            want[s, k] = np.argmax(np.bincount(orig[a:a + n, k], minlength=4))      # first maximum = smallest mode
    assert_array_equal(t.data, want)
    assert_array_equal(t.getSegmentOffsets(), cuts)
    assert_array_equal(t.getSegmentLengthsAsRatio(100), lens / 100.0)
    # without interpolation: the first row of every segment (compressSegments, track.py:594-601)
    t2 = IntegerTrackTable(K, "chrX", 500, 500 + T)
    t2.data[:] = orig
    t2.segment(segs, None, interpolate=False)
    assert_array_equal(t2.data, orig[cuts])


def test_device_pipeline_bed_to_decode(tmp_path):
    """BED files -> device table -> segments -> compressed table -> Viterbi, nothing but interval lists
    and the decoded path crossing PCIe; equals the host route through the reference-named APIs"""
    import torch
    from tehmm_b200 import segmentTracks, synth, trackIO, tracks_device
    from tehmm_b200.engine import get_engine
    from tehmm_b200.track import IntegerTrackTable
    rng = np.random.RandomState(8)
    lo, hi, K = 0, 60_000, 3
    names = ["a", "b", "c"]

    class Map(object):                      # minimal value map: category numbers in order of appearance
        def __init__(self):
            self.m = {}

        def getMissingVal(self):
            return 0

        def getMap(self, v, update=False):
            if v not in self.m and update:
                self.m[v] = len(self.m) + 1
            return self.m.get(v, 0)
    paths = []
    for k in range(K):
        p = str(tmp_path / ("track%d.bed" % k))
        write_bed(p, rng, 1_500, lo, hi, names)
        paths.append(p)
    d = tracks_device.new_table(hi - lo, K)
    host = IntegerTrackTable(K, "chr1", lo, hi)
    for k, p in enumerate(paths):
        tracks_device.fill_column(d, k, 0)
        trackIO.rasterizeBedData(d, k, p, "chr1", lo, hi, valCol=3, valMap=Map(), updateValMap=True)
        host.initRow(k, 0)
        trackIO.readBedData(p, "chr1", lo, hi, valCol=3, valMap=Map(), updateValMap=True, outputBuf=host.getRow(k))
    assert_array_equal(d.cpu().numpy(), host.data)
    args = types.SimpleNamespace(comp="first", thresh=0, maxLen=50, fixLen=0, ignoreList=[0] * K, cutList=[0] * K, stats=None, co=0)
    d_cut, d_off, passes = tracks_device.segment(d, [0, hi - lo], args.ignoreList, args.cutList, args.thresh, args.maxLen, args.fixLen)
    assert_array_equal(d_off.cpu().numpy(), reference_segment_scan(host.data, args))
    d_small = tracks_device.compress(d, d_off, np.ones(K, dtype=np.uint8))
    ratios = tracks_device.segment_ratios(d_off, [0, hi - lo], 50)
    offs = d_off.cpu().numpy()
    host.segment([("chr1", int(a), int(b)) for a, b in zip(offs, np.append(offs[1:], hi - lo))], None)
    assert_array_equal(d_small.cpu().numpy(), host.data)
    assert_array_equal(ratios.cpu().numpy(), host.getSegmentLengthsAsRatio(50))
    # decode the device-resident table
    m = synth.make_model(N=5, syms=(3, 3, 3), seed=2)
    eng = get_engine(0)
    eng.upload_model(m["log_start"], m["log_trans"], m["table"], 1.0, m["widths"])
    eng.use_device_batch(d_small.reshape(-1), 1, np.array([0, d_small.shape[0]], dtype=np.int64))
    lp_dev, st_dev = eng.viterbi()
    eng.upload_batch([host.data])
    lp_host, st_host = eng.viterbi()
    assert_array_equal(st_dev[0], st_host[0])
    assert lp_dev[0] == lp_host[0]
