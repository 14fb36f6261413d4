"""Host side of supervised training: which table rows every labelled interval counts.

IndependentMultinomialEmissionModel.supervisedTrain (emission.py:293-331 of the reference) scans
the tables for each interval from `lastHit`, counts the first run of consecutive tables that
overlap it and stops at the first table after that run that does not; `lastHit` only moves
forward.  When the tables' chromosome order differs from the intervals', some overlaps are
therefore never counted.  interval_triples() returns exactly the (table, first row, end row,
state) triples that scan counts, in the same order, so that one device call
(Engine.supervised_counts) can do all the counting.
"""
import numpy as np

from .track import TrackTable

_COORD_BITS = 40        # coordinates below 2^40: (chromosome block, coordinate) packs into one int64


def _vectorisable(table):
    """this package's TrackTable, unmasked, with its own getOverlapInTableCoords"""
    return (isinstance(table, TrackTable)
            and type(table).getOverlapInTableCoords is TrackTable.getOverlapInTableCoords
            and getattr(table, "maskArray", None) is None)


def _empty():
    z = np.zeros(0, dtype=np.int64)
    return z, z.copy(), z.copy(), z.copy()


def _scan(tables, bedIntervals):
    """the reference's loop, collecting the triples instead of counting them"""
    tix, lo, hi, st = [], [], [], []
    lastHit = 0
    lastOverlapEnd = -1
    for interval in bedIntervals:
        hit = False
        for tableIdx in range(lastHit, len(tables)):
            overlap = tables[tableIdx].getOverlapInTableCoords(interval, lastOverlapEnd)
            if overlap is not None:
                lastHit = tableIdx
                hit = True
                lastOverlapEnd = max(0, overlap[2] - 1)
                tix.append(tableIdx)
                lo.append(int(overlap[1]))
                hi.append(int(overlap[2]))
                st.append(int(overlap[3]))
            elif hit is True:
                break
    if not tix:
        return _empty()
    return (np.asarray(tix, dtype=np.int64), np.asarray(lo, dtype=np.int64),
            np.asarray(hi, dtype=np.int64), np.asarray(st, dtype=np.int64))


def _chrom_blocks(tables):
    """block id per table when the tables of each chromosome are consecutive in the list, sorted by
    start and disjoint (the layout of every TrackData), else None"""
    block, bid = {}, np.empty(len(tables), dtype=np.int64)
    prev = None
    for t, table in enumerate(tables):
        c = table.getChrom()
        if c != prev:
            if c in block:
                return None, None
            block[c] = len(block)
        elif table.getStart() < tables[t - 1].getEnd():
            return None, None
        if table.getStart() < 0 or table.getEnd() >= (1 << _COORD_BITS):
            return None, None
        bid[t] = block[c]
        prev = c
    return block, bid


def interval_triples(tables, bedIntervals):
    """(table index, first row, end row, state) int64 arrays of every count the reference's
    supervisedTrain scan makes, in its order; rows are in table coordinates (segments for a
    segmented table).  Vectorised for this package's tables; other table classes (the reference's
    own, masked tables) go through their getOverlapInTableCoords, one call per interval and table."""
    tables = list(tables)
    if len(tables) == 0 or len(bedIntervals) == 0:
        return _empty()
    if not all(_vectorisable(t) for t in tables):
        return _scan(tables, bedIntervals)
    block, bid = _chrom_blocks(tables)
    if block is None:
        return _scan(tables, bedIntervals)
    ivs = bedIntervals
    n = len(ivs)
    s = np.fromiter((iv[1] for iv in ivs), dtype=np.int64, count=n)
    e = np.fromiter((iv[2] for iv in ivs), dtype=np.int64, count=n)
    if n and (min(s.min(), e.min()) < 0 or max(s.max(), e.max()) >= (1 << _COORD_BITS)):
        return _scan(tables, bedIntervals)
    ib = np.fromiter((block.get(iv[0], -1) for iv in ivs), dtype=np.int64, count=n)
    tstart = np.array([t.getStart() for t in tables], dtype=np.int64)
    tend = np.array([t.getEnd() for t in tables], dtype=np.int64)
    # overlapping tables of interval i: [a, b) -- end > s and start < e within its chromosome's block
    sh = np.int64(1) << _COORD_BITS
    a = np.searchsorted(bid * sh + tend, ib * sh + s, side="right")
    b = np.searchsorted(bid * sh + tstart, ib * sh + e, side="left")
    a[ib < 0] = 0
    b[ib < 0] = 0
    # lastHit before interval i: the last table of the latest earlier run (0 at first)
    last = np.where(a < b, b - 1, -1)
    L = np.zeros(n, dtype=np.int64)
    if n > 1:
        L[1:] = np.maximum(np.maximum.accumulate(last[:-1]), 0)
    first = np.maximum(a, L)
    cnt = np.maximum(b - first, 0)
    total = int(cnt.sum())
    if total == 0:
        return _empty()
    iv = np.repeat(np.arange(n, dtype=np.int64), cnt)
    tix = first[iv] + (np.arange(total, dtype=np.int64) - np.repeat(np.cumsum(cnt) - cnt, cnt))
    lo = np.maximum(tstart[tix], s[iv])
    hi = np.minimum(tend[tix], e[iv])
    rlo, rhi = lo - tstart[tix], hi - tstart[tix]
    for t in np.unique(tix):
        offs = tables[t].getSegmentOffsets()
        if offs is None:
            continue
        sel = np.flatnonzero(tix == t)
        offs = tstart[t] + np.asarray(offs, dtype=np.int64)
        f = np.searchsorted(offs, lo[sel], side="right") - 1
        g = np.searchsorted(offs, hi[sel], side="left") - 1
        assert np.all(f >= 0) and np.all(g >= f)
        rlo[sel], rhi[sel] = f, g + 1
    states = np.array([int(ivs[i][3]) for i in np.flatnonzero(cnt)], dtype=np.int64)
    return tix, rlo, rhi, np.repeat(states, cnt[cnt > 0])
