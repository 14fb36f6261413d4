"""Emission models with the reference's API (/root/reference/emission.py).

IndependentMultinomialEmissionModel keeps the reference's parameter layout --
logProbs[TRACK, STATE, SYMBOL] float64, symbol 0 = "missing" (log-prob 0) when
zeroAsMissingData -- and its method surface.  allLogProbs / accumulateStats /
supervised counting run on the GPU through tehmm_b200._emission (strict float64
drop-ins) or, from MultitrackHmm, through the batched engine.  Parameter
estimation (maximize, Gaussian re-fit, user overrides) is O(K*N*S) host work.
"""
import itertools

import numpy as np
from numpy.testing import assert_array_almost_equal

from ._emission import canFast, fastAccumulateStats, fastAllLogProbs
from .common import EPSILON, NEGINF, assert_almost_equal_fast, logger, myLog, normalize
from .track import is_track_table


class IndependentMultinomialEmissionModel(object):
    def __init__(self, numStates, numSymbolsPerTrack, params=None,
                 zeroAsMissingData=True, fudge=0.0, normalizeFac=0.0,
                 randomize=False, effectiveSegmentLength=None,
                 random_state=None, randRange=(0.1, 0.9), uniformMixProb=0.1):
        self.numStates = numStates
        self.numTracks = len(numSymbolsPerTrack)
        self.numSymbolsPerTrack = numSymbolsPerTrack
        self.random_state = random_state
        if self.random_state is None:
            self.random_state = np.random.mtrand._rand
        #: [TRACK, STATE, SYMBOL]
        self.logProbs = None
        self.zeroAsMissingData = zeroAsMissingData
        #: added to every count during training (flattens the distributions)
        self.fudge = fudge
        # emission.py:50-60: 0 -> scores as is; k -> scores scaled by k / numTracks
        self.normalizeFac = 1.
        if normalizeFac > 0:
            self.normalizeFac = float(normalizeFac) / float(self.numTracks)
        #: length every segment is normalised to (None: no segment correction)
        self.effectiveSegmentLength = effectiveSegmentLength
        self.randRange = float(randRange[0]), float(randRange[1])
        #: uniform mix-in for discretised Gaussians (subclass)
        self.uniformMixProb = float(uniformMixProb)
        self.initParams(params=params, randomize=randomize)

    # ------------------------------------------------------------ accessors
    def getLogProbs(self):
        return self.logProbs

    def getNumStates(self):
        return self.numStates

    def getNumTracks(self):
        return self.numTracks

    def getNumSymbolsPerTrack(self):
        return self.numSymbolsPerTrack

    def _offset(self):
        return 1 if self.zeroAsMissingData is True else 0

    def getTrackSymbols(self, track):
        off = self._offset()
        for i in range(off, self.numSymbolsPerTrack[track] + off):
            yield i

    def getSymbols(self):
        """every possible observation vector (emission.py:101-115)"""
        if self.numTracks == 1:
            for i in self.getTrackSymbols(0):
                yield [i]
        else:
            per_track = [list(self.getTrackSymbols(t)) if self.numSymbolsPerTrack[t] > 0 else [0]
                         for t in range(self.numTracks)]
            for val in itertools.product(*per_track):
                yield val

    def trackTableWidths(self):
        """table columns in use per track (symbols + the missing symbol)"""
        return [int(n) + self._offset() for n in self.numSymbolsPerTrack]

    # ------------------------------------------------------------ parameters
    def _randDist(self, numPoints):
        lo, hi = self.randRange
        samples = lo + self.random_state.random_sample(numPoints) * (hi - lo)
        return normalize(samples)

    def initParams(self, params=None, randomize=False):
        """Flat (or random, or user-given) distributions -> log table (emission.py:125-168)."""
        off = self._offset()
        width = off + max(self.numSymbolsPerTrack)
        self.logProbs = np.zeros((self.numTracks, self.numStates, width), dtype=np.float64)
        for k in range(self.numTracks):
            nk = self.numSymbolsPerTrack[k]
            for j in range(self.numStates):
                if params is None:
                    if randomize is False:
                        dist = normalize(1. + np.zeros(nk, dtype=np.float64))
                    else:
                        dist = normalize(self._randDist(nk))
                else:
                    dist = np.array(params[k][j], dtype=np.float64)
                if off:
                    dist = np.append([1.], dist)      # symbol 0: unknown value, probability 1
                with np.errstate(divide="ignore"):
                    self.logProbs[k, j, :len(dist)] = np.log(dist)
        self.validate()

    def singleLogProb(self, state, singleObs):
        """log P(observation vector | state) (emission.py:170-177)"""
        logProb = 0.0
        for track, obsSymbol in enumerate(singleObs):
            logProb += self.logProbs[track][state][int(obsSymbol)]
        return logProb * self.normalizeFac

    def getSegmentRatios(self, obs):
        """segment length / effective length per observation, or None (emission.py:473-481)"""
        if is_track_table(obs):
            if obs.getSegmentOffsets() is not None and self.effectiveSegmentLength is not None:
                return obs.getSegmentLengthsAsRatio(self.effectiveSegmentLength)
        return None

    # ------------------------------------------------------------ hot path
    def allLogProbs(self, obs):
        """(T, numStates) float64 log-probabilities (emission.py:179-198)."""
        T = obs.shape[0]
        obsLogProbs = np.zeros((T, self.numStates), dtype=np.float64)
        segRatios = self.getSegmentRatios(obs)
        if not canFast(obs):
            # the reference's pure-python branch indexes with int(symbol)
            obs = np.ascontiguousarray(np.asarray(obs).astype(np.int32))
        if T > 0:
            fastAllLogProbs(obs, self.logProbs, obsLogProbs, self.normalizeFac, segRatios)
        return obsLogProbs

    def initStats(self):
        """obsStats[TRACK][STATE][SYMBOL], pre-filled with fudge (emission.py:208-219)."""
        obsStats = np.zeros((self.numTracks, self.numStates, np.max(self.numSymbolsPerTrack) + 1),
                            dtype=np.float64)
        for track in range(self.numTracks):
            obsStats[track, :, :self.numSymbolsPerTrack[track] + 1] += self.fudge
        return obsStats

    def accumulateStats(self, obs, obsStats, posteriors):
        """obsStats[k, j, obs[i,k]] += posteriors[i,j] (* segRatio[i]) (emission.py:221-241)."""
        assert obs.shape[1] == self.numTracks
        segRatios = self.getSegmentRatios(obs)
        if not canFast(obs):
            obs = np.ascontiguousarray(np.asarray(obs).astype(np.int32))
        fastAccumulateStats(obs, obsStats, posteriors, segRatios)
        return obsStats

    def maximize(self, obsStats, trackList=None):
        """M-step of the emission table (emission.py:243-267): per (track, state)
        normalise the counts of the real symbols; zero probabilities become
        log = -1e6 (not LOGZERO); a row without any mass keeps its old values."""
        off = self._offset()
        for track in range(self.numTracks):
            lo, hi = off, self.numSymbolsPerTrack[track] + off
            if hi <= lo:
                continue
            counts = np.asarray(obsStats[track, :, lo:hi], dtype=np.float64)      # (states, symbols)
            # np.cumsum adds left to right, like the reference's `total += c` loop (np.sum is pairwise)
            total = np.cumsum(counts, axis=1)[:, -1]
            denom = np.maximum(self.fudge, total)
            with np.errstate(divide="ignore", invalid="ignore"):
                probs = np.where(denom[:, None] != 0., counts / denom[:, None], 0.)
            trackSum = np.cumsum(probs, axis=1)[:, -1]
            keep = ~(trackSum < EPSILON)              # orphaned state/track: leave as was
            if keep.any():
                self.logProbs[track, keep, lo:hi] = myLog(probs[keep], logZeroVal=-1e6)
        self.validate()

    def validate(self):
        """every state's distribution over observation vectors sums to 1 (emission.py:269-291)"""
        numSymbols = 1
        for n in self.numSymbolsPerTrack:
            numSymbols = max(numSymbols, 1) * max(n, 1)
        if numSymbols >= 1000 or self.normalizeFac != 1.0:
            return
        # product of per-track sums == sum over the product space
        off = self._offset()
        total = np.ones(self.numStates)
        for track in range(self.numTracks):
            if self.numSymbolsPerTrack[track] > 0:
                total *= np.exp(self.logProbs[track, :, off:self.numSymbolsPerTrack[track] + off]).sum(axis=1)
            else:
                total *= np.exp(self.logProbs[track, :, 0])
        assert_almost_equal_fast(total, np.ones(self.numStates))

    def sample(self, state):
        return None

    # ------------------------------------------------------------ supervised
    def supervisedTrain(self, trackData, bedIntervals):
        """Count emissions per labelled interval, then maximize (emission.py:293-331).
        Both trackData and bedIntervals must be sorted.  The rows every interval counts are found
        on the host (supervised.interval_triples: the reference's table scan, lastHit quirk
        included), the tables they fall in go to the device once, and one
        Engine.supervised_counts call counts them all, bit-identical to one fastUpdateCounts per
        interval."""
        from .engine import get_engine
        from .supervised import interval_triples
        tables = trackData.getTrackTableList()
        assert len(tables) > 0
        assert len(bedIntervals) > 0
        obsStats = self.initStats()
        tix, lo, hi, state = interval_triples(tables, bedIntervals)
        if len(tix) > 0:
            # the per-interval path refuses these too (tehmm_strict_update_counts)
            assert state.min() >= 0 and state.max() < self.numStates, "interval state outside [0, %d)" % self.numStates
            used = np.unique(tix)
            eng = get_engine()
            offsets = eng.upload_batch([tables[t] for t in used])
            d_ratios = eng.upload_ratios([self.getSegmentRatios(tables[t]) for t in used])
            base = offsets[np.searchsorted(used, tix)]
            eng.supervised_counts(base + lo, base + hi, state, obsStats, d_ratios)
        self.maximize(obsStats, trackData.getTrackList())
        self.validate()

    # ------------------------------------------------------------ user overrides
    def applyUserEmissions(self, userEmLines, stateMap, trackList):
        """Force user-specified emission probabilities and renormalise the rest
        (emission.py:347-438).  Lines: STATE TRACK SYMBOL PROB."""
        logProbs = self.getLogProbs()
        mask = np.zeros(logProbs.shape, dtype=np.int8)
        for line in userEmLines:
            stripped = line.lstrip()
            if len(stripped) == 0 or stripped[0] == "#":
                continue
            toks = line.split()
            assert len(toks) == 4
            stateName, trackName = toks[0], toks[1]
            if not stateMap.has(stateName):
                raise RuntimeError("User Emission: State %s not found" % stateName)
            state = stateMap.getMap(stateName)
            track = trackList.getTrackByName(trackName)
            if track is None:
                raise RuntimeError("Track %s (in user emissions) not found" % trackName)
            self.applyUserEmissionLine(track, state, toks, logProbs, mask)

        probs = np.exp(logProbs)
        for track in range(self.getNumTracks()):
            if trackList.getTrackByNumber(track).getDist() == "gaussian":
                continue
            symbols = list(self.getTrackSymbols(track))
            for state in range(self.getNumStates()):
                curTotal, tgtTotal = 0.0, 1.0
                for symbol in symbols:
                    if mask[track, state, symbol] == 1:
                        tgtTotal -= probs[track, state, symbol]
                    else:
                        curTotal += probs[track, state, symbol]
                    if tgtTotal < 0.:
                        raise RuntimeError("User defined prob from state %s for track %s exceeds 1 by %e" % (
                            stateMap.getMapBack(state), trackList.getTrackByNumber(track).getName(),
                            0. - tgtTotal))
                additive = False
                addAmt = multAmt = 0.0
                if curTotal == 0. and tgtTotal < 1.:
                    additive = True
                    numUnmasked = self.numSymbolsPerTrack[track] - np.sum(mask[track, state])
                    if numUnmasked == 0:
                        raise RuntimeError("User defined emission prob for state %s track %s total less "
                                           "than 1 (%f) and there are no remaining symbols to assign "
                                           "leftover probability to" % (
                                               stateMap.getMapBack(state),
                                               trackList.getTrackByNumber(track).getName(), tgtTotal))
                    addAmt = (1. - tgtTotal) / float(numUnmasked)
                else:
                    assert curTotal > 0.
                    multAmt = tgtTotal / curTotal
                for symbol in symbols:
                    if mask[track, state, symbol] == 0:
                        if tgtTotal == 0.:
                            probs[track, state, symbol] = 0.
                        elif additive is False:
                            probs[track, state, symbol] *= multAmt
                        else:
                            probs[track, state, symbol] += addAmt
        self.logProbs = myLog(probs)
        self.validate()

    def applyUserEmissionLine(self, track, state, toks, logProbs, mask):
        """one `STATE TRACK SYMBOL PROB` line (emission.py:440-470)"""
        symbolMap = track.getValueMap()
        trackName = track.getName()
        trackNo = track.getNumber()
        symbolName = toks[2]
        prob = float(toks[3])
        if type(symbolMap).__name__ == "BinaryMap":
            if symbolName == "0" or symbolName == "None":
                symbolName = None
            symbol = symbolMap.getMap(symbolName)
        else:
            try:
                hasSymbol = symbolMap.has(symbolName)
                symbol = symbolMap.getMap(symbolName)
            except Exception:
                hasSymbol = False
                symbol = symbolMap.getMissingVal()
            if not hasSymbol:
                logger.warning("Track %s Symbol %s not found in data (setting as null value)" % (
                    trackName, symbolName))
        assert symbol in self.getTrackSymbols(trackNo)
        logProbs[trackNo, state, symbol] = myLog(prob)
        mask[trackNo, state, symbol] = 1


class IndependentMultinomialAndGaussianEmissionModel(IndependentMultinomialEmissionModel):
    """Tracks whose `dist` is "gaussian" are re-fitted to a discretised normal
    (mixed with a uniform) after every M-step (emission.py:483-615).  The hot
    path is unchanged: everything still comes out of the same log table."""

    def __init__(self, numStates, numSymbolsPerTrack, trackList, params=None,
                 zeroAsMissingData=True, fudge=0.0, normalizeFac=0.0,
                 randomize=False, effectiveSegmentLength=None,
                 random_state=None, randRange=(0.1, 0.9)):
        super(IndependentMultinomialAndGaussianEmissionModel, self).__init__(
            numStates, numSymbolsPerTrack, params, zeroAsMissingData, fudge, normalizeFac,
            randomize, effectiveSegmentLength, random_state, randRange)
        #: [TRACK, STATE, (MU, SIGMA)]
        self.gaussParams = None
        self.makeGaussian(trackList)

    def _symbolValues(self, track):
        catMap = track.getValueMap()
        symbols = np.array(list(self.getTrackSymbols(track.getNumber())), dtype=np.int64)
        values = np.array([float(catMap.getMapBack(s)) for s in symbols], dtype=np.float64)
        return symbols, values

    def makeGaussian(self, trackList):
        self.gaussParams = np.zeros((self.numTracks, self.numStates, 2), dtype=np.float64)
        assert self.numTracks == len(trackList)
        for track in trackList:
            if track.getDist() == "gaussian":
                for state in range(self.numStates):
                    mu, sigma = self.computeMuSigma(track, state)
                    self.gaussParams[track.getNumber(), state] = (mu, sigma)
                    self.applyGaussian(track, state)

    def computeMuSigma(self, track, state):
        """moments of the current multinomial of a track (emission.py:530-550)"""
        trackNo = track.getNumber()
        symbols, values = self._symbolValues(track)
        probs = np.exp(self.logProbs[trackNo, state, symbols])
        mu = 0.
        for v, p in zip(values, probs):
            mu += v * p
        var = 0.
        for v, p in zip(values, probs):
            var += np.square(v - mu) * p
        return mu, max(np.sqrt(var), EPSILON)

    def applyGaussian(self, track, state, logProbs=None):
        """write the discretised, uniform-mixed normal back into the table (emission.py:552-584)"""
        from scipy import stats
        trackNo = track.getNumber()
        if logProbs is None:
            logProbs = self.logProbs
        symbols, values = self._symbolValues(track)
        uniformProb = self.uniformMixProb / float(self.numSymbolsPerTrack[trackNo])
        prob = stats.norm.pdf(values, loc=self.gaussParams[trackNo, state, 0],
                              scale=self.gaussParams[trackNo, state, 1])
        prob = uniformProb + (1. - self.uniformMixProb) * prob
        assert np.all(prob > EPSILON)
        logProbs[trackNo, state, symbols] = myLog(prob)
        probs = np.exp(logProbs[trackNo, state, symbols])
        tot = 0.
        for p in probs:
            tot += p
        assert tot > 0.
        logProbs[trackNo, state, symbols] = myLog(probs / tot)

    def getGaussianParams(self, trackNo, state):
        return self.gaussParams[trackNo, state]

    def maximize(self, obsStats, trackList):
        super(IndependentMultinomialAndGaussianEmissionModel, self).maximize(obsStats)
        self.makeGaussian(trackList)

    def applyUserEmissionLine(self, track, state, toks, logProbs, mask):
        """`STATE TRACK MEAN STDEV` for gaussian tracks (emission.py:595-615)"""
        if track.getDist() != "gaussian":
            return super(IndependentMultinomialAndGaussianEmissionModel, self).applyUserEmissionLine(
                track, state, toks, logProbs, mask)
        self.gaussParams[track.getNumber(), state] = (float(toks[2]), float(toks[3]))
        self.applyGaussian(track, state, logProbs)
        mask[track.getNumber(), state, :] = 1
