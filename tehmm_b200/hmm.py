"""MultitrackHmm with the reference's API (/root/reference/hmm.py, basehmm.py).

fit / decode / score / score_samples keep the reference's semantics --
convergence rule, statistics, posterior epsilon, decoder precedence, forward
log-prob bookkeeping -- but the per-sequence Python loop of BaseHMM.fit
(basehmm.py:509-522) and the five Cython calls inside it are replaced by ONE
batched device E-step over all sequences (tehmm_b200.engine), and decoding runs
all tables of a call in one batch.  The M-step is O(N^2 + K*N*S) host work in
float64 and follows hmm.py:576-616.

Nothing CUDA-related is stored on the object: models are pickled
(modelIO.py:26-32) and deep-copied mid-fit (hmm.py:694).
"""
import copy
import string

import numpy as np
from numpy.testing import assert_array_almost_equal

from . import _hmm as _strict_hmm
from . import _lib, parallel
from .common import EPSILON, assert_almost_equal_fast, logger, logsumexp, myLog, normalize
from .engine import as_obs_array, get_engine

decoder_algorithms = ("viterbi", "map")

try:
    from collections.abc import Iterable
except ImportError:  # pragma: no cover
    from collections import Iterable


class BaseHMM(object):
    """Name kept for isinstance checks; the generic machinery lives in MultitrackHmm."""


class MultitrackHmm(BaseHMM):
    def __init__(self, emissionModel=None, startprob=None, transmat=None,
                 startprob_prior=None, transmat_prior=None, algorithm="viterbi",
                 random_state=None, n_iter=10, thresh=1e-2, params=string.ascii_letters,
                 init_params=string.ascii_letters, state_name_map=None, fudge=0.0,
                 fixTrans=False, fixEmission=False, fixStart=True, forceUserTrans=None,
                 forceUserEmissions=None, forceUserStart=None, transMatEpsilons=False,
                 maxProb=False, maxProbCut=None):
        self.n_components = emissionModel.getNumStates() if emissionModel is not None else 1
        self.n_iter = n_iter
        self.thresh = thresh
        self.params = params
        self.init_params = init_params
        self.transMatEpsilons = transMatEpsilons     # read by the transmat_ setter
        self.startprob_ = startprob
        self.startprob_prior = startprob_prior
        self.transmat_ = transmat
        self.transmat_prior = transmat_prior
        self._algorithm = algorithm
        self.random_state = random_state
        self.emissionModel = emissionModel
        self.trackList = None
        self.stateNameMap = state_name_map
        self.fudge = fudge
        self.fixTrans = fixTrans
        self.fixEmission = fixEmission
        self.fixStart = fixStart
        self.current_iteration = None
        self.last_forward_log_prob = None
        self.last_forward_log_prob_it = -1
        self.forceUserTrans = self._read_lines(forceUserTrans)
        self.forceUserEmissions = self._read_lines(forceUserEmissions)
        self.forceUserStart = self._read_lines(forceUserStart)
        self.maxProb = maxProb
        self.best_forward_log_prob = None
        self.bestCopy = None
        self.maxProbCut = maxProbCut
        self.numZeroInitEdges = 0
        self.numZeroInitStarts = 0

    @staticmethod
    def _read_lines(path):
        if path is None:
            return None
        with open(path) as f:
            return f.readlines()

    # ------------------------------------------------------------ properties
    # transitions keep exact zeros as LOGZERO unless transMatEpsilons (hmm.py:625-647)
    def _get_transmat(self):
        return np.exp(self._log_transmat)

    def _set_transmat(self, transmat):
        if transmat is None:
            transmat = np.tile(1.0 / self.n_components, (self.n_components, self.n_components))
        if not np.all(transmat) and self.transMatEpsilons is True:
            normalize(transmat, axis=1)          # in place: adds EPS to every entry
        if np.asarray(transmat).shape != (self.n_components, self.n_components):
            raise ValueError('transmat must have shape (n_components, n_components)')
        if not np.all(np.allclose(np.sum(transmat, axis=1), 1.0)):
            raise ValueError('Rows of transmat must sum to 1.0')
        self._log_transmat = myLog(np.asarray(transmat).copy())

    transmat_ = property(_get_transmat, _set_transmat)

    def _get_startprob(self):
        return np.exp(self._log_startprob)

    def _set_startprob(self, startprob):
        if startprob is None:
            startprob = np.tile(1.0 / self.n_components, self.n_components)
        else:
            startprob = np.asarray(startprob, dtype=np.float64)
        if len(startprob) != self.n_components:
            raise ValueError('startprob must have length n_components')
        if not np.allclose(np.sum(startprob), 1.0):
            raise ValueError('startprob must sum to 1.0')
        self._log_startprob = myLog(np.asarray(startprob).copy())

    startprob_ = property(_get_startprob, _set_startprob)

    def _get_algorithm(self):
        return self._algorithm

    def _set_algorithm(self, algorithm):
        if algorithm not in decoder_algorithms:
            raise ValueError("algorithm must be one of the decoder_algorithms")
        self._algorithm = algorithm

    algorithm = property(_get_algorithm, _set_algorithm)

    # ------------------------------------------------------------ getters
    def getTrackList(self):
        return self.trackList

    def getStartProbs(self):
        return self.startprob_

    def getTransitionProbs(self):
        return self.transmat_

    def getStateNameMap(self):
        return self.stateNameMap

    def getEmissionModel(self):
        return self.emissionModel

    def getLastLogProb(self):
        return self.last_forward_log_prob

    def validate(self):
        N = self.emissionModel.getNumStates()
        assert len(self.startprob_) == N
        assert not isinstance(self.startprob_[0], Iterable)
        assert self.transmat_.shape == (N, N)
        assert_almost_equal_fast(np.sum(self.startprob_), 1.)
        assert_almost_equal_fast(np.sum(self.transmat_, axis=1), np.ones(N))
        self.emissionModel.validate()

    # ------------------------------------------------------------ device plumbing
    def _engine(self):
        eng = get_engine()
        em = self.emissionModel
        widths = em.trackTableWidths() if hasattr(em, "trackTableWidths") else None
        eng.upload_model(self._log_startprob, self._log_transmat, em.getLogProbs(), em.normalizeFac,
                         widths)
        return eng

    def _seg_ratios(self, obs):
        return self.emissionModel.getSegmentRatios(obs)

    # ------------------------------------------------------------ more than 64 states
    # The batched kernels hold a lane's slice of the transition matrix in registers, which stops
    # at 64 states.  Wider models take the reference's own per-sequence flow (basehmm.py:238-359,
    # 507-522; hmm.py:545-574, 668-729) on the strict float64 kernels of tehmm_b200._hmm /
    # _emission -- still on the GPU, one sequence and one (T, N) float64 lattice at a time.
    def _wide(self):
        return self.emissionModel.getNumStates() > _lib.MAX_STATES

    def _wide_lattices(self, frame, ratios):
        T, N = frame.shape
        fwd, bwd = np.zeros((T, N)), np.zeros((T, N))
        _strict_hmm._forward(T, N, self._log_startprob, self._log_transmat, frame, ratios, fwd)
        _strict_hmm._backward(T, N, self._log_startprob, self._log_transmat, frame, ratios, bwd)
        return fwd, bwd

    @staticmethod
    def _wide_posteriors(fwd, bwd):
        gamma = fwd + bwd
        return np.exp(gamma.T - logsumexp(gamma, axis=1)).T

    def _wide_score_samples(self, obs):
        # basehmm.py:261-272: np.asarray(obs) drops the TrackTable, so no segment ratios anywhere
        frame = self.emissionModel.allLogProbs(as_obs_array(obs))
        fwd, bwd = self._wide_lattices(frame, None)
        lp = float(logsumexp(fwd[-1]))
        self._note_forward_logprob(lp)
        post = self._wide_posteriors(fwd, bwd)
        post += np.finfo(np.float32).eps
        post /= np.sum(post, axis=1).reshape((-1, 1))
        return lp, post

    def _wide_decode(self, obs, algorithm):
        if algorithm == "viterbi":
            # basehmm.py:327 / hmm.py:668-676: emission without ratios, DP with the table's
            frame = self.emissionModel.allLogProbs(as_obs_array(obs))
            T, N = frame.shape
            states, lp = _strict_hmm._viterbi(T, N, self._log_startprob, self._log_transmat,
                                              self._seg_ratios(obs), frame)
            return float(lp), states
        _, post = self._wide_score_samples(obs)
        return float(np.max(post, axis=1).sum()), np.argmax(post, axis=1)

    def _wide_estep(self, obs, stats, params, n_total, slots):
        """the E-step of fit() for this rank's sequences; one all-reduce like _device_estep"""
        N = self.n_components
        local = {'start': np.zeros(N), 'trans': np.zeros((N, N)), 'obs': np.zeros_like(stats['obs'])}
        lps = np.zeros(n_total)
        for slot, seq in zip(slots, obs):
            ratios = self._seg_ratios(seq)
            frame = self.emissionModel.allLogProbs(seq)
            fwd, bwd = self._wide_lattices(frame, ratios)
            lps[slot] = logsumexp(fwd[-1])
            post = self._wide_posteriors(fwd, bwd)
            if 's' in params:
                local['start'] += post[0]
            if 't' in params and frame.shape[0] > 1:
                logsum = np.zeros((N, N))
                _strict_hmm._log_sum_lneta(frame.shape[0], N, fwd, self._log_transmat, bwd, frame,
                                           float(lps[slot]), ratios, logsum)
                local['trans'] += np.exp(logsum)
            if 'e' in params:
                self.emissionModel.accumulateStats(seq, local['obs'], post)
        packed = np.concatenate([[float(len(obs))], local['start'], local['trans'].ravel(), local['obs'].ravel(), lps])
        n, _ = parallel.world()
        if n > 1:
            import torch
            t = torch.from_numpy(packed)
            packed = parallel.all_reduce_stats(t.cuda() if parallel._dist().get_backend() == "nccl" else t).cpu().numpy()
        o = 1
        stats['nobs'] += int(round(packed[0]))
        stats['start'] += packed[o:o + N]; o += N
        stats['trans'] += packed[o:o + N * N].reshape(N, N); o += N * N
        stats['obs'] += packed[o:o + stats['obs'].size].reshape(stats['obs'].shape); o += stats['obs'].size
        return packed[o:]

    @staticmethod
    def _gt(a, b):
        """a > b with Python 2 ordering of None (None sorts below every number):
        the reference compares against a best log-prob that starts out as None."""
        if a is None:
            return False
        return True if b is None else a > b

    def _note_forward_logprob(self, lp):
        """Bookkeeping every forward pass does in the reference (hmm.py:688-713):
        running log-prob of the current iteration, --maxProb snapshots, --maxProbCut."""
        if self.last_forward_log_prob_it != self.current_iteration:
            if self.maxProb is True and (self.current_iteration == 1 or
                                         self._gt(self.last_forward_log_prob, self.best_forward_log_prob)):
                self.best_forward_log_prob = self.last_forward_log_prob
                self.bestCopy = copy.deepcopy(self)
            self.last_forward_log_prob = lp
            self.last_forward_log_prob_it = self.current_iteration
            if (self.maxProb is True and self.bestCopy is not None and self.maxProbCut is not None and
                    self.current_iteration is not None and self.bestCopy.current_iteration is not None and
                    self.current_iteration - self.bestCopy.current_iteration > self.maxProbCut):
                logger.info("Stopping due to --maxProbCut %d" % self.maxProbCut)
                self.n_iter = self.current_iteration
        else:
            self.last_forward_log_prob += lp
            if self.maxProb is True and self.current_iteration > 1 and \
                    self._gt(self.last_forward_log_prob, self.best_forward_log_prob):
                self.best_forward_log_prob = self.last_forward_log_prob
                self.bestCopy = copy.deepcopy(self)

    # ------------------------------------------------------------ inference API
    def _compute_log_likelihood(self, obs):
        return self.emissionModel.allLogProbs(obs)

    def score_samples_batch(self, obs_list):
        """score_samples for many sequences in one device batch."""
        if self._wide():
            return [self._wide_score_samples(o) for o in obs_list]
        eng = self._engine()
        eng.upload_batch(obs_list)
        # basehmm.py:261-264: obs = np.asarray(obs) drops the TrackTable, so no
        # segment ratios reach the emission or the DP here.
        out = eng.posteriors(renorm_eps=True, want_post=True)
        res = []
        for lp, post in zip(out["logprob"], out["post"]):
            self._note_forward_logprob(float(lp))
            res.append((float(lp), post))
        return res

    def score_samples(self, obs):
        """(logprob, posteriors (T,N) float64) (basehmm.py:238-273)."""
        return self.score_samples_batch([obs])[0]

    eval = score_samples

    def score(self, obs):
        """forward log-likelihood (basehmm.py:275-299)."""
        if self._wide():
            frame = self.emissionModel.allLogProbs(as_obs_array(obs))
            T, N = frame.shape
            fwd = np.zeros((T, N))
            _strict_hmm._forward(T, N, self._log_startprob, self._log_transmat, frame, None, fwd)
            lp = float(logsumexp(fwd[-1]))
            self._note_forward_logprob(lp)
            return lp
        eng = self._engine()
        eng.upload_batch([obs])
        lp = float(eng.score()[0])
        self._note_forward_logprob(lp)
        return lp

    def decode_batch(self, obs_list, algorithm="viterbi"):
        # basehmm.py:389-392: the model's own algorithm wins over the argument
        if self._algorithm in decoder_algorithms:
            algorithm = self._algorithm
        if algorithm not in decoder_algorithms:
            raise KeyError(algorithm)                # basehmm.py:393-395: decoder[algorithm]
        if self._wide():
            return [self._wide_decode(o, algorithm) for o in obs_list]
        eng = self._engine()
        # host buffers in and out, everything in between inside the library
        if algorithm == "viterbi":
            # basehmm.py:327: emission from np.asarray(obs) (no ratios);
            # hmm.py:674: the DP does see the table's segment ratios
            lps, _, states = eng.decode_host(obs_list, _lib.DECODE_VITERBI,
                                             ratios=[self._seg_ratios(o) for o in obs_list])
            return [(float(lp), st) for lp, st in zip(lps, states)]
        lps, scores, states = eng.decode_host(obs_list, _lib.DECODE_MAP)
        for lp in lps:
            self._note_forward_logprob(float(lp))
        return [(float(sc), st) for sc, st in zip(scores, states)]

    def decode_both_batch(self, obs_list):
        """Viterbi path AND posterior (MAP) decoding of every sequence in ONE pass over the data: what
        decode_batch(obs, "viterbi") followed by decode_batch(obs, "map") return (bit-identical), as
        [(viterbi logprob, viterbi states, map score, map states)], for the price of one upload and one
        emission pass (teHmmEval.py asks for both of the same tracks, teHmmEval.py:127-160; the
        reference computes its frame once per call).  Segment ratios go to the Viterbi path only, as
        in decode_batch.  Models of more than 64 states take the two calls."""
        if self._wide():
            saved = self._algorithm
            try:
                self._algorithm = "viterbi"
                v = self.decode_batch(obs_list, "viterbi")
                self._algorithm = "map"
                m = self.decode_batch(obs_list, "map")
            finally:
                self._algorithm = saved
            return [(a[0], a[1], b[0], b[1]) for a, b in zip(v, m)]
        vlp, vst, msc, mst, flp = self._engine().decode_host_both(obs_list,
                                                                  ratios=[self._seg_ratios(o) for o in obs_list])
        for lp in flp:
            self._note_forward_logprob(float(lp))
        return [(float(a), s, float(b), t) for a, s, b, t in zip(vlp, vst, msc, mst)]

    def decode_both(self, obs):
        return self.decode_both_batch([obs])[0]

    # ------------------------------------------------------------ one long sequence over all ranks
    def decode_sharded(self, obs, algorithm="viterbi", halo=4096, gather=True):
        """decode() of ONE long sequence with its time axis split over the ranks of the
        process group (SURVEY.md section 8e, config 5; parallel.run_time_sharded).  Every
        rank passes the same `obs`; no segment ratios.  Returns (logprob, states): the whole
        int64 path on every rank (gather=True) or this rank's core range only.  For
        algorithm="map" the first value is the forward log-likelihood (score_sharded), not
        the reference's sum of posterior maxima."""
        if self._algorithm in decoder_algorithms:
            algorithm = self._algorithm
        obs = as_obs_array(obs)
        T = obs.shape[0]
        eng = self._engine()
        if algorithm == "viterbi":
            (part, core), _, _ = parallel.run_time_sharded(T, lambda c, w: eng.viterbi_window(obs, c, w), halo)
            lp = parallel.sum_over_ranks(part)
        elif algorithm == "map":
            core, _, _ = parallel.run_time_sharded(T, lambda c, w: eng.map_window(obs, c, w), halo)
            lp = self.score_sharded(obs, halo)
        else:
            raise ValueError("Decoder algorithm %r is not one of %s" % (algorithm, decoder_algorithms))
        return lp, (parallel.gather_states(core, T) if gather else core)

    def score_sharded(self, obs, halo=4096):
        """score() of one long sequence, forward pass split in time over the ranks."""
        obs = as_obs_array(obs)
        eng = self._engine()
        inc, _, _ = parallel.run_time_sharded(obs.shape[0], lambda c, w: eng.score_window(obs, c, w), halo)
        return parallel.sum_over_ranks(inc)

    def decode(self, obs, algorithm="viterbi"):
        """(logprob, state_sequence int64) (basehmm.py:361-396)."""
        return self.decode_batch([obs], algorithm)[0]

    def predict(self, obs, algorithm="viterbi"):
        return self.decode(obs, algorithm)[1]

    def predict_proba(self, obs):
        return self.score_samples(obs)[1]

    def logProb(self, trackData):
        return [self.score(t) for t in trackData.getTrackTableList()]

    def _named(self, states):
        if self.stateNameMap is not None:
            return [self.stateNameMap.getMapBack(s) for s in states]
        return states

    def viterbi(self, trackData, numThreads=1):
        """[(logprob, states)] per track table (hmm.py:221-237)."""
        assert numThreads == 1
        out = self.decode_batch(trackData.getTrackTableList())
        return [(p, self._named(s)) for p, s in out]

    def posteriorDecode(self, trackData, numThreads=1):
        """hmm.py:239-252; note decode() lets the model's algorithm win."""
        out = self.decode_batch(trackData.getTrackTableList(), algorithm="map")
        return [(p, self._named(s)) for p, s in out]

    def posteriorDistribution(self, trackData):
        return [p for _, p in self.score_samples_batch(trackData.getTrackTableList())]

    def emissionDistribution(self, trackData):
        return [self._compute_log_likelihood(t) for t in trackData.getTrackTableList()]

    # ------------------------------------------------------------ training
    def train(self, trackData):
        """Baum-Welch from the current parameters (hmm.py:155-172)."""
        self.bestCopy = None
        self.trackList = trackData.getTrackList()
        self.fit(trackData.getTrackTableList())
        if self.maxProb is True:
            assert self.bestCopy is not None
            self.emissionModel = self.bestCopy.emissionModel
            self.transmat_ = self.bestCopy.transmat_
            self._log_transmat = self.bestCopy._log_transmat
            self.startprob_ = self.bestCopy.startprob_
            self.last_forward_log_prob = self.bestCopy.last_forward_log_prob
            self.last_forward_log_prob_it = self.bestCopy.last_forward_log_prob_it
        self.validate()

    def supervisedTrain(self, trackData, bedIntervals):
        """Counts from labelled, sorted intervals (hmm.py:174-210)."""
        self.trackList = trackData.getTrackList()
        N = self.emissionModel.getNumStates()
        transitionCount = self.fudge + np.zeros((N, N), np.float64)
        freqCount = self.fudge + np.zeros((N,), np.float64)
        # the reference's loop (hmm.py:174-210), vectorised: np.add.at applies the adds one by one in
        # index order, so every float64 sum is taken in the loop's order
        intervals = list(bedIntervals)
        n = len(intervals)
        if n > 0:
            state = np.array([int(iv[3]) for iv in intervals], dtype=np.int64)
            start = np.array([iv[1] for iv in intervals])
            end = np.array([iv[2] for iv in intervals])
            chrom = np.empty(n, dtype=object)
            chrom[:] = [iv[0] for iv in intervals]
            same = np.zeros(n, dtype=bool)
            same[1:] = chrom[1:] == chrom[:-1]
            overlap = np.zeros(n, dtype=bool)
            overlap[1:] = same[1:] & (start[1:] < end[:-1])
            bad_state = np.flatnonzero(~(state < N))
            first_overlap = np.flatnonzero(overlap)
            if len(first_overlap) and (len(bad_state) == 0 or first_overlap[0] < bad_state[0]):
                i = int(first_overlap[0])
                raise RuntimeError("Overlapping or out of order training intervals detected: "
                                   "%s and %s." % (str(intervals[i - 1]), str(intervals[i])))
            assert len(bad_state) == 0
            # per interval: (state, state) += length - 1, then (previous state, state) += 1 when adjacent
            adjacent = np.zeros(n, dtype=bool)
            adjacent[1:] = same[1:] & (start[1:] == end[:-1])
            rows = np.stack([state, np.roll(state, 1)], axis=1)
            cols = np.stack([state, state], axis=1)
            vals = np.stack([end - start - 1, np.ones(n, dtype=np.int64)], axis=1)
            keep = np.stack([np.ones(n, dtype=bool), adjacent], axis=1)
            np.add.at(transitionCount, (rows[keep], cols[keep]), vals[keep])
            np.add.at(freqCount, state, end - start)
        for row in range(N):
            transitionCount[row] /= np.sum(transitionCount[row])
        self.transmat_ = np.copy(transitionCount)
        self._log_transmat = myLog(transitionCount)
        freqCount /= np.sum(freqCount)
        self.startprob_ = freqCount
        self.emissionModel.supervisedTrain(trackData, bedIntervals)
        self.validate()

    def _init(self, obs, params='ste'):
        """hmm.py:530-538.  (BaseHMM._init fills temporaries returned by the
        property getters, a no-op: parameters are NOT re-initialised, SURVEY appendix 2.)"""
        if self.fixTrans is True:
            self.params = self.params.replace("t", "")
        if self.fixEmission is True:
            self.params = self.params.replace("e", "")
        if self.fixStart is True:
            self.params = self.params.replace("s", "")
        if not isinstance(self.random_state, np.random.RandomState):
            if self.random_state is None or self.random_state is np.random:
                self.random_state = np.random.mtrand._rand
            else:
                self.random_state = np.random.RandomState(self.random_state)

    def _initialize_sufficient_statistics(self):
        N = self.n_components
        return {'nobs': 0, 'start': np.zeros(N), 'trans': np.zeros((N, N)),
                'obs': self.emissionModel.initStats()}

    def _local_estep(self, obs, params, n_total, slots, stats_S):
        """This rank's sequences in one device batch -> the packed float64 DEVICE tensor
        [sum logprob | nseq | start N | trans N*N | obs K*N*S | per-sequence logprob of the whole job]
        (Engine.estep).  Replaces basehmm.py:509-522 + hmm.py:545-574 for the shard."""
        eng = self._engine()
        # the observations do not change between EM iterations: they cross PCIe once per fit()
        token = getattr(self, "_fit_batch_token", None)
        if token is None or eng.batch_token != token:
            eng.upload_batch(obs)
            eng.batch_ratios = eng.upload_ratios([self._seg_ratios(o) for o in obs])
            eng.batch_token = token
        return eng.estep(ratios=eng.batch_ratios, want_start='s' in params, want_trans='t' in params,
                         want_obs='e' in params, device_result=True, seq_slots=(n_total, slots),
                         stats_S=stats_S)

    def _device_estep(self, obs, stats, params, n_total, slots):
        """E-step of one EM iteration over the ranks; returns the per-sequence log-probabilities of
        the WHOLE job, in the caller's sequence order.  A rank whose shard is EMPTY (fewer sequences
        than ranks, e.g. single-chromosome training on 8 GPUs) skips the device work and contributes
        zeros to the all-reduce, so that every rank reaches the collective."""
        if self._wide():
            return self._wide_estep(obs, stats, params, n_total, slots)
        N = self.n_components
        K, _, S = stats['obs'].shape
        base = 2 + N + N * N + K * N * S
        if len(obs) > 0:
            packed = self._local_estep(obs, params, n_total, slots, S)
        else:
            import torch
            nccl = parallel._dist() is not None and parallel._dist().get_backend() == "nccl"
            packed = torch.zeros(base + n_total, dtype=torch.float64, device="cuda" if nccl else "cpu")
        packed = parallel.all_reduce_stats(packed)       # the one collective of an EM iteration
        host = packed.cpu().numpy()
        stats['nobs'] += int(round(host[1]))
        if 's' in params:
            stats['start'] += host[2:2 + N]
        if 't' in params:
            stats['trans'] += host[2 + N:2 + N + N * N].reshape(N, N)
        if 'e' in params:
            stats['obs'] += host[2 + N + N * N:base].reshape(K, N, S)
        return host[base:].copy()

    def fit(self, obs, **kwargs):
        """EM (basehmm.py:475-541, hmm.py:618-620).  `obs` is a list of TrackTables /
        arrays.  Under torch.distributed (world_size > 1) the list is sharded over
        the ranks and the sufficient statistics are combined by one all-reduce per
        iteration; every rank ends with the same parameters."""
        self.current_iteration = 1
        if self._algorithm not in decoder_algorithms:
            self._algorithm = "viterbi"
        self._init(obs, self.init_params)
        obs = list(obs)
        slots = parallel.shard_indices([len(o) for o in obs])
        mine = [obs[i] for i in slots]
        logprob = []
        self._fit_batch_token = object()
        try:
            self._fit_loop(mine, obs, slots, logprob)
        finally:
            self._fit_batch_token = None
        return self

    def _fit_loop(self, mine, obs, slots, logprob):
        for i in range(copy.deepcopy(self.n_iter)):
            stats = self._initialize_sufficient_statistics()
            seq_logprobs = self._device_estep(mine, stats, self.params, len(obs), slots)
            curr_logprob = 0
            for lp in seq_logprobs:                 # same order and bookkeeping as the
                self._note_forward_logprob(float(lp))   # reference's per-sequence loop
                curr_logprob += float(lp)
            logprob.append(curr_logprob)
            msg = "BW Iteration %d: LogProb %f" % (i, curr_logprob)
            if i > 0:
                msg += " (delta %f)" % (logprob[-1] - logprob[-2])
            logger.info(msg)
            # converge test BEFORE the M-step (basehmm.py:530-536)
            if i > 0 and abs(logprob[-1] - logprob[-2]) < self.thresh:
                break
            if i == self.n_iter - 1:
                break
            self._do_mstep(stats, self.params)

    def _do_mstep(self, stats, params):
        """hmm.py:576-616."""
        self.validate()
        if self.startprob_prior is None:
            self.startprob_prior = 1.0
        if self.transmat_prior is None:
            self.transmat_prior = 1.0
        if 's' in params:
            self.startprob_ = normalize(np.maximum(self.startprob_prior - 1.0 + stats['start'], 1e-20))
        if 't' in params:
            lastMat = copy.deepcopy(self.transmat_)
            transmat_ = self.transmat_prior - 1.0 + stats['trans']
            for row in range(len(transmat_)):
                rowSum = np.sum(transmat_[row])
                if rowSum < EPSILON:
                    transmat_[row] = lastMat[row]     # orphaned state keeps its old row
                else:
                    transmat_[row] = transmat_[row] / rowSum
            self.transmat_ = transmat_
        if 'e' in params:
            self.emissionModel.maximize(stats['obs'], self.trackList)
        self.current_iteration += 1
        if self.forceUserTrans is not None:
            self.applyUserTrans(self.forceUserTrans)
        if self.forceUserEmissions is not None:
            self.applyUserEmissions(self.forceUserEmissions)
        if self.forceUserStart is not None:
            self.applyUserStarts(self.forceUserStart)
        self.validate()

    # ------------------------------------------------------------ user overrides
    def applyUserEmissions(self, userEmLines):
        assert self.stateNameMap is not None and self.trackList is not None
        self.emissionModel.applyUserEmissions(userEmLines, self.stateNameMap, self.trackList)

    @staticmethod
    def _data_lines(lines, ntok):
        for line in lines:
            stripped = line.lstrip()
            if len(stripped) > 0 and stripped[0] != "#":
                toks = line.split()
                assert len(toks) == ntok
                yield toks

    def applyUserTrans(self, userTransLines):
        """Force `FROM TO PROB` transitions, rescale the free ones (hmm.py:357-429)."""
        N = self.n_components
        mask = np.zeros((N, N), dtype=np.int8)
        transMat = self.transmat_
        catMap = self.stateNameMap
        for fromState, toState, prob in self._data_lines(userTransLines, 3):
            if not catMap.has(fromState) or not catMap.has(toState):
                raise RuntimeError("Cannot apply transition %s->%s to model since at least one of the "
                                   "states was not found in the supervised data." % (fromState, toState))
            fid, tid = catMap.getMap(fromState), catMap.getMap(toState)
            mask[fid, tid] = 1
            transMat[fid, tid] = float(prob)
        for fid in range(N):
            curTotal, tgtTotal = 0.0, 1.0
            for tid in range(N):
                if mask[fid, tid] == 1:
                    tgtTotal -= transMat[fid, tid]
                else:
                    curTotal += transMat[fid, tid]
            if tgtTotal < -EPSILON:
                raise RuntimeError("User defined probability %f from state %s exceeds 1" % (
                    tgtTotal, catMap.getMapBack(fid)))
            for tid in range(N):
                if mask[fid, tid] == 0:
                    if tgtTotal == 0.:
                        transMat[fid, tid] = 0.
                    else:
                        transMat[fid, tid] *= (tgtTotal / curTotal)
        self.numZeroInitEdges = int(np.sum(transMat <= EPSILON))
        self.transmat_ = transMat

    def applyUserStarts(self, userStartLines):
        """Force `STATE PROB` start probabilities (hmm.py:432-488)."""
        N = self.n_components
        startProbs = self.startprob_
        mask = np.zeros(startProbs.shape, dtype=np.int8)
        for stateName, prob in self._data_lines(userStartLines, 2):
            if not self.stateNameMap.has(stateName):
                raise RuntimeError("State %s not found in supervised data" % stateName)
            state = self.stateNameMap.getMap(stateName)
            startProbs[state] = float(prob)
            mask[state] = 1
        curTotal, tgtTotal = 0.0, 1.0
        for state in range(N):
            if mask[state] == 1:
                tgtTotal -= startProbs[state]
            else:
                curTotal += startProbs[state]
            if tgtTotal < 0.:
                raise RuntimeError("User defined start probabiliies exceed 1")
        for state in range(N):
            if mask[state] == 0:
                if tgtTotal == 0.:
                    startProbs[state] = 0.
                else:
                    startProbs[state] *= (tgtTotal / curTotal)
        self.numZeroInitStarts = int(np.sum(startProbs < EPSILON))
        self.startprob_ = startProbs

    def getNumFreeParameters(self):
        """hmm.py:490-518 (fully unsupervised models only)."""
        if self.forceUserTrans is not None or self.forceUserStart is not None or \
                self.forceUserEmissions is not None:
            raise RuntimeError("hmm.getNumFreeParamaters() does not yet support "
                               "forceUsers{Trans,Start,Emissions} functionality.")
        numParams = 0
        N = self.emissionModel.getNumStates()
        if self.fixTrans is False:
            numParams += N * (N - 1) - self.numZeroInitEdges
        if self.fixStart is False:
            numParams += N - 1 - self.numZeroInitStarts
        if self.fixEmission is False:
            for track in self.trackList:
                if track.getDist() == "gaussian":
                    per = 2
                else:
                    per = self.emissionModel.getNumSymbolsPerTrack()[track.getNumber()] - 1
                numParams += N * per
        return numParams

    def __str__(self):
        states = list(range(self.n_components))
        if self.stateNameMap is not None:
            states = [self.stateNameMap.getMapBack(x) for x in states]
        s = "\nNumStates = %d:\n%s\n" % (self.n_components, str(states))
        if self.random_state is not None:
            s += "\nseed = %s\n" % str(self.random_state)
        s += "\nStart probs =\n%s\n" % str(list(zip(states, self.startprob_)))
        s += "\nTransitions =\n%s\n" % str(self.transmat_)
        s += "\nlogTransitions = \n%s\n" % str(myLog(self.transmat_))
        em = self.emissionModel
        s += "\nNumber of symbols per track=\n%s\n" % str(em.getNumSymbolsPerTrack())
        s += "\nEmissions =\n"
        probs = np.exp(em.getLogProbs())
        for state, name in enumerate(states):
            s += "State %s:\n" % name
            for trackNo in range(em.getNumTracks()):
                s += "  Track %d:\n" % trackNo
                for symbol in em.getTrackSymbols(trackNo):
                    p = probs[trackNo][state][symbol]
                    if p > 0.0000005:
                        s += "    %s) %f (log=%s)\n" % (symbol, p, str(myLog(p)))
        return s
