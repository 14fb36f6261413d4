"""NumPy front-end of the CPU oracle (oracle/tehmm_oracle.c).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs -- never from tehmm_b200/.

Function names and argument order mirror the reference's Cython modules
(_hmm.pyx / _emission.pyx) so the parity tests read like the reference's own.
"""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libtehmm_oracle.so")
_lib = None

_D = ctypes.POINTER(ctypes.c_double)
_I64 = ctypes.POINTER(ctypes.c_int64)


def build(force=False):
    """Compile oracle/tehmm_oracle.c with gcc (seconds), next to it or, where oracle/ is
    read-only, into a temporary directory."""
    global _LIB_PATH
    src = os.path.join(_HERE, "tehmm_oracle.c")
    if (force or not os.path.exists(_LIB_PATH)
            or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src)):
        if not os.access(_HERE, os.W_OK):
            tmp = tempfile.mkdtemp(prefix="tehmm_oracle_")
            atexit.register(shutil.rmtree, tmp, True)
            _LIB_PATH = os.path.join(tmp, "libtehmm_oracle.so")
        subprocess.check_call(["make", "-s", "-C", _HERE, "LIB=" + _LIB_PATH])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB_PATH)
        L.orc_logsumexp.restype = ctypes.c_double
        L.orc_viterbi.restype = ctypes.c_double
        L.orc_estep_sequence.restype = ctypes.c_double
        _lib = L
    return _lib


def _d(a):
    return None if a is None else a.ctypes.data_as(_D)


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _obs(obs):
    obs = np.ascontiguousarray(obs)
    if obs.dtype == np.uint8:
        return obs, 1
    if obs.dtype == np.uint16:
        return obs, 2
    if obs.dtype == np.int32:
        return obs, 4
    # the reference's pure-python branch indexes with int(symbol)
    return np.ascontiguousarray(obs.astype(np.int32)), 4


def logsumexp(v):
    v = _f64(v)
    return lib().orc_logsumexp(_d(v), ctypes.c_long(v.size))


def fastAllLogProbs(obs, logProbs, outProbs, normalize, segRatios):
    obs, nb = _obs(obs)
    logProbs = _f64(logProbs)
    assert outProbs.dtype == np.float64 and outProbs.flags.c_contiguous
    T, K = obs.shape
    _, N, S = logProbs.shape
    r = _f64(segRatios)
    lib().orc_all_log_probs(obs.ctypes.data_as(ctypes.c_void_p), nb, ctypes.c_long(T), K,
                            _d(logProbs), N, S, _d(outProbs),
                            ctypes.c_double(normalize), _d(r))


def _forward(T, N, log_startprob, log_transmat, framelogprob, segRatios, fwdlattice):
    a, b, c, r = _f64(log_startprob), _f64(log_transmat), _f64(framelogprob), _f64(segRatios)
    lib().orc_forward(ctypes.c_long(T), N, _d(a), _d(b), _d(c), _d(r), _d(fwdlattice))


def _backward(T, N, log_startprob, log_transmat, framelogprob, segRatios, bwdlattice):
    a, b, c, r = _f64(log_startprob), _f64(log_transmat), _f64(framelogprob), _f64(segRatios)
    lib().orc_backward(ctypes.c_long(T), N, _d(a), _d(b), _d(c), _d(r), _d(bwdlattice))


def _viterbi(T, N, log_startprob, log_transmat, segRatios, framelogprob):
    a, b, c, r = _f64(log_startprob), _f64(log_transmat), _f64(framelogprob), _f64(segRatios)
    states = np.empty(T, dtype=np.int64)
    lp = lib().orc_viterbi(ctypes.c_long(T), N, _d(a), _d(b), _d(r), _d(c),
                           states.ctypes.data_as(_I64))
    return states, lp


def _log_sum_lneta(T, N, fwdlattice, log_transmat, bwdlattice, framelogprob, logprob,
                   segRatios, logsum_lneta):
    f, a, b, c, r = (_f64(fwdlattice), _f64(log_transmat), _f64(bwdlattice),
                     _f64(framelogprob), _f64(segRatios))
    lib().orc_log_sum_lneta(ctypes.c_long(T), N, _d(f), _d(a), _d(b), _d(c),
                            ctypes.c_double(logprob), _d(r), _d(logsum_lneta))


def posteriors(fwdlattice, bwdlattice, renorm_eps=False):
    f, b = _f64(fwdlattice), _f64(bwdlattice)
    T, N = f.shape
    post = np.empty((T, N))
    lib().orc_posteriors(ctypes.c_long(T), N, _d(f), _d(b), _d(post), int(bool(renorm_eps)))
    return post


def fastAccumulateStats(obs, obsStats, posteriors, segRatios):
    obs, nb = _obs(obs)
    T, K = obs.shape
    _, N, S = obsStats.shape
    p, r = _f64(posteriors), _f64(segRatios)
    assert obsStats.dtype == np.float64 and obsStats.flags.c_contiguous
    lib().orc_accumulate_stats(obs.ctypes.data_as(ctypes.c_void_p), nb, ctypes.c_long(T), K,
                               _d(obsStats), N, S, _d(p), _d(r))


def fastUpdateCounts(bedInterval, obs, obsStats, segRatios):
    """bedInterval = (chrom, start, end, state) in TABLE coordinates."""
    obs, nb = _obs(obs)
    _, K = obs.shape
    _, N, S = obsStats.shape
    r = _f64(segRatios)
    lib().orc_update_counts(obs.ctypes.data_as(ctypes.c_void_p), nb, K,
                            ctypes.c_long(int(bedInterval[1])), ctypes.c_long(int(bedInterval[2])),
                            int(bedInterval[3]), _d(obsStats), N, S, _d(r))


def estep_sequence(obs, logProbs, normalize, log_startprob, log_transmat, segRatios,
                   start_stats, trans_stats, obs_stats):
    obs, nb = _obs(obs)
    T, K = obs.shape
    tab = _f64(logProbs)
    _, N, S = tab.shape
    a, b, r = _f64(log_startprob), _f64(log_transmat), _f64(segRatios)
    return lib().orc_estep_sequence(obs.ctypes.data_as(ctypes.c_void_p), nb, ctypes.c_long(T), K,
                                    _d(tab), N, S, ctypes.c_double(normalize), _d(a), _d(b), _d(r),
                                    _d(start_stats), _d(trans_stats), _d(obs_stats),
                                    int(obs_stats.shape[2]))


def sweep_sequence(obs, logProbs, normalize, log_startprob, log_transmat, segRatios=None):
    """emission + forward + backward + MAP + Viterbi for one sequence.
    Returns dict(logprob, map_score, vit_logprob, vit_states, map_states)."""
    obs, nb = _obs(obs)
    T, K = obs.shape
    tab = _f64(logProbs)
    _, N, S = tab.shape
    a, b, r = _f64(log_startprob), _f64(log_transmat), _f64(segRatios)
    vit = np.empty(T, dtype=np.int64)
    mp = np.empty(T, dtype=np.int64)
    out3 = np.zeros(3)
    lib().orc_sweep_sequence(obs.ctypes.data_as(ctypes.c_void_p), nb, ctypes.c_long(T), K,
                             _d(tab), N, S, ctypes.c_double(normalize), _d(a), _d(b), _d(r),
                             vit.ctypes.data_as(_I64), mp.ctypes.data_as(_I64), _d(out3))
    return dict(logprob=out3[0], map_score=out3[1], vit_logprob=out3[2],
                vit_states=vit, map_states=mp)
