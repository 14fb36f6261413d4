"""ctypes binding of libtehmm_b200.so (include/tehmm_b200.h).

There is NO CPU fallback: if the shared library is missing, or no CUDA device is
visible when a context is requested, the call raises.  (The CPU oracle under
oracle/ is test infrastructure and is never imported from here.)
"""
import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TEHMM_B200_LIB") or os.path.join(_HERE, "libtehmm_b200.so")   # override: kernel experiments only

TEHMM_OK, TEHMM_EINVAL, TEHMM_ECUDA, TEHMM_ENOMEM, TEHMM_ESTATE, TEHMM_ELIMIT = 0, -1, -2, -3, -4, -5
F32, F64 = 0, 1
BWD_POSTERIORS, BWD_MAP, BWD_TRANS, BWD_RENORM_EPS = 1, 2, 4, 8
MAX_STATES = 64
DECODE_VITERBI, DECODE_MAP = 0, 1

_c_void = ctypes.c_void_p
_c_i64 = ctypes.c_int64
_c_int = ctypes.c_int
_c_dbl = ctypes.c_double
_c_u64 = ctypes.c_uint64

# name -> (restype, argtypes); every symbol include/tehmm_b200.h declares
SIGNATURES = {
    "tehmm_abi_version": (_c_int, []),
    "tehmm_last_error": (ctypes.c_char_p, []),
    "tehmm_device_count": (_c_int, []),
    "tehmm_ctx_create": (_c_int, [_c_int, ctypes.POINTER(_c_void)]),
    "tehmm_ctx_destroy": (_c_int, [_c_void]),
    "tehmm_ctx_sync": (_c_int, [_c_void]),
    "tehmm_ctx_set_stream": (_c_int, [_c_void, _c_u64]),
    "tehmm_ctx_stream": (_c_u64, [_c_void]),
    "tehmm_ctx_launch_count": (_c_i64, [_c_void]),
    "tehmm_ctx_set_option": (_c_int, [_c_void, ctypes.c_char_p, _c_i64]),
    "tehmm_ctx_get_stat": (_c_i64, [_c_void, ctypes.c_char_p]),
    "tehmm_ctx_check": (_c_int, [_c_void, ctypes.POINTER(_c_i64)]),
    "tehmm_strict_all_log_probs": (_c_int, [_c_void, _c_void, _c_int, _c_i64, _c_int, _c_void, _c_int, _c_int, _c_void, _c_dbl, _c_void]),
    "tehmm_strict_forward": (_c_int, [_c_void, _c_i64, _c_int, _c_void, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_strict_backward": (_c_int, [_c_void, _c_i64, _c_int, _c_void, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_strict_viterbi": (_c_int, [_c_void, _c_i64, _c_int, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_strict_log_sum_lneta": (_c_int, [_c_void, _c_i64, _c_int, _c_void, _c_void, _c_void, _c_void, _c_dbl, _c_void, _c_void]),
    "tehmm_strict_accumulate_stats": (_c_int, [_c_void, _c_void, _c_int, _c_i64, _c_int, _c_void, _c_int, _c_int, _c_void, _c_void]),
    "tehmm_strict_update_counts": (_c_int, [_c_void, _c_void, _c_int, _c_i64, _c_int, _c_i64, _c_i64, _c_int, _c_void, _c_int, _c_int, _c_void]),
    "tehmm_supervised_counts": (_c_int, [_c_void, _c_void, _c_int, _c_i64, _c_int, _c_i64, _c_void, _c_void, _c_void, _c_void, _c_void, _c_int, _c_int]),
    "tehmm_set_model": (_c_int, [_c_void, _c_int, _c_int, _c_int, _c_void, _c_void, _c_void, _c_dbl, _c_void]),
    "tehmm_set_batch": (_c_int, [_c_void, _c_void, _c_int, _c_i64, _c_void]),
    "tehmm_batch_total": (_c_i64, [_c_void]),
    "tehmm_batch_chunks": (_c_i64, [_c_void]),
    "tehmm_lattice_stride": (_c_int, [_c_void]),
    "tehmm_scratch_bytes": (_c_i64, [_c_void, _c_int]),
    "tehmm_run_emission": (_c_int, [_c_void, _c_int, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_emission_rows_supported": (_c_int, [_c_void, _c_int]),
    "tehmm_run_emission_rows": (_c_int, [_c_void, _c_int, _c_void, _c_void, _c_void, _c_void, _c_i64, _c_i64, _c_u64]),
    "tehmm_run_emission_f64": (_c_int, [_c_void, _c_void, _c_void]),
    "tehmm_run_forward": (_c_int, [_c_void, _c_int, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_run_backward": (_c_int, [_c_void, _c_int, _c_int, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_run_emission_stats": (_c_int, [_c_void, _c_int, _c_void, _c_void, _c_void, _c_int, _c_void]),
    "tehmm_viterbi_workspace_bytes": (_c_i64, [_c_void, _c_int]),
    "tehmm_run_viterbi": (_c_int, [_c_void, _c_int, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_fold_ratios": (_c_int, [_c_void, _c_int, _c_void, _c_void, _c_void]),
    "tehmm_ratio_diag_counts": (_c_int, [_c_void, _c_int, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_track_fill": (_c_int, [_c_void, _c_void, _c_i64, _c_int, _c_int, _c_int, ctypes.c_int32]),
    "tehmm_rasterize_intervals": (_c_int, [_c_void, _c_void, _c_void, _c_void, _c_void, _c_i64, _c_i64, _c_i64, _c_void, _c_int, _c_int, _c_int]),
    "tehmm_segment_table": (_c_int, [_c_void, _c_void, _c_i64, _c_int, _c_int, _c_i64, _c_void, _c_void, _c_void, _c_int, _c_i64, _c_i64, _c_int, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_compress_segments": (_c_int, [_c_void, _c_void, _c_i64, _c_int, _c_int, _c_void, _c_i64, _c_void, _c_void]),
    "tehmm_run_sum": (_c_int, [_c_void, _c_void, _c_void, _c_i64]),
    "tehmm_bed_open": (_c_int, [ctypes.c_char_p, ctypes.c_char_p, _c_i64, _c_i64, _c_int, _c_int, _c_int, ctypes.POINTER(_c_void)]),
    "tehmm_bed_count": (_c_i64, [_c_void]),
    "tehmm_bed_nunique": (_c_i64, [_c_void]),
    "tehmm_bed_unique": (ctypes.c_char_p, [_c_void, _c_i64]),
    "tehmm_bed_fetch": (_c_int, [_c_void, _c_void, _c_void, _c_void]),
    "tehmm_bed_close": (None, [_c_void]),
    "tehmm_decode_host": (_c_int, [_c_void, _c_void, _c_i64, _c_int, _c_i64, _c_void, _c_int, _c_int, _c_void, _c_void, _c_void]),
    "tehmm_decode_host_both": (_c_int, [_c_void, _c_void, _c_i64, _c_int, _c_i64, _c_void, _c_int, _c_void, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_decode_host_ratios": (_c_int, [_c_void, _c_void, _c_i64, _c_int, _c_i64, _c_void, _c_void, _c_int, _c_int, _c_void, _c_void, _c_void]),
    "tehmm_decode_host_both_ratios": (_c_int, [_c_void, _c_void, _c_i64, _c_int, _c_i64, _c_void, _c_void, _c_int, _c_void, _c_void, _c_void, _c_void, _c_void]),
    "tehmm_decode_host_bytes": (_c_i64, [_c_void, _c_int]),
    "tehmm_host_pool_selftest": (_c_i64, [_c_int, _c_i64]),
    "tehmm_decode_host_phase_ms": (ctypes.c_double, [_c_void, _c_int]),
    "tehmm_ctx_device": (_c_int, [_c_void]),
    "tehmm_model_dims": (_c_int, [_c_void, _c_void, _c_void, _c_void]),
    "tehmm_path_score": (_c_int, [_c_void, _c_void, _c_void, _c_void, _c_i64, _c_i64, _c_void, _c_void]),
    "tehmm_states_to_bed": (_c_int, [_c_int, ctypes.c_char_p, _c_i64, _c_void, _c_i64, _c_void, _c_void, _c_i64, _c_void, _c_int]),
    "tehmm_scores_to_bed": (_c_int, [_c_int, ctypes.c_char_p, _c_i64, _c_void, _c_i64, _c_void, _c_void, _c_i64]),
    "tehmm_widen_states": (_c_int, [_c_void, _c_void, _c_void, _c_i64]),
    "tehmm_convert_lattice": (_c_int, [_c_void, _c_int, _c_void, _c_void, _c_i64]),
}

_lib = None
_lock = threading.Lock()


class TehmmError(RuntimeError):
    pass


def load():
    """dlopen libtehmm_b200.so (no GPU needed for this step) and type every entry point."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ImportError(
                    "tehmm_b200: %s is missing. Build it with `python -m tehmm_b200.build` "
                    "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)      # AttributeError if the .so lacks a declared symbol
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc):
    if rc == TEHMM_OK:
        return
    msg = load().tehmm_last_error().decode("utf-8", "replace")
    if rc == TEHMM_EINVAL:
        raise AssertionError(msg)          # the reference asserts on bad shapes (_emission.pyx:24-32)
    raise TehmmError("libtehmm_b200 error %d: %s" % (rc, msg))


def ptr(a):
    """void* of a NumPy array (None -> NULL)."""
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        assert tuple(a.shape) == tuple(shape), "expected shape %s, got %s" % (shape, a.shape)
    return a


class Context(object):
    """Owns one tehmm_ctx.  One per (process, device, thread); see engine.get_context()."""

    def __init__(self, device=0):
        lib = load()
        if lib.tehmm_device_count() <= 0:
            raise TehmmError("tehmm_b200: no CUDA device is visible and there is no CPU fallback")
        h = ctypes.c_void_p()
        check(lib.tehmm_ctx_create(int(device), ctypes.byref(h)))
        self.handle = h
        self.device = int(device)
        self.lib = lib

    def close(self):
        if self.handle:
            self.lib.tehmm_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        check(self.lib.tehmm_ctx_sync(self.handle))

    def set_option(self, name, value):
        check(self.lib.tehmm_ctx_set_option(self.handle, name.encode(), int(value)))

    def stat(self, name):
        return int(self.lib.tehmm_ctx_get_stat(self.handle, name.encode()))

    def check(self):
        """deferred verification (option "defer"): wait for the stream; number of chunk
        boundaries that failed verification since the last check (0 = results stand)"""
        n = _c_i64(0)
        check(self.lib.tehmm_ctx_check(self.handle, ctypes.byref(n)))
        return int(n.value)

    def optimistic(self, fn):
        """run fn() with deferred verification; if any boundary failed, run it again with the
        synchronous verify / repair loop.  fn must be a pure function of device state it does
        not overwrite (every engine pass is)."""
        # a refused attempt costs the stages twice, and batches that need repairs tend to need them
        # again (same model, same chunk boundaries): back off to the synchronous loop for a growing
        # number of calls after a refusal, come back when attempts stand again
        skip = getattr(self, "_defer_skip", 0)
        if os.environ.get("TEHMM_NO_DEFER"):      # measurement switch: always the synchronous loop
            return fn()
        if skip > 0:
            self._defer_skip = skip - 1
            return fn()
        self.set_option("defer", 1)
        try:
            out = fn()
        finally:
            self.set_option("defer", 0)
        penalty = getattr(self, "_defer_penalty", 0)
        if self.check() != 0:
            self._defer_penalty = min(256, max(4, 2 * penalty))
            self._defer_skip = self._defer_penalty
            out = fn()
        else:
            self._defer_penalty = penalty // 2
        return out

    @property
    def launches(self):
        return int(self.lib.tehmm_ctx_launch_count(self.handle))


_ctx_local = threading.local()


def set_thread_device(device):
    """the device the calling thread's contexts default to (None: back to TEHMM_B200_DEVICE / LOCAL_RANK)"""
    _ctx_local.device = None if device is None else int(device)


def get_context(device=None):
    """Process-global, per-thread, per-device context cache.  Never stored on model
    objects: they are pickled / deep-copied (modelIO.py:26-32, hmm.py:694)."""
    if device is None:
        device = getattr(_ctx_local, "device", None)          # set_thread_device: replicate training
    if device is None:
        device = int(os.environ.get("TEHMM_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        n = load().tehmm_device_count()
        if n > 0:
            device %= n
    cache = getattr(_ctx_local, "cache", None)
    if cache is None:
        cache = _ctx_local.cache = {}
    ctx = cache.get(device)
    if ctx is None or ctx.handle is None:
        ctx = cache[device] = Context(device)
    return ctx
