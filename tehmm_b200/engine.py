"""Batched device path behind MultitrackHmm / IndependentMultinomialEmissionModel.

PyTorch is used only for plumbing: device buffers, H2D/D2H copies, the CUDA
stream and (in parallel.py) torch.distributed.  All arithmetic is in
libtehmm_b200.so.  Sequences of one call are concatenated along time and
described by row offsets; the library partitions time into chunks and runs one
warp per chunk (see csrc/forward.cu for the speculate / verify / repair scheme).
"""
import ctypes
import mmap
import os
import threading
import weakref

import numpy as np

from . import _lib
from .track import is_track_table

_PRECISION = os.environ.get("TEHMM_B200_PRECISION", "f32").lower()


def set_precision(p):
    """'f32' (production) or 'f64' (verification) element type of the batched lattices."""
    global _PRECISION
    p = str(p).lower()
    assert p in ("f32", "f64")
    _PRECISION = p


def get_precision():
    return _PRECISION


def _torch():
    import torch
    return torch


def as_obs_array(obs):
    """Observation matrix of anything the reference accepts: TrackTable, or an
    ndarray / nested list of any numeric dtype (non-fast dtypes are indexed with
    int(symbol) by the reference, emission.py:176,239)."""
    if is_track_table(obs):
        obs = obs.getNumPyArray()
    a = np.asarray(obs)
    if a.ndim == 1:
        a = a.reshape(-1, 1)
    assert a.ndim == 2, "observations must be (T, numTracks)"
    if a.dtype in (np.dtype(np.uint8), np.dtype(np.uint16), np.dtype(np.int32)):
        return np.ascontiguousarray(a)
    return np.ascontiguousarray(a.astype(np.int32))


class _ResultPool(object):
    """Host memory for the int64 state paths handed back by decode().

    A fresh 80 MB NumPy array costs ~4 ms of first-touch page faults per 10 M steps,
    as much as the rest of the decode call.  Blocks are anonymous mmaps; an array
    handed out is np.frombuffer(block), so it and every slice taken from it keep
    the block's export alive, and a weakref finalizer returns the block to the pool
    only when the last of them is unreachable -- the caller sees ordinary, writable,
    independent int64 arrays."""
    MAX_FREE = 4
    MAX_FREE_BYTES = 512 << 20       # what the pool may keep mapped between calls (a 250 M-step path is 2 GB)

    def __init__(self):
        self._free = []
        self._lock = threading.Lock()
        self._registered = {}            # id(block) -> address: page-locked with cudaHostRegister

    # With TEHMM_PIN_RESULTS=1 (or TEHMM_WIDEN=gpu) blocks are page-locked (cudaHostRegister) so that
    # tehmm_decode_host can let the DMA engine write the int64 path straight into the result (device-side
    # widening, csrc/host.cu) instead of widening on the host's cores.  Off by default: measured slower
    # (profiles/r02_notes_e2e.md).  Registration costs milliseconds per block, paid once: blocks are recycled.
    @staticmethod
    def _address(block):
        c = ctypes.c_char.from_buffer(block)
        try:
            return ctypes.addressof(c)
        finally:
            del c                        # drop the extra buffer export at once

    def _register(self, block):
        if os.environ.get("TEHMM_PIN_RESULTS", "0") != "1" and os.environ.get("TEHMM_WIDEN") != "gpu":
            return
        try:
            torch = _torch()
            if not torch.cuda.is_available():
                return
            addr = self._address(block)
            rc = torch.cuda.cudart().cudaHostRegister(addr, len(block), 0)
            if int(rc) == 0:
                self._registered[id(block)] = addr
        except Exception:
            pass

    def _unregister(self, block):
        addr = self._registered.pop(id(block), None)
        if addr is not None:
            try:
                _torch().cuda.cudart().cudaHostUnregister(addr)
            except Exception:
                pass

    def _put(self, block):
        with self._lock:
            held = sum(len(b) for b in self._free)
            if len(self._free) < self.MAX_FREE and held + len(block) <= self.MAX_FREE_BYTES:
                self._free.append(block)
                return
        # over the cap: the block is simply not kept -- it is unmapped when the dying array releases
        # its buffer export (closing it here would raise: the export is still counted in a finalizer)
        self._unregister(block)

    def empty_int64(self, n):
        nbytes = max(8, int(n) * 8)
        block = None
        with self._lock:
            for i, b in enumerate(self._free):
                if nbytes <= len(b) <= 2 * nbytes + (4 << 20):
                    block = self._free.pop(i)
                    break
        if block is None:
            # PRIVATE: like ordinary heap memory, a forked child (teHmm's --proc workers) gets its own
            # copy-on-write view (mmap's default for fd -1 is a SHARED mapping)
            block = mmap.mmap(-1, (nbytes + (2 << 20) - 1) & ~((2 << 20) - 1),
                              flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS)
            try:                                  # first touch in 2 MB pages where the kernel allows it
                block.madvise(mmap.MADV_HUGEPAGE)
            except (AttributeError, OSError, ValueError):
                pass
            self._register(block)
        arr = np.frombuffer(block, dtype=np.int64, count=int(n))
        weakref.finalize(arr, self._put, block)
        return arr


_result_pool = _ResultPool()


class Engine(object):
    """One per Context.  Holds nothing of the model between calls except what
    upload_model() put on the device."""

    def __init__(self, ctx=None):
        self.ctx = ctx if ctx is not None else _lib.get_context()
        self.lib = self.ctx.lib
        torch = _torch()
        self.torch = torch
        self.device = torch.device("cuda", self.ctx.device)
        self._keep = {}
        self.N = self.K = self.S = None
        self.batch_token = None        # set by fit(): the resident batch is reused across EM iterations
        self.batch_ratios = None

    # ------------------------------------------------------------ plumbing
    def _bind_stream(self):
        torch = self.torch
        torch.cuda.set_device(self.device)
        s = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.tehmm_ctx_set_stream(self.ctx.handle, ctypes.c_uint64(s)))

    def _prec(self, precision=None):
        p = precision or _PRECISION
        return (_lib.F32, self.torch.float32) if p == "f32" else (_lib.F64, self.torch.float64)

    @staticmethod
    def _p(t):
        return None if t is None else ctypes.c_void_p(t.data_ptr())

    def upload_model(self, log_start, log_trans, table, normalize, track_nsym=None):
        self._bind_stream()
        ls = _lib.f64(log_start)
        lt = _lib.f64(log_trans)
        tab = _lib.f64(table)
        K, N, S = tab.shape
        assert ls.shape == (N,) and lt.shape == (N, N)
        ns = None
        if track_nsym is not None:
            ns = np.ascontiguousarray(np.minimum(np.asarray(track_nsym, dtype=np.int64), S), dtype=np.int32)
            assert ns.shape == (K,)
        _lib.check(self.lib.tehmm_set_model(self.ctx.handle, N, K, S, _lib.ptr(ls), _lib.ptr(lt), _lib.ptr(tab),
                                            float(normalize), _lib.ptr(ns)))
        self.N, self.K, self.S = N, K, S
        self.LD = int(self.lib.tehmm_lattice_stride(self.ctx.handle))   # row stride of the device lattices

    def upload_batch(self, obs_list, pinned=None):
        """Concatenate, copy to the device and describe to the library.
        Returns (offsets ndarray int64[nseq+1])."""
        torch = self.torch
        self._bind_stream()
        self.batch_token = None
        arrays = [as_obs_array(o) for o in obs_list]
        assert len(arrays) > 0
        K = arrays[0].shape[1]
        for a in arrays:
            assert a.shape[1] == K, "all sequences must have the same number of tracks"
        dt = arrays[0].dtype
        if any(a.dtype != dt for a in arrays):
            dt = np.dtype(np.int32)
            arrays = [a.astype(np.int32) for a in arrays]
        lens = np.array([a.shape[0] for a in arrays], dtype=np.int64)
        offsets = np.zeros(len(arrays) + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        host = arrays[0] if len(arrays) == 1 else np.concatenate(arrays, axis=0)
        if dt == np.uint16:   # torch has no full uint16 support everywhere: move raw bytes
            d_obs = torch.from_numpy(host.view(np.uint8).reshape(-1)).to(self.device)
        else:
            d_obs = torch.from_numpy(host.reshape(-1)).to(self.device)
        self._keep["obs"] = d_obs
        self._keep["offsets"] = offsets
        _lib.check(self.lib.tehmm_set_batch(self.ctx.handle, self._p(d_obs), dt.itemsize, len(arrays),
                                            _lib.ptr(offsets)))
        self.total = int(offsets[-1])
        self.nseq = len(arrays)
        self.obs_bytes = dt.itemsize
        self.h2d_bytes = host.nbytes
        return offsets

    @staticmethod
    def _host_arrays(obs_list):
        """observation matrices of a host-buffer call: (arrays, dtype, offsets int64[nseq+1], void* table)"""
        arrays = [as_obs_array(o) for o in obs_list]
        assert len(arrays) > 0
        K = arrays[0].shape[1]
        for a in arrays:
            assert a.shape[1] == K, "all sequences must have the same number of tracks"
        dt = arrays[0].dtype
        if any(a.dtype != dt for a in arrays):
            dt = np.dtype(np.int32)
            arrays = [a.astype(np.int32) for a in arrays]
        offsets = np.zeros(len(arrays) + 1, dtype=np.int64)
        np.cumsum([a.shape[0] for a in arrays], out=offsets[1:])
        ptrs = (ctypes.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])   # no concatenation
        return arrays, dt, offsets, ptrs

    @staticmethod
    def _host_ratios(ratios, offsets):
        """per-sequence segment ratios -> (float64 arrays kept alive, double* table), or (None, None) when no
        sequence has any; the library checks the values (finite, > 0)"""
        if ratios is None or all(r is None for r in ratios):
            return None, None
        n = len(offsets) - 1
        assert len(ratios) == n, "one entry of ratios per sequence"
        keep = [None if r is None else np.ascontiguousarray(r, dtype=np.float64).reshape(-1) for r in ratios]
        for i, r in enumerate(keep):
            assert r is None or r.shape[0] == offsets[i + 1] - offsets[i], \
                "sequence %d: %d segment ratios for %d observations" % (i, r.shape[0], offsets[i + 1] - offsets[i])
        return keep, (ctypes.c_void_p * n)(*[None if r is None else r.ctypes.data for r in keep])

    def decode_host(self, obs_list, algorithm, precision=None, ratios=None):
        """The whole decode call with host buffers on both sides, in the library
        (tehmm_decode_host: pinned staging + worker threads in, uint8 states over PCIe and
        widened to the reference's int64 out).  ratios: None, or per sequence an array of
        segment ratios or None (tehmm_decode_host_ratios); the Viterbi DP takes them, the
        emission and MAP decoding do not, as in the reference's decode.
        Returns (logprob float64[nseq], score float64[nseq] (MAP only), [int64 states])."""
        self._bind_stream()
        self.batch_token = None
        prec, _ = self._prec(precision)
        arrays, dt, offsets, ptrs = self._host_arrays(obs_list)
        keep, rptrs = self._host_ratios(ratios, offsets)
        n = len(arrays)
        total = int(offsets[-1])
        states = _result_pool.empty_int64(total)
        logprob = np.empty(n, dtype=np.float64)
        score = np.empty(n, dtype=np.float64)
        if rptrs is None:
            _lib.check(self.lib.tehmm_decode_host(self.ctx.handle, ptrs, n, dt.itemsize, n, _lib.ptr(offsets),
                                                  int(algorithm), prec, _lib.ptr(states), _lib.ptr(logprob),
                                                  _lib.ptr(score)))
        else:
            _lib.check(self.lib.tehmm_decode_host_ratios(self.ctx.handle, ptrs, n, dt.itemsize, n, _lib.ptr(offsets),
                                                         rptrs, int(algorithm), prec, _lib.ptr(states),
                                                         _lib.ptr(logprob), _lib.ptr(score)))
        del keep
        self._keep.pop("obs", None)            # the batch now points into the library's arena
        self._keep["offsets"] = offsets
        self.total, self.nseq = total, n
        self.h2d_bytes = int(self.lib.tehmm_decode_host_bytes(self.ctx.handle, 0))
        self.d2h_bytes = int(self.lib.tehmm_decode_host_bytes(self.ctx.handle, 1))
        return logprob, score, [states[offsets[i]:offsets[i + 1]] for i in range(n)]

    def decode_host_both(self, obs_list, precision=None, ratios=None):
        """Viterbi AND posterior (MAP) decoding of the same observations in one call
        (tehmm_decode_host_both): one upload, one emission pass.  ratios as for decode_host:
        the Viterbi path takes them, the MAP path and the forward log-likelihood do not.  Returns
        (viterbi logprob[nseq], [viterbi states], map score[nseq], [map states], forward logprob[nseq])."""
        self._bind_stream()
        self.batch_token = None
        prec, _ = self._prec(precision)
        arrays, dt, offsets, ptrs = self._host_arrays(obs_list)
        keep, rptrs = self._host_ratios(ratios, offsets)
        n = len(arrays)
        total = int(offsets[-1])
        vst, mst = _result_pool.empty_int64(total), _result_pool.empty_int64(total)
        vlp, msc, flp = (np.empty(n, dtype=np.float64) for _ in range(3))
        if rptrs is None:
            _lib.check(self.lib.tehmm_decode_host_both(self.ctx.handle, ptrs, n, dt.itemsize, n, _lib.ptr(offsets), prec,
                                                       _lib.ptr(vst), _lib.ptr(vlp), _lib.ptr(mst), _lib.ptr(msc),
                                                       _lib.ptr(flp)))
        else:
            _lib.check(self.lib.tehmm_decode_host_both_ratios(self.ctx.handle, ptrs, n, dt.itemsize, n,
                                                              _lib.ptr(offsets), rptrs, prec, _lib.ptr(vst),
                                                              _lib.ptr(vlp), _lib.ptr(mst), _lib.ptr(msc),
                                                              _lib.ptr(flp)))
        del keep
        self._keep.pop("obs", None)
        self._keep["offsets"] = offsets
        self.total, self.nseq = total, n
        self.h2d_bytes = int(self.lib.tehmm_decode_host_bytes(self.ctx.handle, 0))
        self.d2h_bytes = int(self.lib.tehmm_decode_host_bytes(self.ctx.handle, 1))
        cut = lambda st: [st[offsets[i]:offsets[i + 1]] for i in range(n)]
        return vlp, cut(vst), msc, cut(mst), flp

    def use_device_batch(self, d_obs, obs_bytes, offsets):
        """Batch already resident on the device (bench / multi-call reuse)."""
        self._bind_stream()
        self.batch_token = None
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self._keep["obs"] = d_obs
        self._keep["offsets"] = offsets
        _lib.check(self.lib.tehmm_set_batch(self.ctx.handle, self._p(d_obs), int(obs_bytes), len(offsets) - 1,
                                            _lib.ptr(offsets)))
        self.total = int(offsets[-1])
        self.nseq = len(offsets) - 1
        self.obs_bytes = int(obs_bytes)
        return offsets

    def upload_ratios(self, ratios_list):
        """list of per-sequence float64 arrays (or None) -> device tensor or None.
        A sequence without ratios gets 1.0: right for the forward / backward passes and the E-step,
        where the ratio terms vanish at 1.0, but not for the Viterbi DP of a batch that mixes
        sequences with and without ratios (the reference's from-state-0 term applies whenever
        ratios are given, _hmm.pyx:234-237).  Engine.viterbi keeps this; decode_host(ratios=...)
        decodes such batches as the reference does."""
        if ratios_list is None or all(r is None for r in ratios_list):
            return None
        offsets = self._keep["offsets"]
        host = np.ones(self.total, dtype=np.float64)
        for i, r in enumerate(ratios_list):
            if r is not None:
                r = np.asarray(r, dtype=np.float64)
                assert r.shape[0] == offsets[i + 1] - offsets[i]
                host[offsets[i]:offsets[i + 1]] = r
        return self.torch.from_numpy(host).to(self.device)

    def supervised_counts(self, row_start, row_end, state, obs_stats, d_ratios=None):
        """Supervised emission counts of labelled intervals over the current batch (upload_batch or
        use_device_batch) in one device pass (tehmm_supervised_counts).  Interval i covers the
        batch's global rows [row_start[i], row_end[i]) with state[i]; d_ratios (device tensor or host
        array of `total` weights, or None for 1.0) is the concatenation upload_ratios builds.
        obs_stats (K, N, S) float64 is updated in place, bit-identical to one
        _emission.fastUpdateCounts per interval in the given order.  Raises TehmmError, leaving
        obs_stats as it was, for rows outside the batch, states outside [0, N) or a counted symbol >= S."""
        torch = self.torch
        d_obs = self._keep.get("obs")
        if d_obs is None:
            raise _lib.TehmmError("supervised_counts: no device batch (upload_batch or use_device_batch first)")
        assert isinstance(obs_stats, np.ndarray) and obs_stats.dtype == np.float64 and obs_stats.ndim == 3
        assert obs_stats.flags.c_contiguous, "obs_stats must be C-contiguous (it is updated in place)"
        K, N, S = obs_stats.shape
        rs = np.ascontiguousarray(row_start, dtype=np.int64).reshape(-1)
        re = np.ascontiguousarray(row_end, dtype=np.int64).reshape(-1)
        st64 = np.asarray(state, dtype=np.int64).reshape(-1)
        assert rs.shape == re.shape == st64.shape, "row_start, row_end and state must have the same length"
        if rs.size and (st64.min() < 0 or st64.max() >= N):
            bad = int(np.flatnonzero((st64 < 0) | (st64 >= N))[0])
            raise _lib.TehmmError("supervised_counts: interval %d has state %d outside [0, %d)" % (bad, int(st64[bad]), N))
        st = np.ascontiguousarray(st64, dtype=np.int32)
        nbytes = d_obs.numel() * d_obs.element_size()
        if nbytes != self.total * K * self.obs_bytes:
            raise _lib.TehmmError("supervised_counts: the batch is not a (%d, %d) matrix of %d-byte symbols"
                                  % (self.total, K, self.obs_bytes))
        if d_ratios is not None:
            if not torch.is_tensor(d_ratios):
                d_ratios = torch.from_numpy(_lib.f64(d_ratios)).to(self.device)
            assert d_ratios.dtype == torch.float64 and d_ratios.numel() == self.total and d_ratios.is_contiguous()
        self._bind_stream()
        rc = self.lib.tehmm_supervised_counts(self.ctx.handle, self._p(d_obs), int(self.obs_bytes), int(self.total), K,
                                              int(rs.size), _lib.ptr(rs), _lib.ptr(re), _lib.ptr(st), self._p(d_ratios),
                                              _lib.ptr(obs_stats), N, S)
        if rc != _lib.TEHMM_OK:
            raise _lib.TehmmError("libtehmm_b200 error %d: %s" % (rc, self.lib.tehmm_last_error().decode("utf-8", "replace")))
        return obs_stats

    def scratch(self, prec):
        n = int(self.lib.tehmm_scratch_bytes(self.ctx.handle, prec))
        buf = self._keep.get("scratch")
        if buf is None or buf.numel() < n:
            buf = self.torch.empty(max(n, 256), dtype=self.torch.uint8, device=self.device)
            self._keep["scratch"] = buf
        return buf

    def empty(self, shape, dtype):
        return self.torch.empty(shape, dtype=dtype, device=self.device)

    # ------------------------------------------------------------ device -> host
    # A plain tensor.cpu() lands in pageable memory through the driver's bounce
    # buffer (measured ~2 GB/s on the B200 box: 38 ms for 80 MB of states).  Large
    # results go through two cached pinned staging buffers instead, the copy out
    # of chunk i overlapping the transfer of chunk i+1.
    _STAGE_BYTES = 32 << 20

    def _stages(self):
        st = self._keep.get("stages")
        if st is None:
            torch = self.torch
            st = [torch.empty(self._STAGE_BYTES, dtype=torch.uint8).pin_memory() for _ in range(2)]
            st.append([torch.cuda.Event() for _ in range(2)])
            self._keep["stages"] = st
        return st

    def to_host(self, t):
        """device tensor -> NumPy array of the same shape and dtype (fresh, pageable)."""
        torch = self.torch
        nbytes = t.numel() * t.element_size()
        if nbytes <= (1 << 20):
            return t.cpu().numpy()
        src = t.contiguous().reshape(-1).view(torch.uint8)
        out = torch.empty(t.shape, dtype=t.dtype)
        dst = out.reshape(-1).view(torch.uint8)
        s0, s1, ev = self._stages()
        stage = (s0, s1)
        chunk = self._STAGE_BYTES
        nchunk = (nbytes + chunk - 1) // chunk
        for i in range(min(2, nchunk)):
            a, b = i * chunk, min(nbytes, (i + 1) * chunk)
            stage[i][:b - a].copy_(src[a:b], non_blocking=True)
            ev[i].record()
        for i in range(nchunk):
            a, b = i * chunk, min(nbytes, (i + 1) * chunk)
            ev[i & 1].synchronize()
            dst[a:b].copy_(stage[i & 1][:b - a])
            j = i + 2
            if j < nchunk:
                a2, b2 = j * chunk, min(nbytes, (j + 1) * chunk)
                stage[i & 1][:b2 - a2].copy_(src[a2:b2], non_blocking=True)
                ev[i & 1].record()
        return out.numpy()

    def states_to_host(self, d_states_u8):
        """uint8 device states -> int64 host array: 1 byte per step over PCIe, widened by
        the host's cores (the reference API returns int64, basehmm.py:357, _hmm.pyx:210)."""
        torch = self.torch
        n = d_states_u8.numel()
        if n <= (1 << 20):
            return d_states_u8.cpu().to(torch.int64).numpy()
        pin = self._keep.get("pin_states")
        if pin is None or pin.numel() < n:
            pin = torch.empty(n, dtype=torch.uint8).pin_memory()
            self._keep["pin_states"] = pin
        pin[:n].copy_(d_states_u8, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return pin[:n].to(torch.int64).numpy()

    # ------------------------------------------------------------ device ops
    def run_emission(self, prec, tdt, d_ratios, want_log, want_lin):
        n = self.total * self.LD
        elog = self.empty(n, tdt) if want_log else None
        blin = self.empty(n, tdt) if want_lin else None
        rowmax = self.empty(self.total, self.torch.float64)
        _lib.check(self.lib.tehmm_run_emission(self.ctx.handle, prec, self._p(d_ratios), self._p(elog),
                                               self._p(blin), self._p(rowmax)))
        return elog, blin, rowmax

    def fold_ratios(self, prec, d_ratios, blin, rowmax):
        """segment ratios of the forward / backward recursions folded into the linear emission lattice
        (tehmm_fold_ratios): the passes that follow run without ratios, on the tile kernels"""
        if d_ratios is not None:
            _lib.check(self.lib.tehmm_fold_ratios(self.ctx.handle, prec, self._p(d_ratios), self._p(blin), self._p(rowmax)))
        return None

    def run_forward(self, prec, tdt, blin, rowmax, d_ratios, want_alpha=True):
        alpha = self.empty(self.total * self.LD, tdt) if want_alpha else None
        logprob = self.empty(self.nseq, self.torch.float64)
        sc = self.scratch(prec)
        _lib.check(self.lib.tehmm_run_forward(self.ctx.handle, prec, self._p(blin), self._p(rowmax),
                                              self._p(d_ratios), self._p(alpha), self._p(logprob), self._p(sc)))
        return alpha, logprob

    def run_backward(self, prec, tdt, flags, blin, alpha, d_ratios, start_trans=None):
        torch = self.torch
        post = self.empty(self.total * self.LD, tdt) if flags & _lib.BWD_POSTERIORS else None
        mstates = self.empty(self.total, torch.uint8) if flags & _lib.BWD_MAP else None
        mscore = self.empty(self.nseq, torch.float64) if flags & _lib.BWD_MAP else None
        sc = self.scratch(prec)
        _lib.check(self.lib.tehmm_run_backward(self.ctx.handle, prec, flags, self._p(blin), self._p(alpha),
                                               self._p(d_ratios), self._p(post), self._p(mstates),
                                               self._p(mscore), self._p(start_trans), self._p(sc)))
        return post, mstates, mscore

    def run_emission_stats(self, prec, post, d_ratios, obs_stats, stats_S):
        sc = self.scratch(prec)
        _lib.check(self.lib.tehmm_run_emission_stats(self.ctx.handle, prec, self._p(post), self._p(d_ratios),
                                                     self._p(obs_stats), int(stats_S), self._p(sc)))

    def run_viterbi(self, prec, elog, d_ratios_em, d_ratios_dp, want64=True, rowmax=None):
        torch = self.torch
        bp = self.empty(int(self.lib.tehmm_viterbi_workspace_bytes(self.ctx.handle, prec)), torch.uint8)
        states = self.empty(self.total, torch.uint8)
        states64 = self.empty(self.total, torch.int64) if want64 else None
        logprob = self.empty(self.nseq, torch.float64)
        sc = self.scratch(prec)
        _lib.check(self.lib.tehmm_run_viterbi(self.ctx.handle, prec, self._p(elog), self._p(rowmax),
                                              self._p(d_ratios_em), self._p(d_ratios_dp), self._p(bp), self._p(states),
                                              self._p(states64), self._p(logprob), self._p(sc)))
        return states, states64, logprob

    def to_f64(self, prec, t):
        if prec == _lib.F64:
            return t
        out = self.empty(t.numel(), self.torch.float64)
        _lib.check(self.lib.tehmm_convert_lattice(self.ctx.handle, prec, self._p(t), self._p(out), t.numel()))
        return out

    def lattice_to_host(self, prec, t):
        """(total, LD) device lattice -> (total, N) float64 host array (padding dropped on the device)."""
        v = self.to_f64(prec, t).view(self.total, self.LD)
        if self.LD != self.N:
            v = v[:, :self.N].contiguous()
        return self.to_host(v)

    def split(self, host, width=None):
        """Cut a concatenated host array back into per-sequence views."""
        offsets = self._keep["offsets"]
        if width:
            host = host.reshape(-1, width)
        return [host[offsets[i]:offsets[i + 1]] for i in range(len(offsets) - 1)]

    # ------------------------------------------------------------ API-level ops
    def emission_frames(self, ratios_list=None):
        """allLogProbs for the current batch: list of (T_i, N) float64 (emission.py:179-198)."""
        d_r = self.upload_ratios(ratios_list)
        frame = self.empty(self.total * self.N, self.torch.float64)
        _lib.check(self.lib.tehmm_run_emission_f64(self.ctx.handle, self._p(d_r), self._p(frame)))
        return self.split(self.to_host(frame), self.N)

    def score(self, ratios_em=None, ratios_dp=None, precision=None):
        prec, tdt = self._prec(precision)
        d_re, d_rd = self.upload_ratios(ratios_em), self.upload_ratios(ratios_dp)
        _, blin, rowmax = self.run_emission(prec, tdt, d_re, False, True)
        d_rd = self.fold_ratios(prec, d_rd, blin, rowmax)
        # deferred verification (tehmm_ctx_check): one wait per call instead of one per stage
        _, logprob = self.ctx.optimistic(lambda: self.run_forward(prec, tdt, blin, rowmax, d_rd, want_alpha=False))
        return logprob.cpu().numpy()

    def posteriors(self, ratios_em=None, ratios_dp=None, renorm_eps=True, want_map=False,
                   want_post=True, precision=None):
        """score_samples / _decode_map for the batch (basehmm.py:238-273,332-359)."""
        prec, tdt = self._prec(precision)
        d_re, d_rd = self.upload_ratios(ratios_em), self.upload_ratios(ratios_dp)
        _, blin, rowmax = self.run_emission(prec, tdt, d_re, False, True)
        d_rd = self.fold_ratios(prec, d_rd, blin, rowmax)
        flags = (_lib.BWD_POSTERIORS if want_post else 0) | (_lib.BWD_MAP if want_map else 0) | \
                (_lib.BWD_RENORM_EPS if renorm_eps else 0)

        def stages():
            alpha, logprob = self.run_forward(prec, tdt, blin, rowmax, d_rd)
            return (logprob,) + tuple(self.run_backward(prec, tdt, flags, blin, alpha, d_rd))
        logprob, post, mstates, mscore = self.ctx.optimistic(stages)
        out = {"logprob": logprob.cpu().numpy()}
        if want_post:
            out["post"] = self.split(self.lattice_to_host(prec, post))
        if want_map:
            out["map_states"] = self.split(self.states_to_host(mstates))
            out["map_score"] = mscore.cpu().numpy()
        return out

    def viterbi(self, ratios_em=None, ratios_dp=None, precision=None):
        """decode(algorithm='viterbi') for the batch (basehmm.py:301-330, hmm.py:668-676)."""
        prec, tdt = self._prec(precision)
        d_re, d_rd = self.upload_ratios(ratios_em), self.upload_ratios(ratios_dp)
        elog, _, rowmax = self.run_emission(prec, tdt, d_re, True, False)
        states, _, logprob = self.ctx.optimistic(
            lambda: self.run_viterbi(prec, elog, d_re, d_rd, want64=False, rowmax=rowmax))
        return logprob.cpu().numpy(), self.split(self.states_to_host(states))

    # ------------------------------------------------------------ one window of a time-sharded sequence
    # (parallel.run_time_sharded: core = this rank's rows, window = core + halo on both sides)
    def viterbi_window(self, obs, core, window, precision=None):
        """Viterbi on obs[window]; returns what parallel.run_time_sharded needs: the core's
        states (int64), the float64 path score of the core rows, the states at a-1 / b-1 and
        the max-normalised delta rows at those two times."""
        torch = self.torch
        prec, tdt = self._prec(precision)
        (a, b), (w0, w1) = core, window
        self.upload_batch([obs[w0:w1]])
        elog, _, _ = self.run_emission(prec, tdt, None, True, False)
        lattice = self.empty(int(self.lib.tehmm_viterbi_workspace_bytes(self.ctx.handle, prec)), torch.uint8)
        states = self.empty(self.total, torch.uint8)
        logprob = self.empty(1, torch.float64)
        sc = self.scratch(prec)
        _lib.check(self.lib.tehmm_run_viterbi(self.ctx.handle, prec, self._p(elog), None, None, None,
                                              self._p(lattice), self._p(states), None, self._p(logprob), self._p(sc)))
        part = self.empty(1, torch.float64)
        _lib.check(self.lib.tehmm_path_score(self.ctx.handle, self._p(states), None, None, a - w0, b - w0,
                                             self._p(part), self._p(sc)))
        lat = lattice.view(tdt).view(self.total, self.LD)

        def row(t):
            return lat[t - w0, :self.N].double().cpu().numpy()
        out = {"mode": "diff", "tol": 1e-5 if prec == _lib.F32 else 1e-11,
               "right_state": int(states[b - 1 - w0].item()), "right_probe": row(b - 1),
               "left_state": int(states[a - 1 - w0].item()) if a > w0 else None,
               "left_probe": row(a - 1) if a > w0 else None}
        core_states = self.states_to_host(states[a - w0:b - w0])
        out["result"] = (float(part.item()), core_states)
        return out

    def map_window(self, obs, core, window, band=64, precision=None):
        """posterior (MAP) decoding of obs[window]: the core's states; the probes are the
        decoded states in a band around each core boundary, which both neighbours compute
        (one with an exact forward and a speculative backward pass, the other the reverse)."""
        (a, b), (w0, w1) = core, window
        self.upload_batch([obs[w0:w1]])
        out = self.posteriors(renorm_eps=True, want_post=False, want_map=True, precision=precision)
        st = out["map_states"][0]

        def bandv(t):          # states over [t - band, t + band), clipped identically on both ranks
            lo, hi = max(0, t - band), min(obs.shape[0], t + band)
            v = np.full(2 * band, -1.0)
            seg = st[max(lo, w0) - w0:min(hi, w1) - w0]
            v[max(lo, w0) - (t - band):max(lo, w0) - (t - band) + len(seg)] = seg
            return v
        res = {"mode": "equal", "tol": 0.0, "left_state": None, "right_state": None,
               "right_probe": bandv(b), "left_probe": bandv(a) if a > 0 else None}
        res["result"] = st[a - w0:b - w0]
        return res

    def score_window(self, obs, core, window, precision=None):
        """this rank's increment of the forward log-likelihood: logP(x[w0:b)) - logP(x[w0:a)),
        both from a flat start at w0 (rank 0: w0 = a = 0 and the increment is logP(x[0:b)));
        probes are the forward vectors at a-1 and b-1."""
        prec, tdt = self._prec(precision)
        (a, b), (w0, w1) = core, window
        seqs = [obs[w0:b]] + ([obs[w0:a]] if a > w0 else [])
        self.upload_batch(seqs)
        _, blin, rowmax = self.run_emission(prec, tdt, None, False, True)
        alpha, logprob = self.run_forward(prec, tdt, blin, rowmax, None)
        lp = logprob.cpu().numpy()
        al = alpha.view(self.total, self.LD)

        def row(i):
            v = al[i, :self.N].double().cpu().numpy()
            return v / v.max() if v.max() > 0 else v
        res = {"mode": "ratio", "tol": 4e-6 if prec == _lib.F32 else 1e-12, "left_state": None,
               "right_state": None, "right_probe": row(b - w0 - 1),
               "left_probe": row((b - w0) + (a - w0) - 1) if a > w0 else None}
        res["result"] = float(lp[0] - (lp[1] if a > w0 else 0.0))
        return res

    def estep(self, ratios=None, want_start=True, want_trans=True, want_obs=True,
              precision=None, device_result=False, seq_slots=None, stats_S=None):
        """One E-step over the batch (basehmm.py:507-522 + hmm.py:545-574).
        Returns the packed float64 device tensor
            [sum logprob | nseq | start N | trans N*N | obs K*N*S | per-sequence logprob]
        (ready for ONE all-reduce) or, by default, a dict of host arrays.
        seq_slots = (n_total, indices): where this batch's sequences sit in the
        job-wide per-sequence tail (other ranks fill the other slots)."""
        torch = self.torch
        prec, tdt = self._prec(precision)
        N, K = self.N, self.K
        S = self.stats_S = int(stats_S) if stats_S else self.S    # width of the caller's obsStats
        n_total, slots = seq_slots if seq_slots is not None else (self.nseq, list(range(self.nseq)))
        d_r = ratios if (ratios is None or torch.is_tensor(ratios)) else self.upload_ratios(ratios)
        _, blin, rowmax = self.run_emission(prec, tdt, d_r, False, True)
        self.fold_ratios(prec, d_r, blin, rowmax)          # forward / backward below run without ratios
        base = 2 + N + N * N + K * N * S
        flags = 0
        if want_trans or want_start:
            flags |= _lib.BWD_TRANS
        if want_obs or (d_r is not None and flags):
            flags |= _lib.BWD_POSTERIORS                    # the ratios' diagonal counts come from the posteriors

        def stages():
            alpha, logprob = self.run_forward(prec, tdt, blin, rowmax, None)
            packed = torch.zeros(base + n_total, dtype=torch.float64, device=self.device)
            if flags:
                post, _, _ = self.run_backward(prec, tdt, flags, blin, alpha, None,
                                               start_trans=packed[2:2 + N + N * N])
                if d_r is not None and (flags & _lib.BWD_TRANS):
                    _lib.check(self.lib.tehmm_ratio_diag_counts(self.ctx.handle, prec, self._p(post), self._p(d_r),
                                                                self._p(packed[2:2 + N + N * N]), self._p(self.scratch(prec))))
                if want_obs:
                    self.run_emission_stats(prec, post, d_r, packed[2 + N + N * N:base], S)
            return packed, logprob
        # deferred verification: the stages are queued back to back and checked once
        packed, logprob = self.ctx.optimistic(stages)
        packed[0] = logprob.sum()
        packed[1] = float(self.nseq)
        packed[base:].index_copy_(0, torch.as_tensor(slots, dtype=torch.int64, device=self.device), logprob)
        if device_result:
            return packed
        return self.unpack_stats(packed.cpu().numpy())

    def unpack_stats(self, host):
        N, K, S = self.N, self.K, getattr(self, "stats_S", self.S)
        base = 2 + N + N * N + K * N * S
        return {"logprob": float(host[0]), "nobs": int(round(host[1])),
                "start": host[2:2 + N].copy(), "trans": host[2 + N:2 + N + N * N].reshape(N, N).copy(),
                "obs": host[2 + N + N * N:base].reshape(K, N, S).copy(), "logprobs": host[base:].copy()}


_engines = {}


def get_engine(device=None):
    """Engine of the calling thread's context (contexts are per thread, see _lib.get_context)."""
    ctx = _lib.get_context(device)
    eng = _engines.get(id(ctx))
    if eng is None or eng.ctx is not ctx:
        eng = _engines[id(ctx)] = Engine(ctx)
    return eng
