// Host-buffer decode: the whole call MultitrackHmm.decode makes
// (hmm.py:668-676 Viterbi, basehmm.py:332-359 MAP), natively.
//
//   host symbols --(pinned staging, worker threads)--> HBM
//       -> emission -> Viterbi DP + traceback | forward + backward(MAP)
//   uint8 states --PCIe--> pinned --(worker threads, widened)--> caller's int64[T]
//
// Everything between the two host buffers is owned by the library: a grow-only
// device arena per context, two pinned staging rings and a small persistent
// thread pool.  The Python layer used torch for these steps before: a pageable
// 100 MB observation matrix took 9.2 ms to upload (one thread, one bounce
// buffer) and the int64 widening of 10 M states 4.4 ms; see profiles/.
// Built only on the public C ABI (tehmm_set_batch / tehmm_run_*), so it is a
// caller of the batched path, not a second implementation of it.
#include "common.cuh"
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <unistd.h>
#include <vector>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

void tehmm_set_error(int code, const char *msg);   // api.cu

namespace {

// ---------------------------------------------------------------- thread pool
class Pool {
public:
    explicit Pool(int n) : stop_(false), gen_(0), pending_(0), ntasks_(0)
    {
        for (int i = 0; i < n; ++i) workers_.emplace_back([this] { loop(); });
    }
    ~Pool()
    {
        { std::lock_guard<std::mutex> l(mu_); stop_ = true; ++gen_; }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
    }
    int size() const { return (int)workers_.size() + 1; }
    // run fn(i) for i in [0, n); the calling thread takes part
    void parallel_for(int n, const std::function<void(int)> &fn)
    {
        if (n <= 0) return;
        if (workers_.empty() || n == 1) { for (int i = 0; i < n; ++i) fn(i); return; }
        uint64_t gen;
        {
            std::lock_guard<std::mutex> l(mu_);
            fn_ = &fn; ntasks_ = n; pending_ = n; gen = ++gen_;
            next_.store(gen << 32);               // generation in the high half: stale fetches are rejected
        }
        cv_.notify_all();
        work(gen, n, &fn);
        std::unique_lock<std::mutex> l(mu_);
        done_.wait(l, [this] { return pending_ == 0; });
        fn_ = nullptr;
    }
private:
    // A job is (generation, task count, function), snapshotted under the lock by whoever runs it.
    // The task counter carries the generation in its high 32 bits and is advanced by compare-and-swap
    // ONLY while it still belongs to the caller's generation: a worker left over from generation g that
    // comes back for more after parallel_for g+1 has reset the counter must neither run a task of the new
    // job nor consume one of its indices (a plain fetch_add did the latter: task 0 of the new job was
    // never run and parallel_for waited for ever -- seen once in ~25 bench runs).
    void work(uint64_t gen, int ntasks, const std::function<void(int)> *fn)
    {
        for (;;) {
            uint64_t v = next_.load();
            for (;;) {
                if ((v >> 32) != (gen & 0xffffffffu) || (int)(v & 0xffffffffu) >= ntasks) return;
                if (next_.compare_exchange_weak(v, v + 1)) break;
            }
            (*fn)((int)(v & 0xffffffffu));
            std::lock_guard<std::mutex> l(mu_);
            if (--pending_ == 0) done_.notify_all();
        }
    }
    void loop()
    {
        uint64_t seen = 0;
        for (;;) {
            int ntasks;
            const std::function<void(int)> *fn;
            {
                std::unique_lock<std::mutex> l(mu_);
                cv_.wait(l, [&] { return gen_ != seen; });
                seen = gen_;
                if (stop_) return;
                ntasks = ntasks_; fn = fn_;
                if (fn == nullptr) continue;      // the job finished before this worker woke up
            }
            work(seen, ntasks, fn);
        }
    }
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_, done_;
    bool stop_;
    uint64_t gen_;
    int pending_, ntasks_;
    std::atomic<uint64_t> next_;
    const std::function<void(int)> *fn_ = nullptr;
};

// uint8 -> int64 with streaming stores (the output is 8x the input and is not read back here)
void widen_u8_i64(const uint8_t *in, int64_t *out, int64_t n)
{
    int64_t i = 0;
#if defined(__SSE2__)
    while (i < n && ((uintptr_t)(out + i) & 15)) { out[i] = in[i]; ++i; }
    const __m128i z = _mm_setzero_si128();
    for (; i + 16 <= n; i += 16) {
        const __m128i v = _mm_loadu_si128((const __m128i *)(in + i));
        const __m128i w0 = _mm_unpacklo_epi8(v, z), w1 = _mm_unpackhi_epi8(v, z);
        const __m128i d0 = _mm_unpacklo_epi16(w0, z), d1 = _mm_unpackhi_epi16(w0, z);
        const __m128i d2 = _mm_unpacklo_epi16(w1, z), d3 = _mm_unpackhi_epi16(w1, z);
        __m128i *o = (__m128i *)(out + i);
        _mm_stream_si128(o + 0, _mm_unpacklo_epi32(d0, z));
        _mm_stream_si128(o + 1, _mm_unpackhi_epi32(d0, z));
        _mm_stream_si128(o + 2, _mm_unpacklo_epi32(d1, z));
        _mm_stream_si128(o + 3, _mm_unpackhi_epi32(d1, z));
        _mm_stream_si128(o + 4, _mm_unpacklo_epi32(d2, z));
        _mm_stream_si128(o + 5, _mm_unpackhi_epi32(d2, z));
        _mm_stream_si128(o + 6, _mm_unpacklo_epi32(d3, z));
        _mm_stream_si128(o + 7, _mm_unpackhi_epi32(d3, z));
    }
    _mm_sfence();
#endif
    for (; i < n; ++i) out[i] = in[i];
}

constexpr size_t SLICE = (size_t)8 << 20;   // staging slice
constexpr int NRING = 4;

struct HostPipe {
    int device = 0;
    void *arena = nullptr;
    size_t arena_bytes = 0;
    unsigned char *ring[NRING] = {};
    cudaEvent_t ring_ev[NRING] = {};
    bool ring_used[NRING] = {};
    cudaStream_t copy_stream = nullptr;     // host -> device copies, ahead of the compute stream
    cudaEvent_t both_ev = nullptr;          // TEHMM_DECODE_BOTH: the backward pass is done (the MAP path may leave)
    std::vector<cudaEvent_t> slice_ev;      // one per slice of a call, reused
    unsigned char *pin_out = nullptr;       // states + the per-sequence scalars
    size_t pin_out_bytes = 0;
    Pool *pool = nullptr;
    int64_t h2d_bytes = 0, d2h_bytes = 0;
    int64_t redone = 0;                     // calls whose deferred verification failed and ran twice
    int defer_skip = 0, defer_penalty = 0;  // back-off after a refusal
    double phase_ms[4] = {-1, -1, -1, -1};  // last traced call: set_batch, h2d+emission, trellis, d2h+widen (TEHMM_HOST_TRACE)

    ~HostPipe()
    {
        cudaSetDevice(device);
        if (arena) cudaFree(arena);
        for (int i = 0; i < NRING; ++i) {
            if (ring[i]) cudaFreeHost(ring[i]);
            if (ring_ev[i]) cudaEventDestroy(ring_ev[i]);
        }
        if (pin_out) cudaFreeHost(pin_out);
        for (cudaEvent_t e : slice_ev) cudaEventDestroy(e);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (both_ev) cudaEventDestroy(both_ev);
        delete pool;
    }
};

std::mutex g_mu;
std::map<tehmm_ctx *, HostPipe *> g_pipes;

int host_threads()
{
    const char *e = getenv("TEHMM_HOST_THREADS");
    int n = e ? atoi(e) : 0;
    if (n <= 0) {
        n = (int)std::thread::hardware_concurrency();
        if (n > 16) n = 16;
    }
    return n < 1 ? 1 : n;
}

HostPipe *get_pipe(tehmm_ctx *c, int device)
{
    std::lock_guard<std::mutex> l(g_mu);
    auto it = g_pipes.find(c);
    if (it != g_pipes.end()) return it->second;
    HostPipe *p = new HostPipe();
    p->device = device;
    p->pool = new Pool(host_threads() - 1);
    g_pipes[c] = p;
    return p;
}

int herr(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    tehmm_set_error(code, buf);
    return code;
}
#define HCU(x)                                                                                  \
    do {                                                                                        \
        cudaError_t e__ = (x);                                                                  \
        if (e__ != cudaSuccess)                                                                 \
            return herr(TEHMM_ECUDA, "%s failed: %s (%s:%d)", #x, cudaGetErrorString(e__),      \
                        __FILE__, __LINE__);                                                    \
    } while (0)
#define HOK(x) do { int r__ = (x); if (r__ != TEHMM_OK) return r__; } while (0)

size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }

// TEHMM_HOST_TRACE=1: wall-clock phases of tehmm_decode_host on stderr (adds a stream sync per phase)
struct Trace {
    bool on, print;
    cudaStream_t st;
    std::chrono::steady_clock::time_point t0;
    std::string line;
    double *slot;       // HostPipe::phase_ms
    int n = 0;
    Trace(cudaStream_t s, double *ph) : on(false), print(false), st(s), t0(std::chrono::steady_clock::now()), slot(ph)
    {
        const char *e = getenv("TEHMM_HOST_TRACE");
        on = e != nullptr && e[0] != '0';
        print = on && e[0] == '1';            // "1": also a line on stderr; "2": record only
        if (on) for (int i = 0; i < 4; ++i) slot[i] = -1.0;
    }
    void mark(const char *name, bool sync)
    {
        if (!on) return;
        if (sync) cudaStreamSynchronize(st);
        const auto t1 = std::chrono::steady_clock::now();
        const double ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
        if (n < 4) slot[n] = ms;              // a second attempt (failed deferred check) overwrites nothing: n runs on
        n += 1;
        char buf[64];
        snprintf(buf, sizeof buf, " %s %.2f", name, ms);
        line += buf;
        t0 = t1;
    }
    ~Trace() { if (print) fprintf(stderr, "[tehmm_decode_host ms]%s\n", line.c_str()); }
};

}   // namespace

// called by tehmm_ctx_destroy
void tehmm_hostpipe_release(tehmm_ctx *c)
{
    HostPipe *p = nullptr;
    {
        std::lock_guard<std::mutex> l(g_mu);
        auto it = g_pipes.find(c);
        if (it == g_pipes.end()) return;
        p = it->second;
        g_pipes.erase(it);
    }
    delete p;
}

extern "C" {

// algorithm TEHMM_DECODE_BOTH: h_states = the Viterbi path, h_logprob = its log-probability, h_states_map = the
// MAP path, h_score = its score, h_fwd_logprob = the forward log-likelihood.
// h_ratio_ptrs (may be NULL): nseq host arrays of segment ratios, NULL for a sequence without them.  Only the
// Viterbi DP, its traceback and re-score see them (hmm.py:674); the emission and the MAP path do not
// (basehmm.py:261-264, 327).  On the device a sequence without ratios gets -1.0, which the Viterbi kernels
// read as "no ratio terms" (csrc/viterbi.cu).
static int decode_host_impl(tehmm_ctx *c, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes, int64_t nseq,
                            const int64_t *h_offsets, const double *const *h_ratio_ptrs, int algorithm, int prec,
                            int64_t *h_states, double *h_logprob, double *h_score, int64_t *h_states_map,
                            double *h_fwd_logprob)
{
    if (!c || !h_obs_ptrs || !h_offsets || !h_states || !h_logprob) return herr(TEHMM_EINVAL, "NULL argument");
    if (nptr != 1 && nptr != nseq) return herr(TEHMM_EINVAL, "nptr must be 1 (one contiguous matrix) or nseq (one matrix per sequence)");
    for (int64_t i = 0; i < nptr; ++i)
        if (!h_obs_ptrs[i] && (nptr == 1 || h_offsets[i + 1] > h_offsets[i])) return herr(TEHMM_EINVAL, "h_obs_ptrs[%lld] is NULL", (long long)i);
    if (algorithm != TEHMM_DECODE_VITERBI && algorithm != TEHMM_DECODE_MAP && algorithm != TEHMM_DECODE_BOTH) return herr(TEHMM_EINVAL, "bad algorithm");
    if (algorithm != TEHMM_DECODE_VITERBI && !h_score) return herr(TEHMM_EINVAL, "h_score is required for MAP");
    if (algorithm == TEHMM_DECODE_BOTH && (!h_states_map || !h_fwd_logprob)) return herr(TEHMM_EINVAL, "BOTH needs h_states_map and h_fwd_logprob");
    const bool both = algorithm == TEHMM_DECODE_BOTH;
    if (prec != TEHMM_F32 && prec != TEHMM_F64) return herr(TEHMM_EINVAL, "bad prec");
    if (nseq <= 0) return herr(TEHMM_EINVAL, "nseq must be positive");
    int N = 0, K = 0, S = 0;
    HOK(tehmm_model_dims(c, &N, &K, &S));
    const int device = tehmm_ctx_device(c);
    HCU(cudaSetDevice(device));
    const cudaStream_t st = (cudaStream_t)(uintptr_t)tehmm_ctx_stream(c);
    HostPipe *p = get_pipe(c, device);
    Trace tr(st, p->phase_ms);
    const int64_t total = h_offsets[nseq];
    if (total <= 0) return herr(TEHMM_EINVAL, "empty batch");
    // segment ratios are staged only when some sequence has them and a Viterbi path is wanted
    bool use_ratios = false;
    if (h_ratio_ptrs && algorithm != TEHMM_DECODE_MAP)
        for (int64_t i = 0; i < nseq && !use_ratios; ++i) use_ratios = h_ratio_ptrs[i] && h_offsets[i + 1] > h_offsets[i];
    const int LD = tehmm_lattice_stride(c);
    const size_t ts = prec == TEHMM_F32 ? 4 : 8;
    const size_t obs_bytes_total = (size_t)total * K * obs_bytes;
    const size_t lat = (size_t)total * LD * ts;

    // ---- arena layout: obs | states | logprob, score | rowmax | lattice A | lattice B | [int64 states] | [ratios] | scratch
    size_t o = 0;
    const size_t o_obs = o; o = up256(o + obs_bytes_total);
    const size_t o_states = o; o = up256(o + (size_t)total);
    const size_t o_states2 = o; if (both) o = up256(o + (size_t)total);
    const size_t o_lp = o; o = up256(o + (size_t)nseq * 32);        // [first logprob | score | second logprob] x nseq
    const size_t o_rowmax = o; o = up256(o + (size_t)total * 8);
    const size_t o_la = o; o = up256(o + lat);
    const size_t o_lb = o; o = up256(o + lat);
    const size_t o_lc = o; if (both) o = up256(o + lat);          // BOTH: A = log emission, C = linear emission, B = alpha, then delta
    // Where the widening to int64 happens.  Host (default): one byte per step over PCIe, the pool's threads
    // widen behind the copy.  Device (TEHMM_WIDEN=gpu, and only when the caller's result array is page-locked:
    // the Python layer registers its result pool under TEHMM_PIN_RESULTS=1): a kernel widens and the DMA engine
    // writes the int64 path straight into the result.  Measured, not the default: 9.6 vs 8.7 ms per
    // Viterbi + MAP pair on one GPU and 22.4 vs 18.2 ms with eight ranks on one host
    // (profiles/r02_notes_e2e.md) -- eight times the bytes over PCIe and into host memory cost more than the
    // host threads they save; the 1 -> 8 GPU end-to-end curve is bound by the host's memory system either way.
    bool gpu_widen = false;
    {
        cudaPointerAttributes attr;
        const bool pinned_out = cudaPointerGetAttributes(&attr, h_states) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
        const char *w = getenv("TEHMM_WIDEN");
        if (pinned_out) gpu_widen = w != nullptr && !strcmp(w, "gpu");
    }
    const size_t o_s64 = o; if (gpu_widen) o = up256(o + (size_t)total * 8);
    const size_t o_rat = o; if (use_ratios) o = up256(o + (size_t)total * 8);
    const size_t o_scratch = o;
    // the scratch size depends on the partition: describe the batch first, with the obs pointer
    // the arena will have (the arena may have to grow before anything is enqueued)
    auto ensure = [&](size_t need) -> int {
        if (need <= p->arena_bytes) return TEHMM_OK;
        HCU(cudaStreamSynchronize(st));
        if (p->arena) { cudaFree(p->arena); p->arena = nullptr; p->arena_bytes = 0; }
        const size_t want = need + need / 8;
        HCU(cudaMalloc(&p->arena, want));
        p->arena_bytes = want;
        return TEHMM_OK;
    };
    HOK(ensure(o_scratch + ((size_t)96 << 20) + (size_t)total * 8));
    HOK(tehmm_set_batch(c, (char *)p->arena + o_obs, obs_bytes, nseq, h_offsets));
    size_t scratch = (size_t)tehmm_scratch_bytes(c, prec);
    if (o_scratch + scratch > p->arena_bytes) {
        HOK(ensure(o_scratch + scratch));
        HOK(tehmm_set_batch(c, (char *)p->arena + o_obs, obs_bytes, nseq, h_offsets));
        scratch = (size_t)tehmm_scratch_bytes(c, prec);
    }
    char *A = (char *)p->arena;
    tr.mark("set_batch", false);

    // ---- host -> device
    // the batch as a list of host segments (one, or one per sequence -- no host-side concatenation)
    struct Seg { const unsigned char *src; size_t off, n; };
    std::vector<Seg> segs;
    if (nptr == 1) segs.push_back(Seg{(const unsigned char *)h_obs_ptrs[0], 0, obs_bytes_total});
    else
        for (int64_t i = 0; i < nseq; ++i) {
            const size_t off = (size_t)h_offsets[i] * K * obs_bytes, n = (size_t)(h_offsets[i + 1] - h_offsets[i]) * K * obs_bytes;
            if (n) segs.push_back(Seg{(const unsigned char *)h_obs_ptrs[i], off, n});
        }
    bool pinned = nptr == 1;
    if (pinned) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, h_obs_ptrs[0]) == cudaSuccess) pinned = attr.type == cudaMemoryTypeHost;
        else { cudaGetLastError(); pinned = false; }
    }
    // The copy runs on its own stream in slices of whole rows; the emission kernel of a slice is
    // enqueued on the compute stream behind that slice's event, so it overlaps the transfer of the
    // next one (the emission is the only stage that can start before the whole batch has arrived).
    if (!p->copy_stream) HCU(cudaStreamCreateWithFlags(&p->copy_stream, cudaStreamNonBlocking));
    if (!p->both_ev) HCU(cudaEventCreateWithFlags(&p->both_ev, cudaEventDisableTiming));
    double *d_lp = (double *)(A + o_lp), *d_sc = d_lp + nseq, *d_lp2 = d_lp + 2 * nseq;
    uint8_t *d_states = (uint8_t *)(A + o_states), *d_states2 = (uint8_t *)(A + o_states2);
    const bool viterbi = algorithm == TEHMM_DECODE_VITERBI;
    void *em_log = (viterbi || both) ? (void *)(A + o_la) : nullptr;
    void *em_lin = both ? (void *)(A + o_lc) : (viterbi ? nullptr : (void *)(A + o_la));
    const bool piecewise = tehmm_emission_rows_supported(c, prec) == 1;
    const size_t row_bytes = (size_t)K * obs_bytes;
    int64_t slice_rows = (int64_t)(SLICE / row_bytes) & ~(int64_t)31;
    if (slice_rows < 32) return herr(TEHMM_ELIMIT, "a row of %zu bytes does not fit the staging slices", row_bytes);
    const int nth = p->pool->size();
    size_t si = 0;                                       // first segment that reaches into the slice
    int64_t slot = 0;
    for (int64_t r0 = 0; r0 < total; r0 += slice_rows, ++slot) {
        const int64_t r1 = std::min(total, r0 + slice_rows);
        const size_t off = (size_t)r0 * row_bytes, n = (size_t)(r1 - r0) * row_bytes;
        if (pinned) {
            HCU(cudaMemcpyAsync(A + o_obs + off, (const unsigned char *)h_obs_ptrs[0] + off, n, cudaMemcpyHostToDevice, p->copy_stream));
        } else {
            // pageable: worker threads fill a pinned slice while the previous one is on the wire
            const int r = (int)(slot % NRING);
            if (!p->ring[r]) {
                HCU(cudaMallocHost((void **)&p->ring[r], SLICE));
                HCU(cudaEventCreateWithFlags(&p->ring_ev[r], cudaEventDisableTiming));
            }
            if (p->ring_used[r]) HCU(cudaEventSynchronize(p->ring_ev[r]));
            while (si + 1 < segs.size() && segs[si].off + segs[si].n <= off) ++si;
            unsigned char *dst = p->ring[r];
            const size_t per = ((n + nth - 1) / nth + 63) & ~(size_t)63;
            const Seg *sg = segs.data();
            const size_t nsg = segs.size(), si0 = si;
            p->pool->parallel_for(nth, [&](int i) {
                size_t a = off + (size_t)i * per;                       // byte range [a, e) of the batch
                const size_t e = std::min(off + n, a + per);
                size_t k = si0;
                while (a < e) {
                    while (k + 1 < nsg && sg[k].off + sg[k].n <= a) ++k;
                    const size_t m = std::min(e, sg[k].off + sg[k].n) - a;
                    memcpy(dst + (a - off), sg[k].src + (a - sg[k].off), m);
                    a += m;
                }
            });
            HCU(cudaMemcpyAsync(A + o_obs + off, dst, n, cudaMemcpyHostToDevice, p->copy_stream));
            HCU(cudaEventRecord(p->ring_ev[r], p->copy_stream));
            p->ring_used[r] = true;
        }
        if ((size_t)slot >= p->slice_ev.size()) {
            cudaEvent_t ev;
            HCU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            p->slice_ev.push_back(ev);
        }
        HCU(cudaEventRecord(p->slice_ev[slot], p->copy_stream));
        HCU(cudaStreamWaitEvent(st, p->slice_ev[slot], 0));
        if (piecewise) HOK(tehmm_run_emission_rows(c, prec, nullptr, em_log, em_lin, (double *)(A + o_rowmax), r0, r1, UINT64_MAX));
    }
    // The segment ratios follow the observations through the same ring and copy stream (the Viterbi DP is the
    // first stage that needs them): the worker threads gather each slice from the per-sequence arrays, fill -1.0
    // for a sequence without ratios, and check every value on the way.
    const double *d_rat = use_ratios ? (const double *)(A + o_rat) : nullptr;
    if (use_ratios) {
        const int64_t rat_rows = (int64_t)(SLICE / sizeof(double));
        for (int64_t r0 = 0; r0 < total; r0 += rat_rows, ++slot) {
            const int64_t r1 = std::min(total, r0 + rat_rows);
            const int r = (int)(slot % NRING);
            if (!p->ring[r]) {
                HCU(cudaMallocHost((void **)&p->ring[r], SLICE));
                HCU(cudaEventCreateWithFlags(&p->ring_ev[r], cudaEventDisableTiming));
            }
            if (p->ring_used[r]) HCU(cudaEventSynchronize(p->ring_ev[r]));
            double *dst = (double *)p->ring[r];
            const int64_t per = ((r1 - r0 + nth - 1) / nth + 7) & ~(int64_t)7;
            std::atomic<int64_t> bad_row(INT64_MAX);
            p->pool->parallel_for(nth, [&](int t) {
                int64_t a = r0 + (int64_t)t * per;
                const int64_t e = std::min(r1, a + per);
                if (a >= e) return;
                int64_t i = std::upper_bound(h_offsets, h_offsets + nseq + 1, a) - h_offsets - 1;
                while (a < e) {
                    while (h_offsets[i + 1] <= a) ++i;                 // (empty sequences)
                    const int64_t n = std::min(e, h_offsets[i + 1]) - a;
                    double *d = dst + (a - r0);
                    const double *src = h_ratio_ptrs[i];
                    if (!src) {
                        std::fill(d, d + n, -1.0);
                    } else {
                        src += a - h_offsets[i];
                        bool ok = true;
                        for (int64_t k = 0; k < n; ++k) {
                            const double v = src[k];
                            ok &= v > 0.0 && v != INFINITY;            // NaN fails the first test
                            d[k] = v;
                        }
                        if (!ok) {
                            int64_t k = 0;
                            while (src[k] > 0.0 && src[k] != INFINITY) ++k;
                            int64_t cur = bad_row.load();
                            while (a + k < cur && !bad_row.compare_exchange_weak(cur, a + k)) {}
                        }
                    }
                    a += n;
                }
            });
            if (bad_row.load() != INT64_MAX) {
                const int64_t row = bad_row.load();
                const int64_t i = std::upper_bound(h_offsets, h_offsets + nseq + 1, row) - h_offsets - 1;
                return herr(TEHMM_EINVAL, "segment ratio %g of sequence %lld, step %lld: ratios must be finite and > 0",
                            h_ratio_ptrs[i][row - h_offsets[i]], (long long)i, (long long)(row - h_offsets[i]));
            }
            HCU(cudaMemcpyAsync(A + o_rat + (size_t)r0 * 8, dst, (size_t)(r1 - r0) * 8, cudaMemcpyHostToDevice, p->copy_stream));
            HCU(cudaEventRecord(p->ring_ev[r], p->copy_stream));
            p->ring_used[r] = true;
        }
        // one event behind the last ratio slice (the ratio slices themselves record only their ring events)
        while (p->slice_ev.size() <= (size_t)slot) {
            cudaEvent_t ev;
            HCU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            p->slice_ev.push_back(ev);
        }
        HCU(cudaEventRecord(p->slice_ev[slot], p->copy_stream));
        HCU(cudaStreamWaitEvent(st, p->slice_ev[slot], 0));
    }
    p->h2d_bytes = (int64_t)obs_bytes_total + (use_ratios ? total * 8 : 0);
    tr.mark("h2d+emission", true);

    // Two attempts at most.  The first runs the stages with deferred verification (option "defer":
    // no stall of the stream after each stage to read the repair count); the counts are looked at
    // once everything has arrived.  If a speculated chunk boundary failed -- rare -- the trellis and
    // the download run again with the synchronous verify / repair loop.
    struct DeferGuard { tehmm_ctx *c; ~DeferGuard() { tehmm_ctx_set_option(c, "defer", 0); } } defer_guard{c};
    double *pin_lp = nullptr;
    int rc = TEHMM_OK;
    // (after a refusal the next calls go straight to the synchronous loop: a refused attempt costs the
    //  trellis twice, and a model / batch that needed repairs tends to need them again)
    int attempt = 0;
    if (p->defer_skip > 0) { p->defer_skip -= 1; attempt = 1; }
    for (; attempt < 2; ++attempt) {
        HOK(tehmm_ctx_set_option(c, "defer", attempt == 0 ? 1 : 0));
        // ---- the trellis
        if (!piecewise) HOK(tehmm_run_emission(c, prec, nullptr, em_log, em_lin, (double *)(A + o_rowmax)));
        if (both) {
            // forward + backward(MAP) first: their states travel and are widened while the Viterbi kernels run
            HOK(tehmm_run_forward(c, prec, A + o_lc, (double *)(A + o_rowmax), nullptr, A + o_lb, d_lp2, A + o_scratch));
            HOK(tehmm_run_backward(c, prec, TEHMM_BWD_MAP | TEHMM_BWD_RENORM_EPS, A + o_lc, A + o_lb, nullptr, nullptr,
                                   d_states2, d_sc, nullptr, A + o_scratch));
        } else if (viterbi) {
            HOK(tehmm_run_viterbi(c, prec, A + o_la, (const double *)(A + o_rowmax), nullptr, d_rat, A + o_lb, d_states, nullptr, d_lp, A + o_scratch));
        } else {
            HOK(tehmm_run_forward(c, prec, A + o_la, (double *)(A + o_rowmax), nullptr, A + o_lb, d_lp, A + o_scratch));
            HOK(tehmm_run_backward(c, prec, TEHMM_BWD_MAP | TEHMM_BWD_RENORM_EPS, A + o_la, A + o_lb, nullptr, nullptr,
                                   d_states, d_sc, nullptr, A + o_scratch));
        }

        tr.mark("trellis", true);
        // ---- device -> host: one byte per step over PCIe, widened by the host's cores
        const size_t out_bytes = (both ? 2 : 1) * up256((size_t)total) + (size_t)nseq * 32;
        if (p->pin_out_bytes < out_bytes) {
            HCU(cudaStreamSynchronize(st));
            if (p->pin_out) cudaFreeHost(p->pin_out);
            p->pin_out = nullptr; p->pin_out_bytes = 0;
            HCU(cudaMallocHost((void **)&p->pin_out, out_bytes + out_bytes / 8));
            p->pin_out_bytes = out_bytes + out_bytes / 8;
        }
        pin_lp = (double *)(p->pin_out + (both ? 2 : 1) * up256((size_t)total));
        if (!both) HCU(cudaMemcpyAsync(pin_lp, d_lp, (size_t)nseq * 32, cudaMemcpyDeviceToHost, st));
        if (gpu_widen && !both) {
            int64_t *d_s64 = (int64_t *)(A + o_s64);
            HOK(tehmm_widen_states(c, d_states, d_s64, total));
            HCU(cudaMemcpyAsync(h_states, d_s64, (size_t)total * 8, cudaMemcpyDeviceToHost, st));
            HCU(cudaStreamSynchronize(st));
            tr.mark("d2h(int64)", false);
            rc = TEHMM_OK;
            if (attempt == 0) {
                int64_t unverified = 0;
                HOK(tehmm_ctx_set_option(c, "defer", 0));
                HOK(tehmm_ctx_check(c, &unverified));
                if (unverified == 0) { p->defer_penalty /= 2; break; }
                p->redone += 1;
                p->defer_penalty = std::min(256, std::max(4, 2 * p->defer_penalty));
                p->defer_skip = p->defer_penalty;
            }
            continue;
        }
        // slices, so that the widening of slice i overlaps the transfer of slice i+1
        const int nsl = (int)std::min<int64_t>(8, (total + (1 << 20) - 1) >> 20);
        const int64_t per_sl = ((total + nsl - 1) / nsl + 63) & ~(int64_t)63;
        while ((int)p->slice_ev.size() < 2 * nsl) {        // the upload's events are long complete: reuse them
            cudaEvent_t ev;
            HCU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            p->slice_ev.push_back(ev);
        }
        const std::vector<cudaEvent_t> &evs = p->slice_ev;
        // queue the copies of one path (`which` picks the half of the pinned buffer and of the events)
        auto queue_copies = [&](const uint8_t *d_src, int which, cudaStream_t cs) -> int {
            for (int i = 0; i < nsl; ++i) {
                const int64_t a = (int64_t)i * per_sl, n = std::min(per_sl, total - a);
                if (n > 0) HCU(cudaMemcpyAsync(p->pin_out + which * up256((size_t)total) + a, d_src + a, (size_t)n, cudaMemcpyDeviceToHost, cs));
                HCU(cudaEventRecord(evs[which * nsl + i], cs));
            }
            return TEHMM_OK;
        };
        auto widen_slices = [&](int64_t *h_dst, int which) {
            for (int i = 0; i < nsl; ++i) {
                const int64_t a = (int64_t)i * per_sl, n = std::min(per_sl, total - a);
                cudaError_t e = cudaEventSynchronize(evs[which * nsl + i]);
                if (e != cudaSuccess) { rc = herr(TEHMM_ECUDA, "decode failed: %s", cudaGetErrorString(e)); continue; }
                if (n <= 0 || rc != TEHMM_OK) continue;
                const int64_t per = ((n + nth - 1) / nth + 63) & ~(int64_t)63;
                const uint8_t *src = p->pin_out + which * up256((size_t)total) + a;
                int64_t *dst = h_dst + a;
                p->pool->parallel_for(nth, [&](int t) {
                    const int64_t b0 = (int64_t)t * per;
                    if (b0 < n) widen_u8_i64(src + b0, dst + b0, std::min(per, n - b0));
                });
            }
        };
        rc = TEHMM_OK;
        if (both) {
            // the MAP path leaves on the copy stream behind the backward pass; the Viterbi stage is queued on
            // the compute stream meanwhile, and the host widens the MAP path while those kernels run
            HCU(cudaEventRecord(p->both_ev, st));
            HCU(cudaStreamWaitEvent(p->copy_stream, p->both_ev, 0));
            HOK(queue_copies(d_states2, 1, p->copy_stream));
            HOK(tehmm_run_viterbi(c, prec, A + o_la, (const double *)(A + o_rowmax), nullptr, d_rat, A + o_lb, d_states, nullptr, d_lp, A + o_scratch));
            HCU(cudaMemcpyAsync(pin_lp, d_lp, (size_t)nseq * 32, cudaMemcpyDeviceToHost, st));
            HOK(queue_copies(d_states, 0, st));
            widen_slices(h_states_map, 1);
            widen_slices(h_states, 0);
        } else {
            HOK(queue_copies(d_states, 0, st));
            widen_slices(h_states, 0);
        }
        if (rc != TEHMM_OK) return rc;
        HCU(cudaStreamSynchronize(st));
        tr.mark("d2h+widen", false);
        if (attempt == 0) {
            int64_t unverified = 0;
            HOK(tehmm_ctx_set_option(c, "defer", 0));
            HOK(tehmm_ctx_check(c, &unverified));
            if (unverified == 0) { p->defer_penalty /= 2; break; }
            p->redone += 1;
            p->defer_penalty = std::min(256, std::max(4, 2 * p->defer_penalty));
            p->defer_skip = p->defer_penalty;
        }
    }
    memcpy(h_logprob, pin_lp, (size_t)nseq * 8);
    if (h_score) memcpy(h_score, pin_lp + nseq, (size_t)nseq * 8);
    if (both) memcpy(h_fwd_logprob, pin_lp + 2 * nseq, (size_t)nseq * 8);
    p->d2h_bytes = (gpu_widen && !both ? (int64_t)total * 8 : (both ? 2 : 1) * (int64_t)total) + nseq * (both ? 32 : 16);
    return TEHMM_OK;
}

int tehmm_decode_host(tehmm_ctx *c, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes, int64_t nseq,
                      const int64_t *h_offsets, int algorithm, int prec, int64_t *h_states,
                      double *h_logprob, double *h_score)
{
    if (algorithm == TEHMM_DECODE_BOTH) return herr(TEHMM_EINVAL, "TEHMM_DECODE_BOTH goes through tehmm_decode_host_both");
    return decode_host_impl(c, h_obs_ptrs, nptr, obs_bytes, nseq, h_offsets, nullptr, algorithm, prec, h_states, h_logprob, h_score, nullptr, nullptr);
}

int tehmm_decode_host_ratios(tehmm_ctx *c, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes, int64_t nseq,
                             const int64_t *h_offsets, const double *const *h_ratio_ptrs, int algorithm, int prec,
                             int64_t *h_states, double *h_logprob, double *h_score)
{
    if (algorithm == TEHMM_DECODE_BOTH) return herr(TEHMM_EINVAL, "TEHMM_DECODE_BOTH goes through tehmm_decode_host_both_ratios");
    return decode_host_impl(c, h_obs_ptrs, nptr, obs_bytes, nseq, h_offsets, h_ratio_ptrs, algorithm, prec, h_states, h_logprob, h_score, nullptr, nullptr);
}

int tehmm_decode_host_both(tehmm_ctx *c, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes, int64_t nseq,
                           const int64_t *h_offsets, int prec, int64_t *h_viterbi_states, double *h_viterbi_logprob,
                           int64_t *h_map_states, double *h_map_score, double *h_forward_logprob)
{
    return decode_host_impl(c, h_obs_ptrs, nptr, obs_bytes, nseq, h_offsets, nullptr, TEHMM_DECODE_BOTH, prec, h_viterbi_states,
                            h_viterbi_logprob, h_map_score, h_map_states, h_forward_logprob);
}

int tehmm_decode_host_both_ratios(tehmm_ctx *c, const void *const *h_obs_ptrs, int64_t nptr, int obs_bytes, int64_t nseq,
                                  const int64_t *h_offsets, const double *const *h_ratio_ptrs, int prec,
                                  int64_t *h_viterbi_states, double *h_viterbi_logprob, int64_t *h_map_states,
                                  double *h_map_score, double *h_forward_logprob)
{
    return decode_host_impl(c, h_obs_ptrs, nptr, obs_bytes, nseq, h_offsets, h_ratio_ptrs, TEHMM_DECODE_BOTH, prec,
                            h_viterbi_states, h_viterbi_logprob, h_map_score, h_map_states, h_forward_logprob);
}


// Self-test of the host thread pool (no GPU): `rounds` back-to-back parallel_for calls of `threads` tiny tasks;
// returns the number of rounds in which some index did not run exactly once (0 = pass).  A round that loses
// a task would never return; the caller runs this under a timeout.
int64_t tehmm_host_pool_selftest(int threads, int64_t rounds)
{
    if (threads < 1 || rounds < 0) return -1;
    Pool pool(threads - 1);
    std::vector<std::atomic<int>> hits((size_t)threads);
    int64_t bad = 0;
    for (int64_t r = 0; r < rounds; ++r) {
        for (auto &h : hits) h.store(0);
        pool.parallel_for(threads, [&](int i) { hits[(size_t)i].fetch_add(1); });
        for (auto &h : hits) if (h.load() != 1) { ++bad; break; }
    }
    return bad;
}

double tehmm_decode_host_phase_ms(tehmm_ctx *c, int which)
{
    std::lock_guard<std::mutex> l(g_mu);
    auto it = g_pipes.find(c);
    if (it == g_pipes.end() || which < 0 || which > 3) return -1.0;
    return it->second->phase_ms[which];
}

int64_t tehmm_decode_host_bytes(tehmm_ctx *c, int which)
{
    std::lock_guard<std::mutex> l(g_mu);
    auto it = g_pipes.find(c);
    if (it == g_pipes.end()) return 0;
    return which == 0 ? it->second->h2d_bytes : it->second->d2h_bytes;
}


// ---------------------------------------------------------------------------------------
// Decode output path (SURVEY.md section 8f, rank 1): the per-observation BED writer of
// teHmmEval.py:238-262 (statesToBed, bedFile part).  Once the trellis takes milliseconds the
// reference's Python loop -- one "%s\t%d\t%d\t%s\n" per observation, 12 M lines for a genome --
// is what a user waits for.  Same lines, same order (contiguous equal states are NOT merged,
// teHmmEval.py:241-243): interval starts are a prefix sum of the segment lengths (plus the mask's
// running offset), blocks of lines are formatted by a few threads and written in order.
static int fmt_i64(char *p, int64_t v)
{
    static const char D2[] = "0001020304050607080910111213141516171819202122232425262728293031323334353637383940414243444546474849"
                             "5051525354555657585960616263646566676869707172737475767778798081828384858687888990919293949596979899";
    char tmp[24];
    int n = 24;
    uint64_t u = v < 0 ? (uint64_t)(-(v + 1)) + 1u : (uint64_t)v;
    while (u >= 100) { const unsigned r = (unsigned)(u % 100); u /= 100; tmp[--n] = D2[2 * r + 1]; tmp[--n] = D2[2 * r]; }
    if (u >= 10) { tmp[--n] = D2[2 * u + 1]; tmp[--n] = D2[2 * u]; }
    else tmp[--n] = (char)('0' + u);
    int k = 0;
    if (v < 0) p[k++] = '-';
    memcpy(p + k, tmp + n, (size_t)(24 - n));
    return k + 24 - n;
}

// str() of a float64 as Python / NumPy print it ("%s" % np.float64, teHmmEval.py:266-270): the
// shortest decimal that reads back as the same double, positional for 1e-4 <= |x| < 1e16 (always
// with a fractional part: "1.0"), scientific otherwise ("1e-05", "1.5e+16").  At most three
// correctly rounded conversions: 15 significant digits are unique when they round-trip (their
// trailing zeros dropped), else 16, else 17.
static int fmt_pyfloat(char *out, double x)
{
    if (x != x) { memcpy(out, "nan", 3); return 3; }
    int k = 0;
    if (std::signbit(x)) { out[k++] = '-'; x = -x; }
    if (x == INFINITY) { memcpy(out + k, "inf", 3); return k + 3; }
    if (x == 0.0) { memcpy(out + k, "0.0", 3); return k + 3; }
    char tmp[40];
    // (subnormals carry fewer bits: there the 15-digit argument does not hold, search from one digit)
    for (int prec = x < 2.2250738585072014e-308 ? 1 : 15; prec <= 17; ++prec) {
        snprintf(tmp, sizeof tmp, "%.*e", prec - 1, x);
        if (prec == 17 || strtod(tmp, nullptr) == x) break;
    }
    // tmp = d.ddddde[+-]XX
    char dig[24];
    int nd = 0;
    const char *q = tmp;
    for (; *q && *q != 'e'; ++q)
        if (*q >= '0' && *q <= '9') dig[nd++] = *q;
    const int e10 = atoi(q + 1);
    while (nd > 1 && dig[nd - 1] == '0') --nd;
    if (e10 >= 16 || e10 < -4) {
        out[k++] = dig[0];
        if (nd > 1) { out[k++] = '.'; memcpy(out + k, dig + 1, (size_t)(nd - 1)); k += nd - 1; }
        out[k++] = 'e';
        out[k++] = e10 < 0 ? '-' : '+';
        const int a = e10 < 0 ? -e10 : e10;
        if (a >= 100) out[k++] = (char)('0' + a / 100);
        out[k++] = (char)('0' + (a / 10) % 10);
        out[k++] = (char)('0' + a % 10);
        return k;
    }
    if (e10 >= 0) {
        for (int i = 0; i <= e10; ++i) out[k++] = i < nd ? dig[i] : '0';
        out[k++] = '.';
        if (nd > e10 + 1) { memcpy(out + k, dig + e10 + 1, (size_t)(nd - e10 - 1)); k += nd - e10 - 1; }
        else out[k++] = '0';
        return k;
    }
    out[k++] = '0'; out[k++] = '.';
    for (int i = 0; i < -e10 - 1; ++i) out[k++] = '0';
    memcpy(out + k, dig, (size_t)nd);
    return k + nd;
}

// fourth column: the state (index or name), or -- scores != NULL -- a float64 printed as Python does
static int write_bed(int fd, const char *chrom, int64_t start, const int64_t *states, const double *scores,
                     int64_t n, const int64_t *seg_len, const int32_t *mask_off, int64_t mask_n,
                     const char *const *names, int nnames)
{
    if (fd < 0 || !chrom || (!states && !scores && n > 0) || n < 0) return herr(TEHMM_EINVAL, "bad argument");
    if (n == 0) return TEHMM_OK;
    const size_t clen = strlen(chrom);
    std::vector<size_t> nlen((size_t)std::max(nnames, 0));
    size_t maxname = 32;
    for (int i = 0; i < nnames; ++i) {
        if (!names || !names[i]) return herr(TEHMM_EINVAL, "names[%d] is NULL", i);
        nlen[i] = strlen(names[i]);
        maxname = std::max(maxname, nlen[i]);
    }
    const int64_t BLOCK = 1 << 17;
    const int64_t nblocks = (n + BLOCK - 1) / BLOCK;
    // start of every block: prefix sum of the segment lengths (1 per observation without segments)
    std::vector<int64_t> bstart((size_t)nblocks + 1, 0);
    if (seg_len) {
        for (int64_t b = 0; b < nblocks; ++b) {
            int64_t acc = 0;
            const int64_t e = std::min(n, (b + 1) * BLOCK);
            for (int64_t i = b * BLOCK; i < e; ++i) acc += seg_len[i];
            bstart[b + 1] = bstart[b] + acc;
        }
    } else {
        for (int64_t b = 0; b <= nblocks; ++b) bstart[b] = std::min(n, b * BLOCK);
    }
    const size_t line_max = clen + maxname + 2 * 21 + 4;
    int nth = host_threads();
    if ((int64_t)nth > nblocks) nth = (int)nblocks;
    if (nth > 8) nth = 8;
    // rounds of nth blocks: formatted in parallel, written in order
    std::vector<std::vector<char>> buf((size_t)nth);
    std::vector<size_t> used((size_t)nth, 0);
    std::atomic<int> bad_state(0);
    for (int64_t b0 = 0; b0 < nblocks; b0 += nth) {
        const int cnt = (int)std::min<int64_t>(nth, nblocks - b0);
        auto work = [&](int w) {
            const int64_t b = b0 + w, lo = b * BLOCK, hi = std::min(n, lo + BLOCK);
            std::vector<char> &out = buf[w];
            if (out.size() < (size_t)(hi - lo) * line_max) out.resize((size_t)(hi - lo) * line_max);
            char *p = out.data();
            int64_t dist = bstart[b];
            char endtxt[24];                  // without a mask an interval starts where the last one ended:
            int endlen = 0;                   // its text is reused
            for (int64_t i = lo; i < hi; ++i) {
                int64_t cur = start + dist;
                const int64_t len = seg_len ? seg_len[i] : 1;
                dist += len;
                if (mask_off) {
                    const int64_t rel = cur - start;
                    if (rel >= 0 && rel < mask_n) cur += mask_off[rel];
                }
                memcpy(p, chrom, clen); p += clen;
                *p++ = '\t';
                if (endlen && !mask_off) { memcpy(p, endtxt, (size_t)endlen); p += endlen; }
                else p += fmt_i64(p, cur);
                *p++ = '\t';
                endlen = fmt_i64(endtxt, cur + len);
                memcpy(p, endtxt, (size_t)endlen); p += endlen;
                *p++ = '\t';
                if (scores) { p += fmt_pyfloat(p, scores[i]); *p++ = '\n'; continue; }
                const int64_t st = states[i];
                if (nnames > 0) {
                    if (st < 0 || st >= nnames) { bad_state.store(1); p += fmt_i64(p, st); }
                    else { memcpy(p, names[st], nlen[st]); p += nlen[st]; }
                } else p += fmt_i64(p, st);
                *p++ = '\n';
            }
            used[w] = (size_t)(p - out.data());
        };
        std::vector<std::thread> th;
        for (int w = 1; w < cnt; ++w) th.emplace_back(work, w);
        work(0);
        for (auto &t : th) t.join();
        for (int w = 0; w < cnt; ++w) {
            const char *q = buf[w].data();
            size_t left = used[w];
            while (left) {
                const ssize_t k = write(fd, q, left);
                if (k <= 0) return herr(TEHMM_ESTATE, "write failed");
                q += k; left -= (size_t)k;
            }
        }
    }
    if (bad_state.load()) return herr(TEHMM_EINVAL, "a state index has no name");
    return TEHMM_OK;
}

int tehmm_states_to_bed(int fd, const char *chrom, int64_t start, const int64_t *states, int64_t n,
                        const int64_t *seg_len, const int32_t *mask_off, int64_t mask_n,
                        const char *const *names, int nnames)
{
    if (!states && n > 0) return herr(TEHMM_EINVAL, "states is NULL");
    return write_bed(fd, chrom, start, states, nullptr, n, seg_len, mask_off, mask_n, names, nnames);
}

// The posterior / emission score files of the same function (teHmmEval.py:264-270): same intervals,
// fourth column = one float64 per observation, printed as "%s" of a NumPy float64.
int tehmm_scores_to_bed(int fd, const char *chrom, int64_t start, const double *scores, int64_t n,
                        const int64_t *seg_len, const int32_t *mask_off, int64_t mask_n)
{
    if (!scores && n > 0) return herr(TEHMM_EINVAL, "scores is NULL");
    return write_bed(fd, chrom, start, nullptr, scores, n, seg_len, mask_off, mask_n, nullptr, 0);
}

}   // extern "C"
