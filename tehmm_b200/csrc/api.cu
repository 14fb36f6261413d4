// C ABI of libtehmm_b200.so (see include/tehmm_b200.h): context, model and
// batch management, time partitioning, and the speculate / verify / repair
// drivers around the scan kernels.
#include "common.cuh"
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

// ---- launchers defined in the other translation units
void tehmm_launch_strict_emission(cudaStream_t, const void *, int, int64_t, int, const double *, int, int, double *, double, const double *, unsigned long long *);
void tehmm_launch_strict_forward(cudaStream_t, int64_t, int, const double *, const double *, const double *, const double *, double *);
void tehmm_launch_strict_backward(cudaStream_t, int64_t, int, const double *, const double *, const double *, double *);
void tehmm_launch_strict_viterbi(cudaStream_t, int64_t, int, const double *, const double *, const double *, const double *, int16_t *, int64_t *, double *);
void tehmm_launch_strict_lneta(cudaStream_t, int64_t, int, const double *, const double *, const double *, const double *, double, const double *, double *);
void tehmm_launch_strict_accumulate(cudaStream_t, const void *, int, int64_t, int, double *, int, int, const double *, const double *);
void tehmm_launch_strict_counts(cudaStream_t, const void *, int, int, int64_t, int64_t, int, double *, int, int, const double *);
int tehmm_launch_sup_hist(cudaStream_t, const void *, int, int, int, int, int64_t, int64_t, const int64_t *, const int64_t *, const int64_t *, unsigned long long *, double *, int *);
int tehmm_launch_sup_chain(cudaStream_t, const void *, int, int, int, int, const int64_t *, const int64_t *, const int64_t *, const int64_t *, const double *, double *, int *);
size_t tehmm_emission_table_budget(int K);
int tehmm_launch_emission(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const double *, void *, void *, double *, double *, int *, int, cudaError_t *, int64_t, int64_t);
bool tehmm_emission_rows_ok(const TehmmModelDev &, int, const double *);
cudaError_t tehmm_launch_forward(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const void *, const double *, const double *, void *, void *, void *, double *, const int *, int, int);
cudaError_t tehmm_launch_verify(cudaStream_t, const TehmmBatchDev &, int, int, void *, const void *, double, int, int, int *, int *, double *);
cudaError_t tehmm_launch_forward_logprob(cudaStream_t, const TehmmBatchDev &, int, int, const void *, const double *, const double *, double *);
cudaError_t tehmm_launch_backward(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, int, const void *, const void *, const double *, void *, uint8_t *, double *, void *, void *, void *, void *, void *, const int *, int, int);
cudaError_t tehmm_launch_trans_reduce(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const void *, const void *, const void *, double *);
cudaError_t tehmm_launch_map_reduce(cudaStream_t, const TehmmBatchDev &, const double *, double *);
cudaError_t tehmm_launch_viterbi(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const void *, const double *, void *, void *, void *, const int *, int, int, const double *, double *);
bool tehmm_viterbi_dp_scores(const TehmmModelDev &, int, const double *);
cudaError_t tehmm_launch_vit_score_reduce(cudaStream_t, const TehmmBatchDev &, const double *, double *);
cudaError_t tehmm_launch_traceback(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const void *, const double *, uint8_t *, int64_t *, uint8_t *, uint8_t *, const uint8_t *, const int *, int, int);
cudaError_t tehmm_launch_tb_verify(cudaStream_t, const TehmmBatchDev &, uint8_t *, const uint8_t *, uint8_t *, int *, int *);
cudaError_t tehmm_launch_rescore(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, const uint8_t *, const double *, const double *, double *, double *, int64_t, int64_t);
cudaError_t tehmm_launch_emission_stats(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const void *, const double *, double *, double *, int, int);
size_t tehmm_stats_smem_bytes(int tab_rows, int N, int K, int prec);
cudaError_t tehmm_launch_forward_tile(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, const float *, const double *, float *, float *, float *, double *, const int *, int, int, int64_t);
cudaError_t tehmm_launch_backward_tile(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const float *, const float *, float *, uint8_t *, double *, float *, float *, const int *, int, int);
int tehmm_tile_warps(void);
bool tehmm_forward_umma_ok(const TehmmModelDev &, const TehmmBatchDev &, int, int64_t);
cudaError_t tehmm_launch_forward_umma(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, const float *, const double *, float *, float *, float *, double *, int, int64_t, int *);
bool tehmm_backward_umma_ok(const TehmmModelDev &, const TehmmBatchDev &, int, int, int64_t);
cudaError_t tehmm_launch_backward_umma(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const float *, const float *, float *, uint8_t *, double *, float *, float *, int, int64_t, int *);
cudaError_t tehmm_launch_xi_mma(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, const float *, const float *, double *, float *, double *, int);
size_t tehmm_xi_mma_scratch_bytes(int sms);
cudaError_t tehmm_launch_convert(cudaStream_t, int, const void *, double *, int64_t);
cudaError_t tehmm_launch_transfer_ops(cudaStream_t, const TehmmModelDev &, const TehmmChunk *, const int64_t *, int64_t, int, int, const void *, void *, double *, int);
cudaError_t tehmm_launch_ratio_fold(cudaStream_t, const TehmmModelDev &, int64_t, int, const double *, void *, double *, int);
cudaError_t tehmm_launch_ratio_diag(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const double *, const void *, double *, double *, int);
cudaError_t tehmm_launch_chain(cudaStream_t, const TehmmModelDev &, int, int, int, const int64_t *, const int64_t *, int64_t, const void *, const double *, const void *, void *);
cudaError_t tehmm_launch_entry(cudaStream_t, const TehmmBatchDev &, int, int, int64_t, const int64_t *, const double *, void *, int *);
cudaError_t tehmm_launch_vit_exit(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, const void *, int64_t, const int64_t *, const int32_t *, const double *, uint8_t *, uint8_t *, int *);
cudaError_t tehmm_launch_exit(cudaStream_t, const TehmmModelDev &, const TehmmBatchDev &, int, int64_t, const int64_t *, const double *, void *, void *, void *, int);
cudaError_t tehmm_launch_cut_pair(cudaStream_t, const TehmmModelDev &, int, const double *, const void *, double *, double *);
cudaError_t tehmm_launch_convert_rows(cudaStream_t, int, int, int, const void *, int64_t, int, double *, int);

// ---------------------------------------------------------------- errors
static thread_local std::string g_err;
static int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
void tehmm_set_error(int code, const char *msg) { (void)code; g_err = msg ? msg : ""; }   // host.cu
void tehmm_hostpipe_release(tehmm_ctx *c);                                                  // host.cu
#define CU(x)                                                                                 \
    do {                                                                                      \
        cudaError_t e__ = (x);                                                                \
        if (e__ != cudaSuccess)                                                               \
            return fail(TEHMM_ECUDA, "%s failed: %s (%s:%d)", #x, cudaGetErrorString(e__),    \
                        __FILE__, __LINE__);                                                  \
    } while (0)

struct DevBuf {   // RAII device allocation for the strict host-pointer entry points
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t n) { return cudaMalloc(&p, n ? n : 1); }
    template <typename T> T *as() { return (T *)p; }
};

#define TEHMM_TRING 32
#define TEHMM_NPENDING 64
enum { TK_EMISSION, TK_FORWARD, TK_BACKWARD, TK_VITERBI_DP, TK_TRACEBACK, TK_RESCORE, TK_STATS, TK_XI, TEHMM_NTIMED };
static const char *const tk_names[TEHMM_NTIMED] = {"us_emission", "us_forward", "us_backward", "us_viterbi_dp",
                                                    "us_traceback", "us_rescore", "us_emission_stats", "us_xi"};

struct tehmm_ctx {
    int device = 0;
    int sms = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    int64_t launches = 0;
    int64_t opt_chunk_tiles = 0, opt_warmup = 0, opt_max_repair = 0;
    int64_t opt_tile = 1, opt_fine_len = 0;   // tensor-core kernels (tile.cu, umma.cu) on / fine chunk length (0 = auto)
    // option "timing": CUDA events around the first (speculative) launch of each main kernel, on the
    // launching stream; read back in microseconds with tehmm_ctx_get_stat("us_<kernel>")
    int64_t opt_timing = 0;
    int *d_fault = nullptr;           // raised by a kernel whose barrier protocol timed out
    int64_t stat_umma_passes = 0;
    int64_t opt_rescore = 0;          // 1: the Viterbi log-probability is always the float64 re-score of the returned path (default: the fp32 DP's own normaliser sum where the lean kernel runs)
    // ordinary repair passes before the chunks still flagged are resolved exactly by transfer operators
    // (fallback.cu; -1 = never: the plain loop, one pass per link of a chain of bad chunks)
    int64_t opt_fallback_after = 2;
    int64_t stat_fallbacks = 0, stat_fallback_chunks = 0, stat_noise_accepted = 0;
    // modulus of the second eigenvalue of the transition matrix: computed on first use (mix_rho_of) from the
    // row-normalised matrix kept by set_model -- only the exact fallback and the "mix_rho_ppm" statistic ask for it,
    // and the estimate (2000 power iterations) costs more host time than the rest of set_model, once per EM iteration
    double mix_rho = -1.0;
    std::vector<double> mix_A;
    int mix_N = 0;
    cudaEvent_t ev[TEHMM_NTIMED][TEHMM_TRING][2] = {};
    int ev_n[TEHMM_NTIMED] = {};          // launches recorded since "timing" was last set (ring of TEHMM_TRING)
    int64_t stat_repair_fwd = 0, stat_repair_bwd = 0, stat_repair_vit = 0;
    int64_t stat_tile_passes = 0;
    int64_t stat_bad_fwd = 0, stat_bad_bwd = 0, stat_bad_vit = 0, stat_bad_tb = 0, stat_repair_tb = 0;
    int *h_nbad = nullptr;            // pinned
    // option "defer": the verification count of a pass is copied to a pinned slot and read at the
    // next tehmm_ctx_check instead of stalling the stream after every stage (api: tehmm_ctx_check)
    int64_t opt_defer = 0;
    int *h_pending = nullptr;         // pinned, TEHMM_NPENDING slots
    int npending = 0;
    int64_t defer_skip = 0, defer_penalty = 0;   // back-off after a refused check (tehmm_ctx_check)
    int64_t stat_deferred_checks = 0, stat_deferred_bad = 0;
    // model
    bool has_model = false;
    TehmmModelDev m{};
    void *model_blob = nullptr;
    size_t model_blob_bytes = 0;
    std::vector<unsigned char> model_key;     // raw inputs of the last tehmm_set_model
    // batch
    bool has_batch = false;
    TehmmBatchDev b{};            // coarse partition: one chunk per warp (forward.cu, backward.cu, viterbi.cu)
    TehmmBatchDev bf{};           // fine partition: sixteen chunks per warp (tile.cu)
    std::vector<int64_t> batch_key;   // offsets, address and options of the last tehmm_set_batch
    void *batch_blob = nullptr;
    size_t batch_blob_bytes = 0;      // capacity (grow-only: decode calls come back with similar batches)
    int *d_seq_flag = nullptr;
    int64_t seq_flag_n = 0;
    int64_t max_tiles_per_chunk = 1;
    int64_t fine_len = 0;         // steps per chunk of the fine partition
    // boundary conditions of the current batch (tehmm_set_boundary, window.cu; cleared by tehmm_set_batch):
    // blob = cont[nseq] | entry_seq[n_entry] | entry_vec[n_entry][NP] | exit_seq[n_exit] | exit_vec[n_exit][NP]
    //        | the rows exit_kernel saves (n_exit x 2 x LD elements of float64 size)
    int64_t n_entry = 0, n_exit = 0;
    void *bnd_blob = nullptr;
    size_t bnd_blob_bytes = 0;
    const int64_t *d_entry_seq = nullptr, *d_exit_seq = nullptr;
    const double *d_entry_vec = nullptr, *d_exit_vec = nullptr;
    void *d_exit_save = nullptr;
    // Viterbi boundary conditions (tehmm_set_viterbi_boundary; cleared by tehmm_set_batch):
    // vbnd_blob = entry_seq[n_ventry] | entry_delta[n_ventry][NP] | exit_seq[n_vexit] | exit_state[n_vexit] | exit_ratio[n_vexit]
    int64_t n_ventry = 0, n_vexit = 0;
    void *vbnd_blob = nullptr;
    size_t vbnd_blob_bytes = 0;
    const int64_t *d_ventry_seq = nullptr, *d_vexit_seq = nullptr;
    const double *d_ventry_vec = nullptr, *d_vexit_ratio = nullptr;
    const int32_t *d_vexit_state = nullptr;
};

extern "C" {

int tehmm_abi_version(void) { return TEHMM_ABI_VERSION; }
const char *tehmm_last_error(void) { return g_err.c_str(); }

int tehmm_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int tehmm_ctx_create(int device, tehmm_ctx **out)
{
    if (!out) return fail(TEHMM_EINVAL, "out is NULL");
    int n = tehmm_device_count();
    if (n <= 0) return fail(TEHMM_ECUDA, "no CUDA device visible: libtehmm_b200 has no CPU fallback");
    if (device < 0 || device >= n) return fail(TEHMM_EINVAL, "device %d out of range (0..%d)", device, n - 1);
    CU(cudaSetDevice(device));
    tehmm_ctx *c = new tehmm_ctx();
    c->device = device;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    c->sms = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    CU(cudaMallocHost((void **)&c->h_nbad, 2 * sizeof(int)));
    CU(cudaMallocHost((void **)&c->h_pending, TEHMM_NPENDING * sizeof(int)));
    CU(cudaMalloc((void **)&c->d_fault, sizeof(int)));
    CU(cudaMemset(c->d_fault, 0, sizeof(int)));
    *out = c;
    return TEHMM_OK;
}

int tehmm_ctx_destroy(tehmm_ctx *c)
{
    if (!c) return TEHMM_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    tehmm_hostpipe_release(c);
    if (c->model_blob) cudaFree(c->model_blob);
    if (c->batch_blob) cudaFree(c->batch_blob);
    if (c->bnd_blob) cudaFree(c->bnd_blob);
    if (c->vbnd_blob) cudaFree(c->vbnd_blob);
    if (c->d_seq_flag) cudaFree(c->d_seq_flag);
    if (c->h_nbad) cudaFreeHost(c->h_nbad);
    if (c->h_pending) cudaFreeHost(c->h_pending);
    if (c->d_fault) cudaFree(c->d_fault);
    for (int i = 0; i < TEHMM_NTIMED; ++i)
        for (int r = 0; r < TEHMM_TRING; ++r)
            for (int j = 0; j < 2; ++j)
                if (c->ev[i][r][j]) cudaEventDestroy(c->ev[i][r][j]);
    cudaStreamDestroy(c->own_stream);
    delete c;
    return TEHMM_OK;
}

int tehmm_ctx_sync(tehmm_ctx *c)
{
    if (!c) return fail(TEHMM_EINVAL, "ctx is NULL");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return TEHMM_OK;
}

int tehmm_ctx_set_stream(tehmm_ctx *c, uint64_t stream)
{
    if (!c) return fail(TEHMM_EINVAL, "ctx is NULL");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    // 0 is a real stream (the legacy default stream torch uses unless told otherwise)
    c->stream = stream == UINT64_MAX ? c->own_stream : (cudaStream_t)(uintptr_t)stream;
    return TEHMM_OK;
}

uint64_t tehmm_ctx_stream(tehmm_ctx *c) { return c ? (uint64_t)(uintptr_t)c->stream : 0; }
int64_t tehmm_ctx_launch_count(tehmm_ctx *c) { return c ? c->launches : 0; }

int tehmm_ctx_set_option(tehmm_ctx *c, const char *name, int64_t v)
{
    if (!c || !name) return fail(TEHMM_EINVAL, "NULL argument");
    if (!strcmp(name, "chunk_tiles")) c->opt_chunk_tiles = v;
    else if (!strcmp(name, "warmup")) c->opt_warmup = v;
    else if (!strcmp(name, "max_repair")) c->opt_max_repair = v;
    else if (!strcmp(name, "tile")) c->opt_tile = v;
    else if (!strcmp(name, "timing")) { c->opt_timing = v; for (int i = 0; i < TEHMM_NTIMED; ++i) c->ev_n[i] = 0; }
    else if (!strcmp(name, "fine_len")) c->opt_fine_len = v;
    else if (!strcmp(name, "defer")) {
        if (v && c->defer_skip > 0) { c->defer_skip -= 1; v = 0; }
        c->opt_defer = v;
    }
    else if (!strcmp(name, "defer_skip")) c->defer_skip = v;
    else if (!strcmp(name, "rescore")) c->opt_rescore = v;
    else if (!strcmp(name, "fallback_after")) c->opt_fallback_after = v;
    else return fail(TEHMM_EINVAL, "unknown option %s", name);
    return TEHMM_OK;
}

// How fast the chain forgets with NO help from the data (all-missing stretches): rho = |lambda_2(A)|,
// estimated as ||B^256||_F^(1/256), B = A - 1 pi^T (pi = stationary distribution by power iteration).
// Rounding noise of a filter is amplified by 1 / (1 - rho); see tolerance_after_fallback.
static double mix_rho_of(tehmm_ctx *c)
{
    if (c->mix_rho >= 0.0) return c->mix_rho;
    const int N = c->mix_N;
    if (N <= 0 || c->mix_A.size() != (size_t)N * N) return 0.0;
    const std::vector<double> &A = c->mix_A;
    std::vector<double> pi(N, 1.0 / N), tmp(N), B((size_t)N * N), B2((size_t)N * N);
    for (int it = 0; it < 2000; ++it) {
        double sum = 0.0;
        for (int j = 0; j < N; ++j) tmp[j] = 0.0;
        for (int i = 0; i < N; ++i) {
            const double p = pi[i];
            for (int j = 0; j < N; ++j) tmp[j] += p * A[(size_t)i * N + j];
        }
        for (int j = 0; j < N; ++j) sum += tmp[j];
        for (int j = 0; j < N; ++j) pi[j] = sum > 0.0 ? tmp[j] / sum : 1.0 / N;
    }
    for (int i = 0; i < N; ++i) for (int j = 0; j < N; ++j) B[(size_t)i * N + j] = A[(size_t)i * N + j] - pi[j];
    double lognorm = 0.0;                 // log ||B^(2^k)||_F accumulated with renormalisation
    for (int sq = 0; sq < 8; ++sq) {
        double f = 0.0;
        for (double v : B) f += v * v;
        f = sqrt(f);
        if (!(f > 0.0)) { lognorm = -INFINITY; break; }
        for (double &v : B) v /= f;
        lognorm = 2.0 * (lognorm + log(f));
        for (int i = 0; i < N; ++i)
            for (int j = 0; j < N; ++j) { double a = 0.0; for (int k = 0; k < N; ++k) a += B[(size_t)i * N + k] * B[(size_t)k * N + j]; B2[(size_t)i * N + j] = a; }
        B.swap(B2);
    }
    if (lognorm > -INFINITY) { double f = 0.0; for (double v : B) f += v * v; lognorm += f > 0.0 ? 0.5 * log(f) : -INFINITY; }
    const double rho = lognorm > -INFINITY ? exp(lognorm / 256.0) : 0.0;
    c->mix_rho = std::min(1.0, std::max(0.0, rho));
    return c->mix_rho;
}

int64_t tehmm_ctx_get_stat(tehmm_ctx *c, const char *name)
{
    if (!c || !name) return -1;
    if (!strcmp(name, "launches")) return c->launches;
    if (!strcmp(name, "repair_passes_forward")) return c->stat_repair_fwd;
    if (!strcmp(name, "repair_passes_backward")) return c->stat_repair_bwd;
    if (!strcmp(name, "repair_passes_viterbi")) return c->stat_repair_vit;
    if (!strcmp(name, "repaired_chunks_forward")) return c->stat_bad_fwd;
    if (!strcmp(name, "repaired_chunks_backward")) return c->stat_bad_bwd;
    if (!strcmp(name, "repaired_chunks_viterbi")) return c->stat_bad_vit;
    if (!strcmp(name, "repaired_chunks_traceback")) return c->stat_bad_tb;
    if (!strcmp(name, "repair_passes_traceback")) return c->stat_repair_tb;
    if (!strcmp(name, "sms")) return c->sms;
    if (!strcmp(name, "deferred_checks")) return c->stat_deferred_checks;
    if (!strcmp(name, "deferred_bad")) return c->stat_deferred_bad;
    if (!strcmp(name, "defer_skip")) return c->defer_skip;
    if (!strcmp(name, "chunks")) return c->has_batch ? c->b.nchunks : 0;
    if (!strcmp(name, "fine_chunks")) return c->has_batch ? c->bf.nchunks : 0;
    if (!strcmp(name, "tile_passes")) return c->stat_tile_passes;
    if (!strcmp(name, "umma_passes")) return c->stat_umma_passes;
    if (!strcmp(name, "fallbacks")) return c->stat_fallbacks;
    if (!strcmp(name, "fallback_chunks")) return c->stat_fallback_chunks;
    if (!strcmp(name, "noise_accepted")) return c->stat_noise_accepted;
    if (!strcmp(name, "mix_rho_ppm")) return (int64_t)(mix_rho_of(c) * 1e6);
    for (int i = 0; i < TEHMM_NTIMED; ++i)
        if (!strcmp(name, tk_names[i])) {
            // average over the launches recorded since "timing" was set (at most the last TEHMM_TRING)
            const int n = std::min(c->ev_n[i], TEHMM_TRING);
            if (n <= 0) return -1;
            double tot = 0.0;
            for (int r = 0; r < n; ++r) {
                float ms = 0.f;
                if (cudaEventSynchronize(c->ev[i][r][1]) != cudaSuccess || cudaEventElapsedTime(&ms, c->ev[i][r][0], c->ev[i][r][1]) != cudaSuccess) return -1;
                tot += ms;
            }
            return (int64_t)(tot / n * 1000.0 + 0.5);
        }
    if (!strcmp(name, "warmup")) return c->has_batch ? c->b.warmup : 0;
    return -1;
}

// ================================================================ L0 strict
#define STRICT_PROLOGUE()                                                      \
    if (!c) return fail(TEHMM_EINVAL, "ctx is NULL");                          \
    CU(cudaSetDevice(c->device));                                              \
    cudaStream_t st = c->stream
#define H2D(dst, src, bytes) CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st))
#define D2H(dst, src, bytes) CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st))

static int check_obs_bytes(int nb)
{
    if (nb != 1 && nb != 2 && nb != 4) return fail(TEHMM_EINVAL, "obs_bytes must be 1, 2 or 4 (got %d)", nb);
    return 0;
}

int tehmm_strict_all_log_probs(tehmm_ctx *c, const void *obs, int obs_bytes, int64_t T, int K,
                               const double *table, int N, int S, double *out, double normalize,
                               const double *ratios)
{
    STRICT_PROLOGUE();
    if (!obs || !table || !out || T < 0 || K <= 0 || N <= 0 || S <= 0) return fail(TEHMM_EINVAL, "bad argument");
    if (check_obs_bytes(obs_bytes)) return TEHMM_EINVAL;
    if (T == 0) return TEHMM_OK;
    DevBuf dobs, dtab, dout, drat, dfirst;
    size_t ob = (size_t)T * K * obs_bytes, tb = (size_t)K * N * S * 8, fb = (size_t)T * N * 8;
    CU(dobs.alloc(ob)); CU(dtab.alloc(tb)); CU(dout.alloc(fb)); CU(dfirst.alloc(8));
    H2D(dobs.p, obs, ob); H2D(dtab.p, table, tb);
    if (ratios) { CU(drat.alloc((size_t)T * 8)); H2D(drat.p, ratios, (size_t)T * 8); }
    CU(cudaMemsetAsync(dfirst.p, 0xff, 8, st));
    tehmm_launch_strict_emission(st, dobs.p, obs_bytes, T, K, dtab.as<double>(), N, S, dout.as<double>(),
                                 normalize, ratios ? drat.as<double>() : nullptr, dfirst.as<unsigned long long>());
    c->launches += 2;
    CU(cudaGetLastError());
    D2H(out, dout.p, fb);
    CU(cudaStreamSynchronize(st));
    return TEHMM_OK;
}

int tehmm_strict_forward(tehmm_ctx *c, int64_t T, int N, const double *log_start,
                         const double *log_trans, const double *frame, const double *ratios,
                         double *fwd)
{
    STRICT_PROLOGUE();
    if (!log_start || !log_trans || !frame || !fwd || T <= 0 || N <= 0) return fail(TEHMM_EINVAL, "bad argument");
    if ((size_t)N * 16 > 200 * 1024) return fail(TEHMM_ELIMIT, "N=%d too large", N);
    DevBuf ds, dt, df, dr, dout;
    size_t fb = (size_t)T * N * 8;
    CU(ds.alloc((size_t)N * 8)); CU(dt.alloc((size_t)N * N * 8)); CU(df.alloc(fb)); CU(dout.alloc(fb));
    H2D(ds.p, log_start, (size_t)N * 8); H2D(dt.p, log_trans, (size_t)N * N * 8); H2D(df.p, frame, fb);
    if (ratios) { CU(dr.alloc((size_t)T * 8)); H2D(dr.p, ratios, (size_t)T * 8); }
    tehmm_launch_strict_forward(st, T, N, ds.as<double>(), dt.as<double>(), df.as<double>(),
                                ratios ? dr.as<double>() : nullptr, dout.as<double>());
    c->launches += 1;
    CU(cudaGetLastError());
    D2H(fwd, dout.p, fb);
    CU(cudaStreamSynchronize(st));
    return TEHMM_OK;
}

int tehmm_strict_backward(tehmm_ctx *c, int64_t T, int N, const double *log_start,
                          const double *log_trans, const double *frame, const double *ratios,
                          double *bwd)
{
    (void)log_start;   // accepted and ignored, as in _hmm.pyx:160-198
    STRICT_PROLOGUE();
    if (!log_trans || !frame || !bwd || T <= 0 || N <= 0) return fail(TEHMM_EINVAL, "bad argument");
    DevBuf dt, df, dr, dout;
    size_t fb = (size_t)T * N * 8;
    CU(dt.alloc((size_t)N * N * 8)); CU(df.alloc(fb)); CU(dout.alloc(fb));
    H2D(dt.p, log_trans, (size_t)N * N * 8); H2D(df.p, frame, fb);
    if (ratios) { CU(dr.alloc((size_t)T * 8)); H2D(dr.p, ratios, (size_t)T * 8); }
    tehmm_launch_strict_backward(st, T, N, dt.as<double>(), df.as<double>(),
                                 ratios ? dr.as<double>() : nullptr, dout.as<double>());
    c->launches += 1;
    CU(cudaGetLastError());
    D2H(bwd, dout.p, fb);
    CU(cudaStreamSynchronize(st));
    return TEHMM_OK;
}

int tehmm_strict_viterbi(tehmm_ctx *c, int64_t T, int N, const double *log_start,
                         const double *log_trans, const double *ratios, const double *frame,
                         int64_t *states, double *logprob)
{
    STRICT_PROLOGUE();
    if (!log_start || !log_trans || !frame || !states || !logprob || T <= 0 || N <= 0) return fail(TEHMM_EINVAL, "bad argument");
    if (N > 32767) return fail(TEHMM_ELIMIT, "N=%d exceeds the int16 back-pointer range", N);
    DevBuf ds, dt, df, dr, dbp, dst_, dlp;
    size_t fb = (size_t)T * N * 8;
    CU(ds.alloc((size_t)N * 8)); CU(dt.alloc((size_t)N * N * 8)); CU(df.alloc(fb));
    CU(dbp.alloc((size_t)T * N * 2)); CU(dst_.alloc((size_t)T * 8)); CU(dlp.alloc(8));
    H2D(ds.p, log_start, (size_t)N * 8); H2D(dt.p, log_trans, (size_t)N * N * 8); H2D(df.p, frame, fb);
    if (ratios) { CU(dr.alloc((size_t)T * 8)); H2D(dr.p, ratios, (size_t)T * 8); }
    tehmm_launch_strict_viterbi(st, T, N, ds.as<double>(), dt.as<double>(), ratios ? dr.as<double>() : nullptr,
                                df.as<double>(), dbp.as<int16_t>(), dst_.as<int64_t>(), dlp.as<double>());
    c->launches += 1;
    CU(cudaGetLastError());
    D2H(states, dst_.p, (size_t)T * 8);
    D2H(logprob, dlp.p, 8);
    CU(cudaStreamSynchronize(st));
    return TEHMM_OK;
}

int tehmm_strict_log_sum_lneta(tehmm_ctx *c, int64_t T, int N, const double *fwd,
                               const double *log_trans, const double *bwd, const double *frame,
                               double logprob, const double *ratios, double *out)
{
    STRICT_PROLOGUE();
    if (!fwd || !log_trans || !bwd || !frame || !out || T <= 0 || N <= 0) return fail(TEHMM_EINVAL, "bad argument");
    DevBuf dfw, dt, dbw, dfr, dr, dout;
    size_t fb = (size_t)T * N * 8, nb = (size_t)N * N * 8;
    CU(dfw.alloc(fb)); CU(dbw.alloc(fb)); CU(dfr.alloc(fb)); CU(dt.alloc(nb)); CU(dout.alloc(nb));
    H2D(dfw.p, fwd, fb); H2D(dbw.p, bwd, fb); H2D(dfr.p, frame, fb); H2D(dt.p, log_trans, nb); H2D(dout.p, out, nb);
    if (ratios) { CU(dr.alloc((size_t)T * 8)); H2D(dr.p, ratios, (size_t)T * 8); }
    tehmm_launch_strict_lneta(st, T, N, dfw.as<double>(), dt.as<double>(), dbw.as<double>(), dfr.as<double>(),
                              logprob, ratios ? dr.as<double>() : nullptr, dout.as<double>());
    c->launches += 1;
    CU(cudaGetLastError());
    D2H(out, dout.p, nb);
    CU(cudaStreamSynchronize(st));
    return TEHMM_OK;
}

int tehmm_strict_accumulate_stats(tehmm_ctx *c, const void *obs, int obs_bytes, int64_t T, int K,
                                  double *stats, int N, int S, const double *post,
                                  const double *ratios)
{
    STRICT_PROLOGUE();
    if (!obs || !stats || !post || T < 0 || K <= 0 || N <= 0 || S <= 0) return fail(TEHMM_EINVAL, "bad argument");
    if (check_obs_bytes(obs_bytes)) return TEHMM_EINVAL;
    if (T == 0) return TEHMM_OK;
    DevBuf dobs, dst_, dp, dr;
    size_t ob = (size_t)T * K * obs_bytes, sb = (size_t)K * N * S * 8, pb = (size_t)T * N * 8;
    CU(dobs.alloc(ob)); CU(dst_.alloc(sb)); CU(dp.alloc(pb));
    H2D(dobs.p, obs, ob); H2D(dst_.p, stats, sb); H2D(dp.p, post, pb);
    if (ratios) { CU(dr.alloc((size_t)T * 8)); H2D(dr.p, ratios, (size_t)T * 8); }
    tehmm_launch_strict_accumulate(st, dobs.p, obs_bytes, T, K, dst_.as<double>(), N, S, dp.as<double>(),
                                   ratios ? dr.as<double>() : nullptr);
    c->launches += 1;
    CU(cudaGetLastError());
    D2H(stats, dst_.p, sb);
    CU(cudaStreamSynchronize(st));
    return TEHMM_OK;
}

int tehmm_strict_update_counts(tehmm_ctx *c, const void *obs, int obs_bytes, int64_t T, int K,
                               int64_t start, int64_t end, int state, double *stats, int N, int S,
                               const double *ratios)
{
    STRICT_PROLOGUE();
    if (!obs || !stats || T < 0 || K <= 0 || N <= 0 || S <= 0) return fail(TEHMM_EINVAL, "bad argument");
    if (check_obs_bytes(obs_bytes)) return TEHMM_EINVAL;
    if (start < 0 || end > T || state < 0 || state >= N) return fail(TEHMM_EINVAL, "interval [%lld,%lld) state %d outside table (T=%lld, N=%d)", (long long)start, (long long)end, state, (long long)T, N);
    if (end <= start) return TEHMM_OK;
    DevBuf dobs, dst_, dr;
    // only the rows of the interval travel
    size_t ob = (size_t)(end - start) * K * obs_bytes, sb = (size_t)K * N * S * 8;
    CU(dobs.alloc(ob)); CU(dst_.alloc(sb));
    H2D(dobs.p, (const char *)obs + (size_t)start * K * obs_bytes, ob); H2D(dst_.p, stats, sb);
    if (ratios) { CU(dr.alloc((size_t)(end - start) * 8)); H2D(dr.p, ratios + start, (size_t)(end - start) * 8); }
    tehmm_launch_strict_counts(st, dobs.p, obs_bytes, K, 0, end - start, state, dst_.as<double>(), N, S,
                               ratios ? dr.as<double>() : nullptr);
    c->launches += 1;
    CU(cudaGetLastError());
    D2H(stats, dst_.p, sb);
    CU(cudaStreamSynchronize(st));
    return TEHMM_OK;
}

int tehmm_supervised_counts(tehmm_ctx *c, const void *d_obs, int obs_bytes, int64_t total, int K, int64_t n,
                            const int64_t *h_row_start, const int64_t *h_row_end, const int32_t *h_state,
                            const double *d_ratios, double *h_stats, int N, int S)
{
    STRICT_PROLOGUE();
    if (!d_obs || !h_stats || total < 0 || n < 0 || K <= 0 || N <= 0 || S <= 0) return fail(TEHMM_EINVAL, "bad argument");
    if (n > 0 && (!h_row_start || !h_row_end || !h_state)) return fail(TEHMM_EINVAL, "NULL interval arrays");
    if (check_obs_bytes(obs_bytes)) return TEHMM_EINVAL;
    // group the non-empty intervals by state, interval order kept within a state (counting sort)
    std::vector<int64_t> sbeg(N + 2, 0);
    int64_t rows = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t a = h_row_start[i], b = h_row_end[i];
        if (a < 0 || a > total || b > total)
            return fail(TEHMM_EINVAL, "interval %lld: rows [%lld,%lld) outside [0,%lld)", (long long)i, (long long)a, (long long)b, (long long)total);
        if (h_state[i] < 0 || h_state[i] >= N)
            return fail(TEHMM_EINVAL, "interval %lld: state %d outside [0,%d)", (long long)i, h_state[i], N);
        if (b > a) { sbeg[h_state[i] + 2] += 1; rows += b - a; }
    }
    if (rows == 0) return TEHMM_OK;
    for (int s = 0; s < N; ++s) sbeg[s + 2] += sbeg[s + 1];
    const int64_t m = sbeg[N + 1];
    // blob: istart[m] | pfx[m + 1] | sbeg[N + 1] | sflat[N + 1]
    std::vector<int64_t> blob(2 * m + 1 + 2 * (N + 1));
    int64_t *istart = blob.data(), *pfx = istart + m, *hs = pfx + m + 1, *hf = hs + N + 1;
    std::vector<int64_t> len(m);
    for (int64_t i = 0; i < n; ++i) {
        const int64_t a = h_row_start[i], b = h_row_end[i];
        if (b <= a) continue;
        const int64_t j = sbeg[h_state[i] + 1]++;
        istart[j] = a;
        len[j] = b - a;
    }
    pfx[0] = 0;
    for (int64_t j = 0; j < m; ++j) pfx[j + 1] = pfx[j] + len[j];
    for (int s = 0; s <= N; ++s) { hs[s] = sbeg[s]; hf[s] = pfx[sbeg[s]]; }
    // integer regime: unit weights and initial values that stay exact integers after every count is added
    const size_t bins = (size_t)K * N * S;
    bool integral = d_ratios == nullptr;
    for (size_t i = 0; integral && i < bins; ++i) {
        const double v = h_stats[i];
        integral = v == floor(v) && fabs(v) + (double)rows <= 9007199254740992.0;
    }
    DevBuf dblob, dstats, dcounts, dflag;
    CU(dblob.alloc(blob.size() * 8)); CU(dstats.alloc(bins * 8)); CU(dflag.alloc(sizeof(int)));
    H2D(dblob.p, blob.data(), blob.size() * 8);
    H2D(dstats.p, h_stats, bins * 8);
    CU(cudaMemsetAsync(dflag.p, 0, sizeof(int), st));
    const int64_t *d_istart = dblob.as<int64_t>(), *d_pfx = d_istart + m, *d_sbeg = d_pfx + m + 1, *d_sflat = d_sbeg + N + 1;
    if (integral) {
        CU(dcounts.alloc(bins * 8));
        CU(cudaMemsetAsync(dcounts.p, 0, bins * 8, st));
        c->launches += tehmm_launch_sup_hist(st, d_obs, obs_bytes, K, N, S, m, rows, d_istart, d_pfx, d_sflat,
                                             dcounts.as<unsigned long long>(), dstats.as<double>(), dflag.as<int>());
    } else {
        c->launches += tehmm_launch_sup_chain(st, d_obs, obs_bytes, K, N, S, d_istart, d_pfx, d_sbeg, d_sflat,
                                              d_ratios, dstats.as<double>(), dflag.as<int>());
    }
    CU(cudaGetLastError());
    int h_flag = 0;
    std::vector<double> out(bins);
    D2H(&h_flag, dflag.p, sizeof(int));
    D2H(out.data(), dstats.p, bins * 8);
    CU(cudaStreamSynchronize(st));
    if (h_flag) return fail(TEHMM_EINVAL, "an observation in a counted row is >= S=%d (or negative)", S);
    memcpy(h_stats, out.data(), bins * 8);
    return TEHMM_OK;
}

// ================================================================ L1 batched
static size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

int tehmm_set_model(tehmm_ctx *c, int N, int K, int S, const double *log_start,
                    const double *log_trans, const double *table, double normalize,
                    const int32_t *track_nsym)
{
    if (!c || !log_start || !log_trans || !table) return fail(TEHMM_EINVAL, "NULL argument");
    if (N <= 0 || K <= 0 || S <= 0) return fail(TEHMM_EINVAL, "bad shape N=%d K=%d S=%d", N, K, S);
    if (N > TEHMM_MAX_STATES) return fail(TEHMM_ELIMIT, "batched path supports N <= %d (got %d)", TEHMM_MAX_STATES, N);
    {   // decode()/score() hand the same model over on every call: skip the rebuild when nothing changed
        const size_t nb = (size_t)N * 8 + (size_t)N * N * 8 + (size_t)K * N * S * 8;
        std::vector<unsigned char> key(32 + nb + (size_t)K * 4, 0);
        int32_t hdr[4] = {N, K, S, track_nsym ? 1 : 0};
        memcpy(&key[0], hdr, 16);
        memcpy(&key[16], &normalize, 8);
        unsigned char *q = &key[32];
        memcpy(q, log_start, (size_t)N * 8); q += (size_t)N * 8;
        memcpy(q, log_trans, (size_t)N * N * 8); q += (size_t)N * N * 8;
        memcpy(q, table, (size_t)K * N * S * 8); q += (size_t)K * N * S * 8;
        if (track_nsym) memcpy(q, track_nsym, (size_t)K * 4);
        if (c->has_model && key == c->model_key) return TEHMM_OK;
        c->model_key.swap(key);
        c->has_model = false;
    }
    CU(cudaSetDevice(c->device));
    const int NS = N <= 32 ? 1 : 2, NP = 32 * NS;
    std::vector<int32_t> nsym(K), off(K);
    int rows = 0;
    for (int k = 0; k < K; ++k) {
        int n = track_nsym ? track_nsym[k] : S;
        if (n < 1 || n > S) return fail(TEHMM_EINVAL, "track_nsym[%d]=%d outside 1..%d", k, n, S);
        nsym[k] = n; off[k] = rows; rows += n;
    }
    // host-side staging of everything in one blob
    size_t o_ls = 0, o_lt = align_up(o_ls + (size_t)N * 8), o_tab = align_up(o_lt + (size_t)N * N * 8);
    size_t o_tt = align_up(o_tab + (size_t)K * N * S * 8), o_off = align_up(o_tt + (size_t)rows * N * 8);
    size_t o_ns = align_up(o_off + (size_t)K * 4), o_lins = align_up(o_ns + (size_t)K * 4);
    size_t o_lint = align_up(o_lins + (size_t)NP * 8), o_cuts = align_up(o_lint + (size_t)NP * NP * 8);
    size_t o_cutt = align_up(o_cuts + (size_t)NP * 8), o_end = align_up(o_cutt + (size_t)NP * NP * 8);
    // merged emission tables (fp32 path, N <= 32): group tracks so that a row of the batch
    // needs as few table look-ups as possible within the shared-memory budget.  Greedy:
    // repeatedly merge the two groups whose merge adds the fewest rows.
    struct Grp { std::vector<int> trk; int64_t rows; };
    auto make_groups = [&](int64_t row_budget, int max_groups, std::vector<Grp> &grp, bool wide_ok) -> int64_t {
        int64_t total_rows = 0;
        grp.clear();
        if (NS != 1 && !wide_ok) return 0;
        for (int k = 0; k < K; ++k) { grp.push_back(Grp{{k}, nsym[k]}); total_rows += nsym[k]; }
        for (;;) {
            int bi = -1, bj = -1;
            int64_t best = 0;
            for (size_t i = 0; i < grp.size(); ++i)
                for (size_t j = i + 1; j < grp.size(); ++j) {
                    if (grp[i].trk.size() + grp[j].trk.size() > 4) continue;
                    const int64_t add = grp[i].rows * grp[j].rows - grp[i].rows - grp[j].rows;
                    if (total_rows + add > row_budget) continue;
                    if (bi < 0 || add < best) { bi = (int)i; bj = (int)j; best = add; }
                }
            if (bi < 0) break;
            grp[bi].trk.insert(grp[bi].trk.end(), grp[bj].trk.begin(), grp[bj].trk.end());
            grp[bi].rows *= grp[bj].rows;
            grp.erase(grp.begin() + bj);
            total_rows += best;
        }
        if ((int)grp.size() > max_groups || total_rows > row_budget) { grp.clear(); total_rows = 0; }
        return total_rows;
    };
    auto write_desc = [&](const std::vector<Grp> &grp, int32_t *gd) {
        int64_t base = 0;
        for (size_t gi = 0; gi < grp.size(); ++gi) {
            int32_t *d = gd + gi * TEHMM_GDESC;
            d[0] = (int32_t)grp[gi].trk.size();
            d[1] = (int32_t)base;
            int64_t stride = 1;
            for (size_t i = 0; i < grp[gi].trk.size(); ++i) {
                d[2 + i] = grp[gi].trk[i];
                d[6 + i] = (int32_t)stride;
                stride *= nsym[grp[gi].trk[i]];
            }
            base += grp[gi].rows;
        }
    };
    std::vector<Grp> grp, sgrp;
    // 33..64 states: a merged row is 256 bytes, so half the rows fit (emission_merged_kernel<.., NS = 2>)
    const int64_t grows = make_groups(TEHMM_GROWS_MAX / NS, TEHMM_GMAX, grp, true);
    // second grouping for the emission histograms (stats.cu): a merged row costs 256 bytes there
    const int64_t srows = make_groups(TEHMM_SROWS_MAX, 8, sgrp, false);
    const int SG = (int)sgrp.size();
    const int G = (int)grp.size();
    size_t o_gtab = o_end, o_gc = align_up(o_gtab + (size_t)grows * NP * 4);
    size_t o_gd = align_up(o_gc + (size_t)grows * 8), o_sgd = align_up(o_gd + (size_t)std::max(G, 1) * TEHMM_GDESC * 4);
    size_t total = align_up(o_sgd + (size_t)std::max(SG, 1) * TEHMM_GDESC * 4);
    std::vector<unsigned char> h(total, 0);
    if (SG > 0) write_desc(sgrp, (int32_t *)&h[o_sgd]);
    if (G > 0) {
        float *gtab = (float *)&h[o_gtab];
        double *gc = (double *)&h[o_gc];
        int32_t *gd = (int32_t *)&h[o_gd];
        int64_t base = 0;
        std::vector<double> acc(N);
        for (int gi = 0; gi < G; ++gi) {
            const Grp &gr = grp[gi];
            int32_t *d = gd + (size_t)gi * TEHMM_GDESC;
            d[0] = (int32_t)gr.trk.size();
            d[1] = (int32_t)base;
            int64_t stride = 1;
            for (size_t i = 0; i < gr.trk.size(); ++i) {
                d[2 + i] = gr.trk[i];
                d[6 + i] = (int32_t)stride;
                stride *= nsym[gr.trk[i]];
            }
            for (int64_t row = 0; row < gr.rows; ++row) {
                for (int j = 0; j < N; ++j) acc[j] = 0.0;
                int64_t rem = row;
                for (size_t i = 0; i < gr.trk.size(); ++i) {       // same track order as the reference's sum
                    const int k = gr.trk[i];
                    const int sym = (int)(rem % nsym[k]);
                    rem /= nsym[k];
                    for (int j = 0; j < N; ++j) acc[j] += table[((size_t)k * N + j) * S + sym];
                }
                double mx = -INFINITY;
                for (int j = 0; j < N; ++j) { acc[j] *= normalize; mx = std::max(mx, acc[j]); }
                if (!(mx > -INFINITY)) mx = 0.0;
                gc[base + row] = mx;
                for (int j = 0; j < NP; ++j) gtab[(size_t)(base + row) * NP + j] = j < N ? (float)(acc[j] - mx) : -INFINITY;   // padding never wins a maximum
            }
            base += gr.rows;
        }
    }
    memcpy(&h[o_ls], log_start, (size_t)N * 8);
    memcpy(&h[o_lt], log_trans, (size_t)N * N * 8);
    memcpy(&h[o_tab], table, (size_t)K * N * S * 8);
    double *tt = (double *)&h[o_tt];
    for (int k = 0; k < K; ++k)
        for (int s = 0; s < nsym[k]; ++s)
            for (int j = 0; j < N; ++j)
                tt[(size_t)(off[k] + s) * N + j] = table[((size_t)k * N + j) * S + s];
    memcpy(&h[o_off], off.data(), (size_t)K * 4);
    memcpy(&h[o_ns], nsym.data(), (size_t)K * 4);
    double *lins = (double *)&h[o_lins], *lint = (double *)&h[o_lint];
    double *cuts = (double *)&h[o_cuts], *cutt = (double *)&h[o_cutt];
    const double NEG = -INFINITY;
    for (int i = 0; i < NP; ++i) {
        bool ok = i < N && log_start[i] > TEHMM_LOGZERO_CUT;
        lins[i] = ok ? exp(log_start[i]) : 0.0;
        cuts[i] = ok ? log_start[i] : NEG;
        for (int j = 0; j < NP; ++j) {
            bool okt = i < N && j < N && log_trans[(size_t)i * N + j] > TEHMM_LOGZERO_CUT;
            lint[(size_t)i * NP + j] = okt ? exp(log_trans[(size_t)i * N + j]) : 0.0;
            cutt[(size_t)i * NP + j] = okt ? log_trans[(size_t)i * N + j] : NEG;
        }
    }
    {   // the row-normalised transition matrix, for mix_rho_of
        c->mix_A.assign((size_t)N * N, 0.0);
        c->mix_N = N;
        c->mix_rho = -1.0;
        for (int i = 0; i < N; ++i) {
            double rs = 0.0;
            for (int j = 0; j < N; ++j) rs += lint[(size_t)i * NP + j];
            for (int j = 0; j < N; ++j) c->mix_A[(size_t)i * N + j] = rs > 0.0 ? lint[(size_t)i * NP + j] / rs : (i == j ? 1.0 : 0.0);
        }
    }
    CU(cudaStreamSynchronize(c->stream));
    if (total > c->model_blob_bytes) {
        if (c->model_blob) { cudaFree(c->model_blob); c->model_blob = nullptr; c->model_blob_bytes = 0; }
        CU(cudaMalloc(&c->model_blob, total));
        c->model_blob_bytes = total;
    }
    CU(cudaMemcpy(c->model_blob, h.data(), total, cudaMemcpyHostToDevice));
    unsigned char *d = (unsigned char *)c->model_blob;
    TehmmModelDev &m = c->m;
    m.N = N; m.K = K; m.S = S; m.NS = NS; m.NP = NP; m.tab_rows = rows; m.normalize = normalize;
    m.LD = NP;                      // rows of 32 or 64 elements: 16-byte vector / bulk / tensor-map accesses (N..LD-1 are padding)
    m.table_in_smem = (size_t)rows * N * 8 <= tehmm_emission_table_budget(K) ? 1 : 0;
    m.log_start = (const double *)(d + o_ls); m.log_trans = (const double *)(d + o_lt);
    m.table = (const double *)(d + o_tab); m.table_t = (const double *)(d + o_tt);
    m.tab_off = (const int32_t *)(d + o_off); m.track_nsym = (const int32_t *)(d + o_ns);
    m.lin_start = (const double *)(d + o_lins); m.lin_trans = (const double *)(d + o_lint);
    m.cut_start = (const double *)(d + o_cuts); m.cut_trans = (const double *)(d + o_cutt);
    m.G = normalize > 0.0 ? G : 0;      // a negative factor would flip the row maxima
    m.grows = (int)grows;
    m.gtab = (const float *)(d + o_gtab); m.gc = (const double *)(d + o_gc); m.gdesc = (const int32_t *)(d + o_gd);
    m.SG = SG; m.srows = (int)srows; m.sgdesc = (const int32_t *)(d + o_sgd);
    c->has_model = true;
    return TEHMM_OK;
}

int tehmm_set_batch(tehmm_ctx *c, const void *d_obs, int obs_bytes, int64_t nseq,
                    const int64_t *h_offsets)
{
    if (!c || !d_obs || !h_offsets) return fail(TEHMM_EINVAL, "NULL argument");
    if (check_obs_bytes(obs_bytes)) return TEHMM_EINVAL;
    if (nseq <= 0) return fail(TEHMM_EINVAL, "nseq must be positive");
    if (h_offsets[0] != 0) return fail(TEHMM_EINVAL, "offsets[0] must be 0");
    for (int64_t s = 0; s < nseq; ++s)
        if (h_offsets[s + 1] < h_offsets[s]) return fail(TEHMM_EINVAL, "offsets must be non-decreasing");
    CU(cudaSetDevice(c->device));
    const int64_t total = h_offsets[nseq];
    if (total <= 0) return fail(TEHMM_EINVAL, "empty batch");
    c->n_entry = c->n_exit = 0;               // a new batch starts without boundary vectors
    c->n_ventry = c->n_vexit = 0;
    c->b.cont = c->bf.cont = nullptr;
    {   // the same batch shape at the same address again (a stream of decode calls): keep the partition
        std::vector<int64_t> key(h_offsets, h_offsets + nseq + 1);
        key.push_back((int64_t)(uintptr_t)d_obs); key.push_back(obs_bytes);
        key.push_back(c->opt_chunk_tiles); key.push_back(c->opt_fine_len); key.push_back(c->opt_warmup);
        if (c->has_batch && key == c->batch_key) {
            if (c->opt_warmup <= 0 && c->b.warmup != 64) c->b.warmup = c->bf.warmup = 64;   // forget an adapted warm-up
            return TEHMM_OK;
        }
        c->batch_key.swap(key);
        c->has_batch = false;
    }
    // time partition: tiles of TEHMM_TILE steps, chunks of `tpc` tiles
    int64_t tpc = c->opt_chunk_tiles;
    if (tpc <= 0) {
        const int64_t target = (int64_t)c->sms * 24;          // one chunk per resident warp (3 CTAs of 8 warps per SM)
        tpc = (total + target * TEHMM_TILE - 1) / (target * TEHMM_TILE);
        tpc = std::max<int64_t>(4, std::min<int64_t>(tpc, 2048));
    }
    const int64_t L = tpc * TEHMM_TILE;
    // fine partition for the tile kernels: one 16-chunk tile per resident warp
    int64_t Lf = c->opt_fine_len;
    if (Lf <= 0) {
        const int64_t target = (int64_t)c->sms * tehmm_tile_warps() * 16;
        Lf = std::max<int64_t>(64, (total + target - 1) / target);
    }
    std::vector<TehmmChunk> chunks, fchunks;
    std::vector<int64_t> seq_chunk0(nseq + 1), seq_fchunk0(nseq + 1);
    int64_t tile_base = 0;
    for (int64_t s = 0; s < nseq; ++s) {
        seq_chunk0[s] = (int64_t)chunks.size();
        seq_fchunk0[s] = (int64_t)fchunks.size();
        const int64_t s0 = h_offsets[s], s1 = h_offsets[s + 1];
        for (int64_t t0 = s0; t0 < s1; t0 += L) {
            TehmmChunk ch;
            ch.t0 = t0; ch.t1 = std::min(s1, t0 + L); ch.s0 = s0; ch.s1 = s1;
            ch.seq = (int32_t)s;
            ch.ntiles = (int32_t)((ch.t1 - ch.t0 + TEHMM_TILE - 1) / TEHMM_TILE);
            ch.tile0 = tile_base;
            tile_base += ch.ntiles;
            chunks.push_back(ch);
        }
        for (int64_t t0 = s0; t0 < s1; t0 += Lf) {
            TehmmChunk ch;
            ch.t0 = t0; ch.t1 = std::min(s1, t0 + Lf); ch.s0 = s0; ch.s1 = s1;
            ch.seq = (int32_t)s;
            ch.ntiles = 0; ch.tile0 = 0;
            fchunks.push_back(ch);
        }
    }
    seq_chunk0[nseq] = (int64_t)chunks.size();
    seq_fchunk0[nseq] = (int64_t)fchunks.size();
    const int64_t nchunks = (int64_t)chunks.size(), nfchunks = (int64_t)fchunks.size();
    size_t o_off = 0, o_sc = align_up(o_off + (size_t)(nseq + 1) * 8), o_ch = align_up(o_sc + (size_t)(nseq + 1) * 8);
    size_t o_fsc = align_up(o_ch + (size_t)nchunks * sizeof(TehmmChunk));
    size_t o_fch = align_up(o_fsc + (size_t)(nseq + 1) * 8);
    size_t bytes = align_up(o_fch + (size_t)nfchunks * sizeof(TehmmChunk));
    std::vector<unsigned char> h(bytes, 0);
    memcpy(&h[o_off], h_offsets, (size_t)(nseq + 1) * 8);
    memcpy(&h[o_sc], seq_chunk0.data(), (size_t)(nseq + 1) * 8);
    memcpy(&h[o_ch], chunks.data(), (size_t)nchunks * sizeof(TehmmChunk));
    memcpy(&h[o_fsc], seq_fchunk0.data(), (size_t)(nseq + 1) * 8);
    memcpy(&h[o_fch], fchunks.data(), (size_t)nfchunks * sizeof(TehmmChunk));
    CU(cudaStreamSynchronize(c->stream));
    if (bytes > c->batch_blob_bytes) {
        if (c->batch_blob) { cudaFree(c->batch_blob); c->batch_blob = nullptr; c->batch_blob_bytes = 0; }
        CU(cudaMalloc(&c->batch_blob, bytes + bytes / 4));
        c->batch_blob_bytes = bytes + bytes / 4;
    }
    CU(cudaMemcpy(c->batch_blob, h.data(), bytes, cudaMemcpyHostToDevice));
    if (nseq > c->seq_flag_n) {
        if (c->d_seq_flag) { cudaFree(c->d_seq_flag); c->d_seq_flag = nullptr; c->seq_flag_n = 0; }
        CU(cudaMalloc((void **)&c->d_seq_flag, sizeof(int) * (size_t)(nseq + nseq / 4 + 1)));
        c->seq_flag_n = nseq + nseq / 4 + 1;
    }
    unsigned char *d = (unsigned char *)c->batch_blob;
    TehmmBatchDev &b = c->b;
    b.obs = d_obs; b.obs_bytes = obs_bytes; b.nseq = nseq; b.total = total;
    b.nchunks = nchunks; b.ntiles = tile_base;
    b.seq_off = (const int64_t *)(d + o_off); b.seq_chunk0 = (const int64_t *)(d + o_sc);
    b.chunks = (const TehmmChunk *)(d + o_ch);
    b.warmup = (int)(c->opt_warmup > 0 ? c->opt_warmup : 64);
    b.cont = nullptr;
    c->bf = b;
    c->bf.nchunks = nfchunks;
    c->bf.seq_chunk0 = (const int64_t *)(d + o_fsc);
    c->bf.chunks = (const TehmmChunk *)(d + o_fch);
    c->max_tiles_per_chunk = tpc;
    c->fine_len = Lf;
    c->has_batch = true;
    return TEHMM_OK;
}

int64_t tehmm_batch_total(tehmm_ctx *c) { return c && c->has_batch ? c->b.total : 0; }
int tehmm_ctx_device(tehmm_ctx *c) { return c ? c->device : -1; }
int tehmm_model_dims(tehmm_ctx *c, int *N, int *K, int *S)
{
    if (!c) return fail(TEHMM_EINVAL, "ctx is NULL");
    if (!c->has_model) return fail(TEHMM_ESTATE, "tehmm_set_model has not been called");
    if (N) *N = c->m.N;
    if (K) *K = c->m.K;
    if (S) *S = c->m.S;
    return TEHMM_OK;
}
int tehmm_lattice_stride(tehmm_ctx *c) { return c && c->has_model ? c->m.LD : 0; }
int64_t tehmm_batch_chunks(tehmm_ctx *c) { return c && c->has_batch ? c->b.nchunks : 0; }
int64_t tehmm_viterbi_workspace_bytes(tehmm_ctx *c, int prec)
{
    if (!c || !c->has_batch || !c->has_model) return 0;
    return c->b.total * (int64_t)c->m.LD * (prec == TEHMM_F32 ? 4 : 8);   // the delta lattice
}

// scratch carving shared by tehmm_scratch_bytes and the run_* entry points
struct Scratch {
    size_t start_vec, end_vec, cscale, part_a, bad, nbad, xi, xdiag, gamma0, tilemap, cmap, chunk_end, hist, total;
    int nparts;
};
static Scratch carve(const tehmm_ctx *c, int prec)
{
    const size_t ts = prec == TEHMM_F32 ? 4 : 8;
    const size_t NP = (size_t)c->m.NP, nc = (size_t)c->b.nchunks;
    const size_t nb = (size_t)std::max(c->b.nchunks, c->bf.nchunks);   // either partition
    Scratch s;
    size_t o = 0;
    s.start_vec = o; o = align_up(o + nb * NP * ts);
    s.end_vec = o; o = align_up(o + nb * NP * ts);
    s.cscale = o; o = align_up(o + nb * 8);
    s.part_a = o; o = align_up(o + nb * 8);
    s.bad = o; o = align_up(o + nb * 4);
    s.nbad = o; o = align_up(o + 4);
    s.xi = o; o = align_up(o + std::max(nc * NP * NP * ts, tehmm_xi_mma_scratch_bytes(c->sms)));
    s.xdiag = o; o = align_up(o + nc * NP * ts);
    s.gamma0 = o; o = align_up(o + (size_t)c->b.nseq * NP * ts);
    s.tilemap = o; o = align_up(o + (size_t)c->b.ntiles * NP);
    s.cmap = o; o = align_up(o + std::max(nc * NP, 3 * nb));
    s.chunk_end = o; o = align_up(o + nc);
    const size_t smem = tehmm_stats_smem_bytes(c->m.tab_rows, c->m.N, c->m.K, prec);
    s.nparts = 0;
    if (smem <= 200 * 1024) {
        int per_sm = smem <= 100 * 1024 ? 2 : 1;
        int64_t want = (int64_t)c->sms * per_sm;
        int64_t cap = (c->b.total + 255) / 256;     // at least 256 steps per CTA
        s.nparts = (int)std::max<int64_t>(1, std::min(want, cap));
    }
    s.hist = o; o = align_up(o + (size_t)s.nparts * std::max(c->m.tab_rows, c->m.srows) * c->m.N * 8 + 16);   // + the ratio cap (stats.cu)
    s.total = o;
    return s;
}

int64_t tehmm_scratch_bytes(tehmm_ctx *c, int prec)
{
    if (!c || !c->has_batch || !c->has_model) return 0;
    return (int64_t)carve(c, prec).total;
}

#define RUN_PROLOGUE()                                                                  \
    if (!c) return fail(TEHMM_EINVAL, "ctx is NULL");                                   \
    if (!c->has_model) return fail(TEHMM_ESTATE, "tehmm_set_model has not been called");\
    if (!c->has_batch) return fail(TEHMM_ESTATE, "tehmm_set_batch has not been called");\
    if (prec != TEHMM_F32 && prec != TEHMM_F64) return fail(TEHMM_EINVAL, "bad prec");  \
    CU(cudaSetDevice(c->device));                                                       \
    cudaStream_t st = c->stream

static int scan_grid(const tehmm_ctx *c)
{
    int64_t need = (c->b.nchunks + TEHMM_WARPS_PER_CTA - 1) / TEHMM_WARPS_PER_CTA;
    int64_t cap = (int64_t)c->sms * 3;      // resident CTAs of the scan kernels (80 registers, 8 warps)
    return (int)std::max<int64_t>(1, std::min(need, cap));
}

// timing brackets (no-ops unless the "timing" option is set)
static void tk_begin(tehmm_ctx *c, int which)
{
    if (!c->opt_timing) return;
    const int r = c->ev_n[which] % TEHMM_TRING;
    if (!c->ev[which][r][0]) { cudaEventCreate(&c->ev[which][r][0]); cudaEventCreate(&c->ev[which][r][1]); }
    cudaEventRecord(c->ev[which][r][0], c->stream);
}
static void tk_end(tehmm_ctx *c, int which)
{
    if (!c->opt_timing) return;
    cudaEventRecord(c->ev[which][c->ev_n[which] % TEHMM_TRING][1], c->stream);
    c->ev_n[which] += 1;
}

static int read_nbad(tehmm_ctx *c, const int *d_nbad, int *out, bool may_defer = true)
{
    if (may_defer && c->opt_defer && c->npending < TEHMM_NPENDING) {
        // optimistic: the count travels to a pinned slot behind the kernels already queued and
        // the caller carries on as if nothing had to be repaired; tehmm_ctx_check tells
        CU(cudaMemcpyAsync(c->h_pending + c->npending, d_nbad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        c->npending += 1;
        *out = 0;
        return TEHMM_OK;
    }
    CU(cudaMemcpyAsync(c->h_nbad, d_nbad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    *out = *c->h_nbad;
    return TEHMM_OK;
}

// Deferred verification (option "defer"): waits for the stream and returns in *unverified the
// number of chunks whose speculated boundary failed verification in any pass run since the last
// check.  0: every result produced since then stands.  > 0: those results must be recomputed
// with the option off (the synchronous verify / repair loop); nothing else is invalidated.
// When something was deferred, the check also moves the context's back-off: a refusal doubles the
// penalty (4 .. 256) and leaves "defer" off for that many requests (set_option counts "defer_skip"
// down), a check that stands halves it -- a refused attempt costs its stages twice, and a model /
// batch that needed repairs tends to need them again.
int tehmm_ctx_check(tehmm_ctx *c, int64_t *unverified)
{
    if (!c || !unverified) return fail(TEHMM_EINVAL, "NULL argument");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    int64_t n = 0;
    for (int i = 0; i < c->npending; ++i) n += c->h_pending[i];
    if (n > 0) {
        c->defer_penalty = std::min<int64_t>(256, std::max<int64_t>(4, 2 * c->defer_penalty));
        c->defer_skip = c->defer_penalty;
    } else if (c->npending > 0) {
        c->defer_penalty /= 2;
    }
    c->stat_deferred_checks += c->npending;
    c->stat_deferred_bad += n;
    c->npending = 0;
    *unverified = n;
    return TEHMM_OK;
}

int tehmm_run_emission(tehmm_ctx *c, int prec, const double *d_ratios, void *d_elog, void *d_blin,
                       double *d_rowmax)
{
    RUN_PROLOGUE();
    if (!d_rowmax || (!d_elog && !d_blin)) return fail(TEHMM_EINVAL, "need d_rowmax and at least one of d_elog / d_blin");
    cudaError_t e;
    tk_begin(c, TK_EMISSION);
    int n = tehmm_launch_emission(st, c->m, c->b, prec, d_ratios, d_elog, d_blin, d_rowmax, nullptr, c->d_seq_flag, c->sms, &e, 0, c->b.total);
    tk_end(c, TK_EMISSION);
    if (n < 0) return fail(TEHMM_ECUDA, "emission launch failed: %s", cudaGetErrorString(e));
    c->launches += n;
    return TEHMM_OK;
}

int tehmm_emission_rows_supported(tehmm_ctx *c, int prec)
{
    return c && c->has_model && tehmm_emission_rows_ok(c->m, prec, nullptr) ? 1 : 0;
}

int tehmm_run_emission_rows(tehmm_ctx *c, int prec, const double *d_ratios, void *d_elog, void *d_blin,
                            double *d_rowmax, int64_t row0, int64_t row1, uint64_t stream)
{
    RUN_PROLOGUE();
    if (!d_rowmax || (!d_elog && !d_blin)) return fail(TEHMM_EINVAL, "need d_rowmax and at least one of d_elog / d_blin");
    if (row0 < 0 || row1 > c->b.total || row0 >= row1 || (row0 & 31)) return fail(TEHMM_EINVAL, "bad row range [%lld,%lld) (row0 must be a multiple of 32)", (long long)row0, (long long)row1);
    if (!tehmm_emission_rows_ok(c->m, prec, d_ratios)) return fail(TEHMM_ESTATE, "this model / precision cannot run the emission in pieces (tehmm_emission_rows_supported)");
    if (stream != UINT64_MAX) st = (cudaStream_t)(uintptr_t)stream;
    cudaError_t e;
    int n = tehmm_launch_emission(st, c->m, c->b, prec, d_ratios, d_elog, d_blin, d_rowmax, nullptr, c->d_seq_flag, c->sms, &e, row0, row1);
    if (n < 0) return fail(TEHMM_ECUDA, "emission launch failed: %s", cudaGetErrorString(e));
    c->launches += n;
    return TEHMM_OK;
}

int tehmm_run_emission_f64(tehmm_ctx *c, const double *d_ratios, double *d_frame)
{
    int prec = TEHMM_F64;
    RUN_PROLOGUE();
    if (!d_frame) return fail(TEHMM_EINVAL, "d_frame is NULL");
    cudaError_t e;
    int n = tehmm_launch_emission(st, c->m, c->b, prec, d_ratios, nullptr, nullptr, nullptr, d_frame, c->d_seq_flag, c->sms, &e, 0, c->b.total);
    if (n < 0) return fail(TEHMM_ECUDA, "emission launch failed: %s", cudaGetErrorString(e));
    c->launches += n;
    return TEHMM_OK;
}

// verification tolerance: spread of component ratios (linear space) or of
// component differences (log space); see verify_kernel
static double tolerance(int prec, bool log_space)
{
    if (log_space) return prec == TEHMM_F32 ? 1e-5 : 1e-11;
    return prec == TEHMM_F32 ? 4e-6 : 1e-12;
}

// The warm-up length adapts: if more than 2% of the chunks of a pass had to be
// repaired, later passes of this context speculate twice as far back.
static void adapt_warmup(tehmm_ctx *c, int first_pass_bad, int64_t nchunks)
{
    if (c->opt_warmup > 0) return;
    // (capped: beyond a few hundred steps a longer warm-up costs more than resolving the flagged chunks
    //  exactly, resolve_flagged below)
    if ((int64_t)first_pass_bad * 50 > nchunks && c->b.warmup < 256) {
        c->b.warmup *= 2;
        c->bf.warmup = c->b.warmup;
    }
}

// ---------------------------------------------------------------- exact resolution of flagged chunks
// (fallback.cu)  The chunks flagged in `bad` get the boundary vector the serial recursion would hand
// them: transfer operators of the flagged chunks on the device, the chain over each run of flagged
// chunks on the host in float64, the vectors written into start_vec.  The caller re-runs the flagged
// chunks (mode 1).  kind 0 forward / 1 backward (linear space, lat = blin), 2 Viterbi (log space,
// lat = elog).  Blocks the stream; this is the slow path.
static int resolve_flagged(tehmm_ctx *c, cudaStream_t st, const TehmmBatchDev &PB, int prec, int kind,
                           const void *lat, void *sv, const void *ev, int *bad, int64_t reach)
{
    // A chunk that is NOT flagged agrees with what its neighbour handed it -- which proves it right only
    // if everything further up the recursion is right.  Downstream of a flagged chunk the standing chunks
    // are usually consistent with the WRONG vector (inside an uninformative stretch they all converged to
    // the same stable guess), so the chain also runs through `reach` chunks beyond every flagged one and
    // those are re-run as well; the verification after the re-run flags the next chunk if the truth has
    // not met the guess yet, and the caller comes back with four times the reach.
    const int N = c->m.N, NP = c->m.NP;
    const int dir = kind == 1 ? -1 : +1;
    const size_t ts = prec == TEHMM_F32 ? 4 : 8;
    const int64_t nch = PB.nchunks;
    std::vector<int> hb(nch);
    std::vector<TehmmChunk> hch(nch);
    CU(cudaMemcpyAsync(hb.data(), bad, sizeof(int) * (size_t)nch, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hch.data(), PB.chunks, sizeof(TehmmChunk) * (size_t)nch, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    std::vector<char> want(nch, 0);
    int64_t nflag = 0;
    for (int64_t i = 0; i < nch; ++i) {
        if (!hb[i]) continue;
        nflag += 1;
        want[i] = 1;
        int64_t j = i;
        for (int64_t g = 1; g <= reach; ++g) {
            if (dir > 0 ? hch[j].t1 >= hch[j].s1 : hch[j].t0 <= hch[j].s0) break;    // end of the sequence
            j += dir;
            want[j] = 1;
        }
    }
    if (nflag == 0) return TEHMM_OK;
    // chain order, run after run (a run = consecutive wanted chunks of one sequence; its first chunk is
    // flagged, so it has a neighbour on the side the recursion comes from)
    std::vector<int64_t> list, run_off;
    for (int64_t q = 0; q < nch; ++q) {
        const int64_t i = dir > 0 ? q : nch - 1 - q;
        if (!want[i]) continue;
        const int64_t p = i - dir;
        const bool linked = p >= 0 && p < nch && want[p] && hch[p].seq == hch[i].seq;
        if (!linked) run_off.push_back((int64_t)list.size());
        list.push_back(i);
        hb[i] = 1;
    }
    const int64_t B = (int64_t)list.size(), nruns = (int64_t)run_off.size();
    run_off.push_back(B);
    DevBuf d_list, d_run, d_end, d_scale;
    CU(d_list.alloc((size_t)B * 8)); CU(d_run.alloc((size_t)(nruns + 1) * 8));
    CU(d_end.alloc((size_t)B * N * NP * ts)); CU(d_scale.alloc((size_t)B * N * 8));
    CU(cudaMemcpyAsync(d_list.p, list.data(), (size_t)B * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_run.p, run_off.data(), (size_t)(nruns + 1) * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(bad, hb.data(), sizeof(int) * (size_t)nch, cudaMemcpyHostToDevice, st));
    CU(tehmm_launch_transfer_ops(st, c->m, PB.chunks, d_list.as<int64_t>(), B, prec, kind, lat, d_end.p, d_scale.as<double>(), c->sms));
    CU(tehmm_launch_chain(st, c->m, prec, kind, dir, d_list.as<int64_t>(), d_run.as<int64_t>(), nruns, d_end.p, d_scale.as<double>(), ev, sv));
    c->launches += 2;
    CU(cudaStreamSynchronize(st));     // the temporaries go out of scope
    c->stat_fallbacks += 1;
    c->stat_fallback_chunks += B;
    return TEHMM_OK;
}

// The same for the traceback: a flagged chunk assumed the wrong end state.  Its walk is a MAP from end
// state to the state it implies for the left neighbour; N walks per chunk (the ordinary kernel on a list
// of virtual chunks, forced end = each state), the maps composed right to left on the host.  Unlike the
// vector recursions the standing chunks to the LEFT of a flagged one are usually wrong too, consistently
// (inside an uninformative stretch every walk stays in the state it entered with), so the maps are also
// computed for `reach` chunks to the left of every flagged chunk and the chain runs on for as long as it
// contradicts what those chunks assumed; `reach` grows fourfold per round.  Integer work: the result is
// exactly the serial traceback's.
static int resolve_flagged_tb(tehmm_ctx *c, cudaStream_t st, const TehmmBatchDev &TBP, int prec,
                              const void *d_lattice, uint8_t *states, uint8_t *spec_end, const uint8_t *pred,
                              uint8_t *forced, int *bad, int tb_grid, int64_t reach)
{
    const int N = c->m.N;
    const int64_t nch = TBP.nchunks;
    std::vector<int> hb(nch);
    std::vector<TehmmChunk> hch(nch);
    std::vector<uint8_t> hpred(nch), hspec(nch), hforced(nch);
    CU(cudaMemcpyAsync(hb.data(), bad, sizeof(int) * (size_t)nch, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hch.data(), TBP.chunks, sizeof(TehmmChunk) * (size_t)nch, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hpred.data(), pred, (size_t)nch, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hspec.data(), spec_end, (size_t)nch, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hforced.data(), forced, (size_t)nch, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    // chunks whose maps are needed: the flagged ones and up to `reach` chunks to the left of each, inside
    // the same sequence (a chunk without a left neighbour ends the chain: nobody consumes its pred)
    std::vector<char> want(nch, 0);
    int64_t nflag = 0;
    for (int64_t i = nch - 1; i >= 0; --i) {
        if (!hb[i]) continue;
        nflag += 1;
        want[i] = 1;
        for (int64_t g = 1, j = i; g <= reach && hch[j].t0 > hch[j].s0; ++g) { j -= 1; want[j] = 1; }
    }
    if (nflag == 0) return TEHMM_OK;
    std::vector<int64_t> list;                     // ascending
    std::vector<int64_t> slot(nch, -1);
    for (int64_t i = 0; i < nch; ++i) if (want[i]) { slot[i] = (int64_t)list.size(); list.push_back(i); }
    const int64_t B = (int64_t)list.size(), nv = B * N;
    std::vector<TehmmChunk> v((size_t)nv);
    std::vector<uint8_t> vf((size_t)nv);
    std::vector<int> vb((size_t)nv, 1);
    for (int64_t k = 0; k < B; ++k)
        for (int i = 0; i < N; ++i) { v[(size_t)(k * N + i)] = hch[list[k]]; vf[(size_t)(k * N + i)] = (uint8_t)i; }
    DevBuf d_v, d_vf, d_vb, d_vs, d_vp;
    CU(d_v.alloc(v.size() * sizeof(TehmmChunk))); CU(d_vf.alloc((size_t)nv)); CU(d_vb.alloc((size_t)nv * 4));
    CU(d_vs.alloc((size_t)nv)); CU(d_vp.alloc((size_t)nv));
    CU(cudaMemcpyAsync(d_v.p, v.data(), v.size() * sizeof(TehmmChunk), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_vf.p, vf.data(), (size_t)nv, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_vb.p, vb.data(), (size_t)nv * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(d_vp.p, 0, (size_t)nv, st));
    TehmmBatchDev VB = TBP;
    VB.nchunks = nv;
    VB.chunks = d_v.as<TehmmChunk>();
    const int vgrid = (int)std::max<int64_t>(1, std::min<int64_t>((nv + TEHMM_WARPS_PER_CTA - 1) / TEHMM_WARPS_PER_CTA, (int64_t)tb_grid));
    // (the walks scribble over these chunks' rows of `states`; every chunk whose map was computed is re-run below)
    CU(tehmm_launch_traceback(st, c->m, VB, prec, d_lattice, nullptr, states, nullptr, d_vs.as<uint8_t>(), d_vp.as<uint8_t>(),
                              d_vf.as<uint8_t>(), d_vb.as<int>(), 1, vgrid));
    c->launches += 1;
    std::vector<uint8_t> vp((size_t)nv);
    CU(cudaMemcpyAsync(vp.data(), d_vp.p, (size_t)nv, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    // right to left: `have` = the chain holds the true state at t0 - 1 of chunk i + 1 in `cur`
    bool have = false;
    int cur = 0;
    for (int64_t i = nch - 1; i >= 0; --i) {
        if (!want[i]) { have = false; continue; }
        const bool seq_end = hch[i].t1 == hch[i].s1;
        int end;
        if (seq_end) { have = false; end = (int)hspec[i]; }                   // exact by construction (never flagged)
        else if (have) end = cur;
        else end = hb[i] ? (int)hpred[i + 1] : (int)hspec[i];                  // the right neighbour stands
        // every chunk whose rows were scribbled over is re-run from the end state the chain gives it
        // (the one it had, where the chain agrees with it)
        hb[i] = 1;
        hforced[i] = hspec[i] = (uint8_t)end;
        cur = end < N ? (int)vp[(size_t)(slot[i] * N + end)] : 0;
        have = true;
    }
    CU(cudaMemcpyAsync(forced, hforced.data(), (size_t)nch, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(spec_end, hspec.data(), (size_t)nch, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(bad, hb.data(), sizeof(int) * (size_t)nch, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    c->stat_fallbacks += 1;
    c->stat_fallback_chunks += B;
    return TEHMM_OK;
}

// Tolerance of the verifications that follow an exact resolution.  The chained vector and the vector the
// re-run neighbour ends on are two roundings of the same quantity, and a filter's rounding noise (eps per
// step: 2^-21 for the 3 x TF32 products, 2^-52 in float64) is amplified by 1 / (1 - rho) where the data
// do not help (rho = |lambda_2| of the transition matrix): what is left after a resolution is compared
// against that floor, not against the band a speculated boundary has to meet.
static double tolerance_after_fallback(const tehmm_ctx *c, int prec, bool log_space)
{
    const double base = 100.0 * tolerance(prec, log_space);
    if (log_space) return base;
    const double eps = prec == TEHMM_F32 ? 4.8e-7 : 2.3e-16;
    const double floor_ = 8.0 * eps / std::max(1e-9, 1.0 - mix_rho_of(const_cast<tehmm_ctx *>(c)));
    return std::min(0.1, std::max(base, floor_));
}
#define TEHMM_MAX_FALLBACK_ROUNDS 10    // reach 8 * 4^round chunks: far beyond any partition; then the plain loop

// The speculate / verify / repair loop of the forward (kind 0), backward (1) and Viterbi DP (2) passes over the
// chunks of partition PB: the first pass (timed), then verify -> repair until every chunk boundary stands.
// launch(mode) runs the pass (mode 0: every chunk, speculated starts; mode 1: the flagged chunks from start_vec).
// kind, lat and the exact fallback are resolve_flagged's (linear space for 0 / 1, log space for 2); lkap: the
// forward pass's per-chunk log factors (verify_kernel).  The fallback needs a chain without segment ratios.
// umma_used (forward / backward): raised by launch when the tcgen05 kernel took the first pass -- its fault flag
// is checked after that pass and its verification count is never deferred.
}   // extern "C" (a template below)
template <typename Launch>
static int repair_loop(tehmm_ctx *c, cudaStream_t st, const TehmmBatchDev &PB, int prec, int kind, const void *lat,
                       void *sv, void *ev, int *bad, int *nbad, double *lkap, bool fallback_ok,
                       const bool *umma_used, Launch launch)
{
    static const int timer[3] = {TK_FORWARD, TK_BACKWARD, TK_VITERBI_DP};
    static const char *const what[3] = {"forward", "backward", "viterbi"};
    static const char *const umma_kernel[3] = {"fwd_umma_kernel", "bwd_umma_kernel", ""};
    int64_t *const stat_repair[3] = {&c->stat_repair_fwd, &c->stat_repair_bwd, &c->stat_repair_vit};
    int64_t *const stat_bad[3] = {&c->stat_bad_fwd, &c->stat_bad_bwd, &c->stat_bad_vit};
    const bool log_space = kind == 2;
    tk_begin(c, timer[kind]);
    CU(launch(0));
    tk_end(c, timer[kind]);
    c->launches += 1;
    const int64_t n_entry = kind == 0 ? c->n_entry : kind == 2 ? c->n_ventry : 0;
    if (n_entry > 0) {
        // continued sequences (tehmm_set_boundary / tehmm_set_viterbi_boundary): their first chunks are exact
        // from the entry vectors, run like repaired chunks; the verification below then checks the chunks after
        // them as usual (a first chunk is never flagged, so the exact fallback chains from its end vector)
        CU(tehmm_launch_entry(st, PB, prec, c->m.NP, n_entry, kind == 0 ? c->d_entry_seq : c->d_ventry_seq,
                              kind == 0 ? c->d_entry_vec : c->d_ventry_vec, sv, bad));
        CU(launch(1));
        c->launches += 2;
    }
    const bool umma = umma_used && *umma_used;
    double tol = tolerance(prec, log_space);
    const int64_t max_pass = c->opt_max_repair > 0 ? c->opt_max_repair : PB.nchunks + 1;
    int fb_rounds = 0;
    for (int64_t pass = 0;; ++pass) {
        CU(tehmm_launch_verify(st, PB, prec, c->m.NP, sv, ev, tol, kind == 1 ? -1 : +1, log_space ? 0 : 1, bad, nbad, lkap));
        c->launches += 1;
        int nb = 0;
        if (umma && pass == 0) CU(cudaMemcpyAsync(c->h_nbad + 1, c->d_fault, sizeof(int), cudaMemcpyDeviceToHost, st));
        if (read_nbad(c, nbad, &nb, !umma)) return TEHMM_ECUDA;
        if (umma && pass == 0 && c->h_nbad[1]) {
            CU(cudaMemsetAsync(c->d_fault, 0, sizeof(int), st));
            return fail(TEHMM_ECUDA, "%s: a barrier wait timed out (tensor-memory protocol fault)", umma_kernel[kind]);
        }
        if (pass == 0) adapt_warmup(c, nb, PB.nchunks);
        if (nb == 0) break;
        if (pass >= max_pass) return fail(TEHMM_ESTATE, "%s repair did not converge (%d chunks left)", what[kind], nb);
        if (c->opt_fallback_after >= 0 && pass >= c->opt_fallback_after && fallback_ok && fb_rounds < TEHMM_MAX_FALLBACK_ROUNDS) {
            // slow mixing: resolve the flagged chunks exactly (transfer operators + chain) instead of one link per pass
            if (resolve_flagged(c, st, PB, prec, kind, lat, sv, ev, bad, (int64_t)8 << (2 * fb_rounds))) return TEHMM_ECUDA;
            tol = tolerance_after_fallback(c, prec, log_space);
            fb_rounds += 1;
        }
        *stat_repair[kind] += 1; *stat_bad[kind] += nb;
        CU(launch(1));
        c->launches += 1;
    }
    return TEHMM_OK;
}
extern "C" {

// fp32 without segment ratios, unless option "tile" is 0: the mma.sync tile kernels (tile.cu) at <= 32 states,
// the tcgen05 kernels (umma.cu) for the first pass over a single-sequence batch at 33..64 states
static bool use_tile(const tehmm_ctx *c, int prec, const double *d_ratios)
{
    return c->opt_tile != 0 && prec == TEHMM_F32 && c->m.NS == 1 && d_ratios == nullptr;
}
static bool use_umma(const tehmm_ctx *c, int prec, const double *d_ratios)
{
    return c->opt_tile != 0 && prec == TEHMM_F32 && c->m.NS == 2 && d_ratios == nullptr && c->b.nseq == 1;
}

int tehmm_run_forward(tehmm_ctx *c, int prec, const void *d_blin, const double *d_rowmax,
                      const double *d_ratios, void *d_alpha, double *d_logprob, void *d_scratch)
{
    RUN_PROLOGUE();
    if (!d_blin || !d_rowmax || !d_logprob || !d_scratch) return fail(TEHMM_EINVAL, "NULL argument");
    const Scratch s = carve(c, prec);
    char *w = (char *)d_scratch;
    void *sv = w + s.start_vec, *ev = w + s.end_vec;
    double *cs = (double *)(w + s.cscale), *lkap = (double *)(w + s.part_a);
    int *bad = (int *)(w + s.bad), *nbad = (int *)(w + s.nbad);
    const int grid = scan_grid(c);
    const bool tile = use_tile(c, prec, d_ratios);
    // 33..64 states: the tcgen05 kernel (csrc/umma.cu, M128 N64 K8 tf32, state and accumulator in tensor memory,
    // transition matrix in shared memory) takes the first pass over a single-sequence batch on the fine
    // partition; repairs and everything else stay with the one-chunk-per-warp kernel
    const bool wide_umma = use_umma(c, prec, d_ratios);
    const TehmmBatchDev &PB = (tile || wide_umma) ? c->bf : c->b;       // the partition this pass runs on
    bool umma_used = false;
    auto launch = [&](int mode) -> cudaError_t {
        if (wide_umma && tehmm_forward_umma_ok(c->m, PB, mode, c->fine_len)) {
            cudaError_t eu = tehmm_launch_forward_umma(st, c->m, PB, (const float *)d_blin, d_rowmax, (float *)d_alpha,
                                                       (float *)sv, (float *)ev, cs, c->sms, c->fine_len, c->d_fault);
            if (eu == cudaSuccess) { c->stat_umma_passes += 1; umma_used = true; return eu; }
            if (eu != cudaErrorNotSupported) return eu;
            cudaGetLastError();          // no tensor map: the one-chunk-per-warp kernel below
        }
        if (tile) {
            c->stat_tile_passes += 1;
            return tehmm_launch_forward_tile(st, c->m, PB, (const float *)d_blin, d_rowmax, (float *)d_alpha, (float *)sv, (float *)ev, cs, bad, mode, c->sms, c->fine_len);
        }
        return tehmm_launch_forward(st, c->m, PB, prec, d_blin, d_rowmax, d_ratios, d_alpha, sv, ev, cs, bad, mode, grid);
    };
    if (int rc = repair_loop(c, st, PB, prec, 0, d_blin, sv, ev, bad, nbad, lkap, d_ratios == nullptr, &umma_used, launch)) return rc;
    CU(tehmm_launch_forward_logprob(st, PB, prec, c->m.NP, ev, cs, lkap, d_logprob));
    c->launches += 1;
    return TEHMM_OK;
}

int tehmm_run_backward(tehmm_ctx *c, int prec, int flags, const void *d_blin, const void *d_alpha,
                       const double *d_ratios, void *d_post, uint8_t *d_map_states,
                       double *d_map_score, double *d_start_trans, void *d_scratch)
{
    RUN_PROLOGUE();
    if (!d_blin || !d_alpha || !d_scratch) return fail(TEHMM_EINVAL, "NULL argument");
    if ((flags & TEHMM_BWD_POSTERIORS) && !d_post) return fail(TEHMM_EINVAL, "POSTERIORS needs d_post");
    if ((flags & TEHMM_BWD_MAP) && (!d_map_states || !d_map_score)) return fail(TEHMM_EINVAL, "MAP needs d_map_states and d_map_score");
    if ((flags & TEHMM_BWD_TRANS) && !d_start_trans) return fail(TEHMM_EINVAL, "TRANS needs d_start_trans");
    // the in-kernel diagonal count of unfolded ratios treats every sequence's first row as a start; a continued
    // sequence's first row is not one: such batches fold the ratios and count them with tehmm_ratio_diag_counts
    if ((flags & TEHMM_BWD_TRANS) && d_ratios && c->n_entry > 0)
        return fail(TEHMM_EINVAL, "TRANS with unfolded segment ratios and entry vectors: fold the ratios (tehmm_fold_ratios) and use tehmm_ratio_diag_counts");
    const Scratch s = carve(c, prec);
    char *w = (char *)d_scratch;
    void *sv = w + s.start_vec, *ev = w + s.end_vec;
    double *mp = (double *)(w + s.part_a);
    int *bad = (int *)(w + s.bad), *nbad = (int *)(w + s.nbad);
    void *xi = w + s.xi, *xd = w + s.xdiag, *g0 = w + s.gamma0;
    const int grid = scan_grid(c);
    // Expected transition counts on the tensor-core path: posteriors from bwd_tile_kernel, then
    // xi_mma_kernel (two dense products per 16 steps).  Needs the posterior lattice, un-renormalised.
    const bool xi_mma = use_tile(c, prec, d_ratios) && (flags & TEHMM_BWD_TRANS) && (flags & TEHMM_BWD_POSTERIORS) &&
                         !(flags & TEHMM_BWD_RENORM_EPS);
    if (xi_mma) flags &= ~TEHMM_BWD_TRANS;
    const bool tile = use_tile(c, prec, d_ratios) && !(flags & TEHMM_BWD_TRANS);
    // 33..64 states, one sequence, no transition counts: the tcgen05 twin of the forward kernel (csrc/umma.cu) takes the
    // first pass on the fine partition; repairs stay with the one-chunk-per-warp kernel on the same partition
    const bool wide_umma = use_umma(c, prec, d_ratios) && !(flags & TEHMM_BWD_TRANS);
    const TehmmBatchDev &PB = (tile || wide_umma) ? c->bf : c->b;
    // exit vectors: the last rows of alpha and blin are scaled by A u until the end of the call (window.cu); the
    // guard queues their restore on every way out, so a failing launch below never leaves the caller's lattices changed
    struct ExitRows {
        tehmm_ctx *c = nullptr;
        cudaStream_t st;
        int prec;
        void *alpha, *blin;
        cudaError_t restore()
        {
            tehmm_ctx *cc = c;
            c = nullptr;
            if (!cc) return cudaSuccess;
            cc->launches += 1;
            return tehmm_launch_exit(st, cc->m, cc->b, prec, cc->n_exit, cc->d_exit_seq, cc->d_exit_vec, alpha, blin, cc->d_exit_save, 1);
        }
        ~ExitRows() { restore(); }
    } exit_rows;
    if (c->n_exit > 0) {
        CU(tehmm_launch_exit(st, c->m, c->b, prec, c->n_exit, c->d_exit_seq, c->d_exit_vec, const_cast<void *>(d_alpha),
                             const_cast<void *>(d_blin), c->d_exit_save, 0));
        c->launches += 1;
        exit_rows.c = c;
        exit_rows.st = st;
        exit_rows.prec = prec;
        exit_rows.alpha = const_cast<void *>(d_alpha);
        exit_rows.blin = const_cast<void *>(d_blin);
    }
    bool umma_used = false;
    auto launch = [&](int mode) -> cudaError_t {
        if (wide_umma && tehmm_backward_umma_ok(c->m, PB, flags, mode, c->fine_len)) {
            cudaError_t eu = tehmm_launch_backward_umma(st, c->m, PB, flags, (const float *)d_blin, (const float *)d_alpha, (float *)d_post,
                                                        d_map_states, mp, (float *)sv, (float *)ev, c->sms, c->fine_len, c->d_fault);
            if (eu == cudaSuccess) { c->stat_umma_passes += 1; umma_used = true; return eu; }
            if (eu != cudaErrorNotSupported) return eu;
            cudaGetLastError();
        }
        if (tile) {
            c->stat_tile_passes += 1;
            return tehmm_launch_backward_tile(st, c->m, PB, flags, (const float *)d_blin, (const float *)d_alpha, (float *)d_post, d_map_states, mp, (float *)sv, (float *)ev, bad, mode, c->sms);
        }
        return tehmm_launch_backward(st, c->m, PB, prec, flags, d_blin, d_alpha, d_ratios, d_post, d_map_states, mp, xi, xd, g0, sv, ev, bad, mode, grid);
    };
    if (int rc = repair_loop(c, st, PB, prec, 1, d_blin, sv, ev, bad, nbad, nullptr, d_ratios == nullptr, &umma_used, launch)) return rc;
    if (flags & TEHMM_BWD_MAP) { CU(tehmm_launch_map_reduce(st, PB, mp, d_map_score)); c->launches += 1; }
    if (flags & TEHMM_BWD_TRANS) { CU(tehmm_launch_trans_reduce(st, c->m, c->b, prec, xi, xd, g0, d_start_trans)); c->launches += 1; }
    if (xi_mma) {
        tk_begin(c, TK_XI);
        CU(tehmm_launch_xi_mma(st, c->m, c->bf, (const float *)d_alpha, (const float *)d_post, (double *)xi, (float *)g0, d_start_trans, c->sms));
        tk_end(c, TK_XI);
        c->launches += 2;
    }
    CU(exit_rows.restore());
    return TEHMM_OK;
}

int tehmm_fold_ratios(tehmm_ctx *c, int prec, const double *d_ratios, void *d_blin, double *d_rowmax)
{
    RUN_PROLOGUE();
    if (!d_ratios || !d_blin || !d_rowmax) return fail(TEHMM_EINVAL, "NULL argument");
    CU(tehmm_launch_ratio_fold(st, c->m, c->b.total, prec, d_ratios, d_blin, d_rowmax, c->sms));
    c->launches += 1;
    return TEHMM_OK;
}

int tehmm_ratio_diag_counts(tehmm_ctx *c, int prec, const void *d_post, const double *d_ratios,
                            double *d_start_trans, void *d_scratch)
{
    RUN_PROLOGUE();
    if (!d_post || !d_ratios || !d_start_trans || !d_scratch) return fail(TEHMM_EINVAL, "NULL argument");
    const Scratch s = carve(c, prec);
    double *part = (double *)((char *)d_scratch + s.xi);       // >= nchunks * NP * NP * ts bytes: room for nchunks * 64 doubles
    // one warp per chunk walks its rows one after the other: the fine partition (5x as many, 5x shorter) where it fits
    const size_t room = (size_t)c->b.nchunks * c->m.NP * c->m.NP * (prec == TEHMM_F32 ? 4 : 8);
    const TehmmBatchDev &PB = (size_t)c->bf.nchunks * 64 * 8 <= room ? c->bf : c->b;
    CU(tehmm_launch_ratio_diag(st, c->m, PB, prec, d_ratios, d_post, part, d_start_trans, c->sms));
    c->launches += 2;
    return TEHMM_OK;
}

int tehmm_run_emission_stats(tehmm_ctx *c, int prec, const void *d_post, const double *d_ratios,
                             double *d_obs_stats, int stats_S, void *d_scratch)
{
    RUN_PROLOGUE();
    if (!d_post || !d_obs_stats || !d_scratch) return fail(TEHMM_EINVAL, "NULL argument");
    if (stats_S <= 0) return fail(TEHMM_EINVAL, "stats_S must be positive");
    const Scratch s = carve(c, prec);
    double *part = (double *)((char *)d_scratch + s.hist);
    tk_begin(c, TK_STATS);
    CU(tehmm_launch_emission_stats(st, c->m, c->b, prec, d_post, d_ratios, d_obs_stats, part, s.nparts, stats_S));
    tk_end(c, TK_STATS);
    c->launches += s.nparts > 0 ? 2 * ((c->m.K + 31) / 32) : 1;
    return TEHMM_OK;
}

int tehmm_run_viterbi(tehmm_ctx *c, int prec, const void *d_elog, const double *d_rowmax,
                      const double *d_ratios_emission, const double *d_ratios_dp, void *d_lattice,
                      uint8_t *d_states, int64_t *d_states64, double *d_logprob, void *d_scratch)
{
    RUN_PROLOGUE();
    if (!d_elog || !d_lattice || !d_states || !d_logprob || !d_scratch) return fail(TEHMM_EINVAL, "NULL argument (d_states is required; d_states64 is optional)");
    const Scratch s = carve(c, prec);
    char *w = (char *)d_scratch;
    void *sv = w + s.start_vec, *ev = w + s.end_vec;
    double *sp = (double *)(w + s.part_a);
    int *bad = (int *)(w + s.bad), *nbad = (int *)(w + s.nbad);
    // the traceback is latency bound (one dependent arg-max per step): it walks the FINE partition,
    // five times as many chunks in flight, while the issue-bound DP keeps the coarse one
    const TehmmBatchDev &TBP = c->bf;
    uint8_t *spec_end = (uint8_t *)(w + s.cmap), *pred = spec_end + TBP.nchunks, *forced = pred + TBP.nchunks;
    const int grid = scan_grid(c);
    const int tb_grid = (int)std::max<int64_t>(1, std::min<int64_t>((TBP.nchunks + TEHMM_WARPS_PER_CTA - 1) / TEHMM_WARPS_PER_CTA, (int64_t)c->sms * 5));
    const int64_t max_pass = c->opt_max_repair > 0 ? c->opt_max_repair : c->b.nchunks + 1;
    // The log-probability: the DP's own value (sum of the row maxima it takes out, float64 across steps,
    // plus rowmax) where the lean fp32 kernel runs and the caller passed rowmax; otherwise -- float64
    // mode, segment ratios, more than 32 states, option "rescore" -- the float64 re-score of the path.
    const bool dp_score = d_rowmax != nullptr && c->opt_rescore == 0 && tehmm_viterbi_dp_scores(c->m, prec, d_ratios_dp);
    double *dsp = dp_score ? (double *)(w + s.cscale) : nullptr;
    // ---- DP: delta lattice, chunk starts speculated / verified / repaired
    auto launch = [&](int mode) -> cudaError_t {
        return tehmm_launch_viterbi(st, c->m, c->b, prec, d_elog, d_ratios_dp, d_lattice, sv, ev, bad, mode, grid, d_rowmax, dsp);
    };
    if (int rc = repair_loop(c, st, c->b, prec, 2, d_elog, sv, ev, bad, nbad, nullptr, d_ratios_dp == nullptr, nullptr, launch)) return rc;
    // ---- traceback: chunk end states speculated / verified / repaired
    CU(cudaMemsetAsync(bad, 0, sizeof(int) * (size_t)TBP.nchunks, st));
    tk_begin(c, TK_TRACEBACK);
    CU(tehmm_launch_traceback(st, c->m, TBP, prec, d_lattice, d_ratios_dp, d_states, d_states64, spec_end, pred, forced, bad, 0, tb_grid));
    tk_end(c, TK_TRACEBACK);
    c->launches += 1;
    if (c->n_vexit > 0) {
        // exit states (tehmm_set_viterbi_boundary): the last chunks of those sequences are walked again from
        // the forced state of their last row before the verification, which then checks the chunks to their
        // left against that walk; the exact fallback takes their end state as known (spec_end)
        CU(tehmm_launch_vit_exit(st, c->m, TBP, prec, d_lattice, c->n_vexit, c->d_vexit_seq, c->d_vexit_state,
                                 c->d_vexit_ratio, spec_end, forced, bad));
        CU(tehmm_launch_traceback(st, c->m, TBP, prec, d_lattice, d_ratios_dp, d_states, d_states64, spec_end, pred, forced, bad, 1, tb_grid));
        c->launches += 2;
    }
    int64_t tb_reach = 8;
    for (int64_t pass = 0;; ++pass) {
        CU(tehmm_launch_tb_verify(st, TBP, spec_end, pred, forced, bad, nbad));
        c->launches += 1;
        int nb = 0;
        if (read_nbad(c, nbad, &nb)) return TEHMM_ECUDA;
        if (pass == 0) adapt_warmup(c, nb, TBP.nchunks);
        if (nb == 0) break;
        if (pass >= TBP.nchunks + 1 && pass >= max_pass) return fail(TEHMM_ESTATE, "traceback repair did not converge (%d chunks left)", nb);
        if (c->opt_fallback_after >= 0 && pass >= c->opt_fallback_after && d_ratios_dp == nullptr && tb_reach < ((int64_t)1 << 40)) {
            if (resolve_flagged_tb(c, st, TBP, prec, d_lattice, d_states, spec_end, pred, forced, bad, tb_grid, tb_reach)) return TEHMM_ECUDA;
            tb_reach *= 4;
        }
        c->stat_repair_tb += 1; c->stat_bad_tb += nb;
        CU(tehmm_launch_traceback(st, c->m, TBP, prec, d_lattice, d_ratios_dp, d_states, d_states64, spec_end, pred, forced, bad, 1, tb_grid));
        c->launches += 1;
    }
    tk_begin(c, TK_RESCORE);
    if (dp_score) {
        CU(tehmm_launch_vit_score_reduce(st, c->b, dsp, d_logprob));
        c->launches += 1;
    } else {
        CU(tehmm_launch_rescore(st, c->m, TBP, d_states, d_ratios_emission, d_ratios_dp, sp, d_logprob, 0, TBP.total));   // latency bound too: fine partition
        c->launches += 2;
    }
    tk_end(c, TK_RESCORE);
    return TEHMM_OK;
}

int tehmm_path_score(tehmm_ctx *c, const uint8_t *d_states, const double *d_ratios_emission,
                     const double *d_ratios_dp, int64_t lo, int64_t hi, double *d_logprob, void *d_scratch)
{
    int prec = TEHMM_F32;
    RUN_PROLOGUE();
    if (!d_states || !d_logprob || !d_scratch) return fail(TEHMM_EINVAL, "NULL argument");
    if (lo < 0 || hi > c->b.total || lo > hi) return fail(TEHMM_EINVAL, "row range [%lld,%lld) outside the batch", (long long)lo, (long long)hi);
    const Scratch s = carve(c, prec);
    double *sp = (double *)((char *)d_scratch + s.part_a);
    CU(tehmm_launch_rescore(st, c->m, c->bf, d_states, d_ratios_emission, d_ratios_dp, sp, d_logprob, lo, hi));
    c->launches += 2;
    return TEHMM_OK;
}

// ---------------------------------------------------------------- windows of longer sequences (window.cu)
static int check_seqs(const char *what, int64_t n, const int64_t *seq, int64_t nseq, const std::vector<int64_t> &off)
{
    for (int64_t k = 0; k < n; ++k) {
        if (seq[k] < 0 || seq[k] >= nseq) return fail(TEHMM_EINVAL, "%s %lld: sequence %lld outside [0,%lld)", what, (long long)k, (long long)seq[k], (long long)nseq);
        if (k > 0 && seq[k] <= seq[k - 1]) return fail(TEHMM_EINVAL, "%s sequences must be increasing", what);
        if (off[seq[k] + 1] <= off[seq[k]]) return fail(TEHMM_EINVAL, "%s %lld: sequence %lld is empty", what, (long long)k, (long long)seq[k]);
    }
    return 0;
}

static int check_vectors(const char *what, int64_t n, const int64_t *seq, const double *vec, int64_t nseq, int N,
                         const std::vector<int64_t> &off)
{
    if (check_seqs(what, n, seq, nseq, off)) return TEHMM_EINVAL;
    for (int64_t k = 0; k < n; ++k) {
        double sum = 0.0;
        for (int j = 0; j < N; ++j) {
            const double x = vec[k * N + j];
            if (!(x >= 0.0) || !std::isfinite(x)) return fail(TEHMM_EINVAL, "%s %lld: component %d is %g (must be finite and >= 0)", what, (long long)k, j, x);
            sum += x;
        }
        if (!(sum > 0.0)) return fail(TEHMM_EINVAL, "%s %lld: the vector is zero", what, (long long)k);
    }
    return 0;
}

int tehmm_set_boundary(tehmm_ctx *c, int64_t n_entry, const int64_t *h_entry_seq, const double *h_entry_vec,
                       int64_t n_exit, const int64_t *h_exit_seq, const double *h_exit_vec)
{
    if (!c) return fail(TEHMM_EINVAL, "ctx is NULL");
    if (!c->has_model) return fail(TEHMM_ESTATE, "tehmm_set_model has not been called");
    if (!c->has_batch) return fail(TEHMM_ESTATE, "tehmm_set_batch has not been called");
    if (n_entry < 0 || n_exit < 0 || (n_entry > 0 && (!h_entry_seq || !h_entry_vec)) || (n_exit > 0 && (!h_exit_seq || !h_exit_vec)))
        return fail(TEHMM_EINVAL, "bad argument");
    CU(cudaSetDevice(c->device));
    const int64_t nseq = c->b.nseq;
    const int N = c->m.N, NP = c->m.NP;
    const std::vector<int64_t> off(c->batch_key.begin(), c->batch_key.begin() + nseq + 1);
    if (check_vectors("entry", n_entry, h_entry_seq, h_entry_vec, nseq, N, off)) return TEHMM_EINVAL;
    if (check_vectors("exit", n_exit, h_exit_seq, h_exit_vec, nseq, N, off)) return TEHMM_EINVAL;
    CU(cudaStreamSynchronize(c->stream));     // the passes queued so far read the vectors being replaced
    c->n_entry = c->n_exit = 0;
    c->b.cont = c->bf.cont = nullptr;
    if (n_entry == 0 && n_exit == 0) return TEHMM_OK;
    size_t o_cont = 0, o_es = align_up((size_t)nseq), o_ev = align_up(o_es + (size_t)n_entry * 8);
    size_t o_xs = align_up(o_ev + (size_t)n_entry * NP * 8), o_xv = align_up(o_xs + (size_t)n_exit * 8);
    size_t o_save = align_up(o_xv + (size_t)n_exit * NP * 8), bytes = align_up(o_save + (size_t)n_exit * 2 * c->m.LD * 8);
    std::vector<unsigned char> h(bytes, 0);
    for (int64_t k = 0; k < n_entry; ++k) {
        h[o_cont + h_entry_seq[k]] = 1;
        ((int64_t *)&h[o_es])[k] = h_entry_seq[k];
        double sum = 0.0;                     // sum 1: the first chunk's log-likelihood is the increment
        for (int j = 0; j < N; ++j) sum += h_entry_vec[k * N + j];
        for (int j = 0; j < N; ++j) ((double *)&h[o_ev])[k * NP + j] = h_entry_vec[k * N + j] / sum;
    }
    for (int64_t k = 0; k < n_exit; ++k) {
        ((int64_t *)&h[o_xs])[k] = h_exit_seq[k];
        double mx = 0.0;                      // any scale: brought to a maximum of 1
        for (int j = 0; j < N; ++j) mx = std::max(mx, h_exit_vec[k * N + j]);
        for (int j = 0; j < N; ++j) ((double *)&h[o_xv])[k * NP + j] = h_exit_vec[k * N + j] / mx;
    }
    if (bytes > c->bnd_blob_bytes) {
        if (c->bnd_blob) { cudaFree(c->bnd_blob); c->bnd_blob = nullptr; c->bnd_blob_bytes = 0; }
        CU(cudaMalloc(&c->bnd_blob, bytes));
        c->bnd_blob_bytes = bytes;
    }
    CU(cudaMemcpy(c->bnd_blob, h.data(), bytes, cudaMemcpyHostToDevice));
    unsigned char *d = (unsigned char *)c->bnd_blob;
    c->n_entry = n_entry;
    c->n_exit = n_exit;
    c->d_entry_seq = (const int64_t *)(d + o_es);
    c->d_entry_vec = (const double *)(d + o_ev);
    c->d_exit_seq = (const int64_t *)(d + o_xs);
    c->d_exit_vec = (const double *)(d + o_xv);
    c->d_exit_save = d + o_save;
    if (n_entry > 0) c->b.cont = c->bf.cont = (const uint8_t *)(d + o_cont);
    return TEHMM_OK;
}

int tehmm_set_viterbi_boundary(tehmm_ctx *c, int64_t n_entry, const int64_t *h_entry_seq, const double *h_entry_delta,
                               int64_t n_exit, const int64_t *h_exit_seq, const int32_t *h_exit_state,
                               const double *h_exit_ratio)
{
    if (!c) return fail(TEHMM_EINVAL, "ctx is NULL");
    if (!c->has_model) return fail(TEHMM_ESTATE, "tehmm_set_model has not been called");
    if (!c->has_batch) return fail(TEHMM_ESTATE, "tehmm_set_batch has not been called");
    if (n_entry < 0 || n_exit < 0 || (n_entry > 0 && (!h_entry_seq || !h_entry_delta)) ||
        (n_exit > 0 && (!h_exit_seq || !h_exit_state)))
        return fail(TEHMM_EINVAL, "bad argument");
    CU(cudaSetDevice(c->device));
    const int64_t nseq = c->b.nseq;
    const int N = c->m.N, NP = c->m.NP;
    const std::vector<int64_t> off(c->batch_key.begin(), c->batch_key.begin() + nseq + 1);
    if (check_seqs("entry", n_entry, h_entry_seq, nseq, off) || check_seqs("exit", n_exit, h_exit_seq, nseq, off))
        return TEHMM_EINVAL;
    for (int64_t k = 0; k < n_entry; ++k) {
        double mx = -INFINITY;
        for (int j = 0; j < N; ++j) {
            const double x = h_entry_delta[k * N + j];
            if (std::isnan(x) || x == INFINITY) return fail(TEHMM_EINVAL, "entry %lld: component %d is %g (must be finite or -inf)", (long long)k, j, x);
            mx = std::max(mx, x);
        }
        if (!(mx > -INFINITY)) return fail(TEHMM_EINVAL, "entry %lld: every component is -inf", (long long)k);
    }
    for (int64_t k = 0; k < n_exit; ++k) {
        if (h_exit_state[k] < 0 || h_exit_state[k] >= N) return fail(TEHMM_EINVAL, "exit %lld: state %d outside [0,%d)", (long long)k, (int)h_exit_state[k], N);
        const double r = h_exit_ratio ? h_exit_ratio[k] : -1.0;
        if (r >= 0.0 && !(r > 0.0 && std::isfinite(r))) return fail(TEHMM_EINVAL, "exit %lld: ratio %g (must be finite and > 0, or < 0 for none)", (long long)k, r);
        if (std::isnan(r)) return fail(TEHMM_EINVAL, "exit %lld: ratio is NaN", (long long)k);
    }
    CU(cudaStreamSynchronize(c->stream));     // the passes queued so far read the vectors being replaced
    c->n_ventry = c->n_vexit = 0;
    if (n_entry == 0 && n_exit == 0) return TEHMM_OK;
    const size_t o_es = 0, o_ev = align_up(o_es + (size_t)n_entry * 8), o_xs = align_up(o_ev + (size_t)n_entry * NP * 8);
    const size_t o_xst = align_up(o_xs + (size_t)n_exit * 8), o_xr = align_up(o_xst + (size_t)n_exit * 4);
    const size_t bytes = align_up(o_xr + (size_t)n_exit * 8);
    std::vector<unsigned char> h(bytes, 0);
    for (int64_t k = 0; k < n_entry; ++k) {
        ((int64_t *)&h[o_es])[k] = h_entry_seq[k];
        double mx = -INFINITY;                // brought to a maximum of 0, as the DP keeps its rows; padding -inf
        for (int j = 0; j < N; ++j) mx = std::max(mx, h_entry_delta[k * N + j]);
        for (int j = 0; j < NP; ++j) ((double *)&h[o_ev])[k * NP + j] = j < N ? h_entry_delta[k * N + j] - mx : -INFINITY;
    }
    for (int64_t k = 0; k < n_exit; ++k) {
        ((int64_t *)&h[o_xs])[k] = h_exit_seq[k];
        ((int32_t *)&h[o_xst])[k] = h_exit_state[k];
        ((double *)&h[o_xr])[k] = h_exit_ratio && h_exit_ratio[k] > 0.0 ? h_exit_ratio[k] : -1.0;
    }
    if (bytes > c->vbnd_blob_bytes) {
        if (c->vbnd_blob) { cudaFree(c->vbnd_blob); c->vbnd_blob = nullptr; c->vbnd_blob_bytes = 0; }
        CU(cudaMalloc(&c->vbnd_blob, bytes));
        c->vbnd_blob_bytes = bytes;
    }
    CU(cudaMemcpy(c->vbnd_blob, h.data(), bytes, cudaMemcpyHostToDevice));
    unsigned char *d = (unsigned char *)c->vbnd_blob;
    c->n_ventry = n_entry;
    c->n_vexit = n_exit;
    c->d_ventry_seq = (const int64_t *)(d + o_es);
    c->d_ventry_vec = (const double *)(d + o_ev);
    c->d_vexit_seq = (const int64_t *)(d + o_xs);
    c->d_vexit_state = (const int32_t *)(d + o_xst);
    c->d_vexit_ratio = (const double *)(d + o_xr);
    return TEHMM_OK;
}

int tehmm_forward_row(tehmm_ctx *c, int prec, const void *d_alpha, int64_t row, double *h_out)
{
    RUN_PROLOGUE();
    if (!d_alpha || !h_out) return fail(TEHMM_EINVAL, "NULL argument");
    if (row < 0 || row >= c->b.total) return fail(TEHMM_EINVAL, "row %lld outside the batch", (long long)row);
    const int N = c->m.N, LD = c->m.LD;
    const size_t ts = prec == TEHMM_F32 ? 4 : 8;
    std::vector<unsigned char> raw((size_t)LD * ts);
    CU(cudaMemcpyAsync(raw.data(), (const char *)d_alpha + (size_t)row * LD * ts, raw.size(), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    double sum = 0.0;
    for (int j = 0; j < N; ++j) {
        h_out[j] = prec == TEHMM_F32 ? (double)((const float *)raw.data())[j] : ((const double *)raw.data())[j];
        sum += h_out[j];
    }
    if (!(sum > 0.0) || !std::isfinite(sum)) return fail(TEHMM_ESTATE, "forward row %lld sums to %g", (long long)row, sum);
    for (int j = 0; j < N; ++j) h_out[j] /= sum;
    return TEHMM_OK;
}

int tehmm_cut_pair(tehmm_ctx *c, int prec, const double *h_v, const void *d_post_row, double *d_trans, double *h_u)
{
    RUN_PROLOGUE();
    if (!h_v || !d_post_row || !h_u) return fail(TEHMM_EINVAL, "NULL argument");
    const int N = c->m.N;
    DevBuf dv;
    CU(dv.alloc((size_t)2 * N * 8));
    CU(cudaMemcpyAsync(dv.p, h_v, (size_t)N * 8, cudaMemcpyHostToDevice, st));
    CU(tehmm_launch_cut_pair(st, c->m, prec, dv.as<double>(), d_post_row, d_trans, dv.as<double>() + N));
    c->launches += 1;
    CU(cudaMemcpyAsync(h_u, dv.as<double>() + N, (size_t)N * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return TEHMM_OK;
}

int tehmm_convert_rows(tehmm_ctx *c, int prec, const void *d_in, int64_t rows, int renorm, double *d_out)
{
    RUN_PROLOGUE();
    if (!d_in || !d_out || rows < 0) return fail(TEHMM_EINVAL, "bad argument");
    if (rows == 0) return TEHMM_OK;
    CU(tehmm_launch_convert_rows(st, prec, c->m.N, c->m.LD, d_in, rows, renorm, d_out, c->sms));
    c->launches += 1;
    return TEHMM_OK;
}

int tehmm_convert_lattice(tehmm_ctx *c, int prec, const void *d_in, double *d_out, int64_t n)
{
    if (!c || !d_in || !d_out || n < 0) return fail(TEHMM_EINVAL, "bad argument");
    CU(cudaSetDevice(c->device));
    if (n == 0) return TEHMM_OK;
    CU(tehmm_launch_convert(c->stream, prec, d_in, d_out, n));
    c->launches += 1;
    return TEHMM_OK;
}

}   // extern "C"

// ---------------------------------------------------------------- tiny utility kernels
template <typename T>
__global__ void convert_kernel(const T *__restrict__ in, double *__restrict__ out, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = (double)in[i];
}
cudaError_t tehmm_launch_convert(cudaStream_t st, int prec, const void *in, double *out, int64_t n)
{
    int grid = (int)std::min<int64_t>((n + 255) / 256, 148 * 16);
    if (prec == TEHMM_F32) convert_kernel<float><<<grid, 256, 0, st>>>((const float *)in, out, n);
    else convert_kernel<double><<<grid, 256, 0, st>>>((const double *)in, out, n);
    return cudaGetLastError();
}
