// Supervised emission counts of many labelled intervals in one device pass
// (tehmm_supervised_counts, api.cu).  The result equals one strict_counts_kernel
// call per interval in interval order (strict.cu), bit for bit: every bin
// (track, state, symbol) ends as init + w_1 + w_2 + ... with sequential float64
// adds, interval order first, positions ascending within an interval.
//
// The host groups the non-empty intervals by state, keeping interval order
// within a state, and describes them by
//   istart[j]  first table row of interval j (grouped order)
//   pfx[j]     rows of the intervals before j (pfx[m] = all rows): the flattened
//              (interval, position) space
//   sbeg[s]    first interval of state s, sflat[s] = pfx[sbeg[s]]  (N + 1 each)
//
// Two kernels, chosen by the host from the inputs:
//   sup_hist_kernel   unit weights and integer initial values: integer counting
//                     is exact, so order does not matter.  Blocks tile the
//                     flattened rows; a shared-memory histogram of the tile's
//                     current state is flushed with 64-bit integer atomics, and
//                     sup_finalize_kernel adds each count with one float64 add.
//   sup_chain_kernel  anything else: one warp per (track, state) walks that
//                     state's rows in order, 32 at a time; lanes holding the same
//                     symbol form a group (__match_any_sync) and its lowest lane
//                     adds the group's weights in lane order.  Every bin is one
//                     warp's sequential chain, so results are deterministic.
// A symbol >= S is not counted and raises *flag.
#include "common.cuh"
#include <algorithm>

#define SUP_HIST_THREADS 256
#define SUP_HIST_ROWS (SUP_HIST_THREADS * 32)     // flattened rows per block
#define SUP_CHAIN_WARPS 4
#define SUP_CHAIN_STEPS 4                           // 32-row steps loaded ahead of the chains

// interval j in [lo, hi] with pfx[j] <= f < pfx[j + 1]
__device__ __forceinline__ int64_t sup_find(const int64_t *__restrict__ pfx, int64_t lo, int64_t hi, int64_t f)
{
    while (lo < hi) {
        int64_t mid = (lo + hi + 1) >> 1;
        if (pfx[mid] <= f) lo = mid; else hi = mid - 1;
    }
    return lo;
}

template <typename OBS, bool SMEM>
__global__ void __launch_bounds__(SUP_HIST_THREADS)
sup_hist_kernel(const OBS *__restrict__ obs, int K, int N, int S, int64_t m,
                const int64_t *__restrict__ istart, const int64_t *__restrict__ pfx,
                const int64_t *__restrict__ sflat, unsigned long long *__restrict__ counts, int *flag)
{
    extern __shared__ unsigned int hist[];          // K * S (SMEM only)
    __shared__ int64_t s_j[2];
    const int64_t total = pfx[m];
    const int64_t r0 = (int64_t)blockIdx.x * SUP_HIST_ROWS;
    if (r0 >= total) return;
    const int64_t r1 = min(total, r0 + (int64_t)SUP_HIST_ROWS);
    const int KS = K * S;
    if (threadIdx.x == 0) {
        s_j[0] = sup_find(pfx, 0, m - 1, r0);
        s_j[1] = sup_find(pfx, s_j[0], m - 1, r1 - 1);
    }
    if (SMEM)
        for (int b = threadIdx.x; b < KS; b += blockDim.x) hist[b] = 0u;
    __syncthreads();
    const int64_t jlo = s_j[0], jhi = s_j[1];
    int s = 0;
    while (sflat[s + 1] <= r0) ++s;                 // state of the tile's first row
    int bad = 0;
    for (;;) {
        const int64_t a = max(r0, sflat[s]), b = min(r1, sflat[s + 1]);
        int64_t j = jlo;
        for (int64_t f = a + threadIdx.x; f < b; f += blockDim.x) {
            j = sup_find(pfx, j, jhi, f);
            const OBS *row = obs + (istart[j] + (f - pfx[j])) * (int64_t)K;
            for (int k = 0; k < K; ++k) {
                const unsigned sym = (unsigned)row[k];
                if (sym >= (unsigned)S) { bad = 1; continue; }
                if (SMEM) atomicAdd(&hist[k * S + sym], 1u);
                else atomicAdd(&counts[((int64_t)k * N + s) * S + sym], 1ull);
            }
        }
        if (SMEM) {
            __syncthreads();
            for (int e = threadIdx.x; e < KS; e += blockDim.x) {
                const unsigned c = hist[e];
                if (c) {
                    const int k = e / S;
                    atomicAdd(&counts[((int64_t)k * N + s) * S + (e - k * S)], (unsigned long long)c);
                    hist[e] = 0u;
                }
            }
            __syncthreads();
        }
        if (b >= r1) break;
        do { ++s; } while (sflat[s + 1] <= b);
    }
    if (bad) *flag = 1;
}

__global__ void sup_finalize_kernel(const unsigned long long *__restrict__ counts, double *__restrict__ stats,
                                    int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long c = counts[i];
        if (c) stats[i] = stats[i] + (double)c;     // c < 2^53 (checked by the host): exact
    }
}

template <typename OBS>
__global__ void __launch_bounds__(SUP_CHAIN_WARPS * 32)
sup_chain_kernel(const OBS *__restrict__ obs, int K, int N, int S,
                 const int64_t *__restrict__ istart, const int64_t *__restrict__ pfx,
                 const int64_t *__restrict__ sbeg, const int64_t *__restrict__ sflat,
                 const double *__restrict__ ratios, double *stats, int *flag)
{
    __shared__ double sw[SUP_CHAIN_WARPS][SUP_CHAIN_STEPS * 32];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * SUP_CHAIN_WARPS + wib;           // warp-uniform
    if (g >= K * N) return;
    const int s = g % N, k = g / N;
    const int64_t f0 = sflat[s], f1 = sflat[s + 1];
    double *bins = stats + ((int64_t)k * N + s) * S;
    const unsigned NOKEY = 0xffffffffu;
    int64_t j = sbeg[s];
    int bad = 0;
    for (int64_t base = f0; base < f1; base += SUP_CHAIN_STEPS * 32) {
        unsigned key[SUP_CHAIN_STEPS];
        int64_t jj = j;
#pragma unroll
        for (int u = 0; u < SUP_CHAIN_STEPS; ++u) {
            const int64_t f = base + u * 32 + lane;
            key[u] = NOKEY;
            double w = 0.0;
            if (f < f1) {
                while (pfx[jj + 1] <= f) ++jj;
                const int64_t r = istart[jj] + (f - pfx[jj]);
                const unsigned sym = (unsigned)obs[r * K + k];
                w = ratios ? ratios[r] : 1.0;
                if (sym < (unsigned)S) key[u] = sym; else bad = 1;
            }
            sw[wib][u * 32 + lane] = w;
        }
        j = __shfl_sync(0xffffffffu, jj, 31);      // lane 31 holds the furthest row of this round
        __syncwarp();
#pragma unroll
        for (int u = 0; u < SUP_CHAIN_STEPS; ++u) {
            const unsigned grp = __match_any_sync(0xffffffffu, key[u]);
            if (key[u] != NOKEY && lane == __ffs(grp) - 1) {
                double v = bins[key[u]];
                for (unsigned rest = grp; rest; rest &= rest - 1)
                    v += sw[wib][u * 32 + __ffs(rest) - 1];
                bins[key[u]] = v;
            }
            __syncwarp();                          // this step's stores before the next step's loads
        }
    }
    if (bad) *flag = 1;
}

#define SUP_OBS_DISPATCH(BYTES, CALL)                                          \
    do {                                                                       \
        if ((BYTES) == 1) { typedef uint8_t OBS_T; CALL; }                     \
        else if ((BYTES) == 2) { typedef uint16_t OBS_T; CALL; }               \
        else { typedef int32_t OBS_T; CALL; }                                  \
    } while (0)

// bytes of shared memory the histogram kernel uses per block (0: counts straight into global memory)
size_t tehmm_sup_hist_smem(int K, int S)
{
    size_t b = (size_t)K * S * sizeof(unsigned int);
    return b <= 48 * 1024 ? b : 0;
}

// returns the number of kernel launches
int tehmm_launch_sup_hist(cudaStream_t st, const void *obs, int obs_bytes, int K, int N, int S, int64_t m,
                          int64_t rows, const int64_t *istart, const int64_t *pfx, const int64_t *sflat,
                          unsigned long long *counts, double *stats, int *flag)
{
    const int64_t blocks = (rows + SUP_HIST_ROWS - 1) / SUP_HIST_ROWS;
    const size_t smem = tehmm_sup_hist_smem(K, S);
    if (smem)
        SUP_OBS_DISPATCH(obs_bytes, (sup_hist_kernel<OBS_T, true><<<(unsigned)blocks, SUP_HIST_THREADS, smem, st>>>(
            (const OBS_T *)obs, K, N, S, m, istart, pfx, sflat, counts, flag)));
    else
        SUP_OBS_DISPATCH(obs_bytes, (sup_hist_kernel<OBS_T, false><<<(unsigned)blocks, SUP_HIST_THREADS, 0, st>>>(
            (const OBS_T *)obs, K, N, S, m, istart, pfx, sflat, counts, flag)));
    const int64_t bins = (int64_t)K * N * S;
    const int64_t fb = std::min<int64_t>((bins + 255) / 256, 148 * 8);
    sup_finalize_kernel<<<(unsigned)fb, 256, 0, st>>>(counts, stats, bins);
    return 2;
}

int tehmm_launch_sup_chain(cudaStream_t st, const void *obs, int obs_bytes, int K, int N, int S,
                           const int64_t *istart, const int64_t *pfx, const int64_t *sbeg, const int64_t *sflat,
                           const double *ratios, double *stats, int *flag)
{
    const int warps = K * N;
    const int blocks = (warps + SUP_CHAIN_WARPS - 1) / SUP_CHAIN_WARPS;
    SUP_OBS_DISPATCH(obs_bytes, (sup_chain_kernel<OBS_T><<<blocks, SUP_CHAIN_WARPS * 32, 0, st>>>(
        (const OBS_T *)obs, K, N, S, istart, pfx, sbeg, sflat, ratios, stats, flag)));
    return 1;
}
