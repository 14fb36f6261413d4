// Shared declarations for libtehmm_b200 (sm_100a).  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/tehmm_b200.h"

#define TEHMM_TILE 64           // time steps per traceback tile
#define TEHMM_WARPS_PER_CTA 8   // scan kernels: one chunk per warp
#define TEHMM_FULL 0xffffffffu

// Numerics contract (reference common.py:24-33, _hmm.pyx:59-60, _emission.pyx:11-12)
#define TEHMM_ZEROLOGPROB (-1e200)
#define TEHMM_MINDBL (-1e20)
// batched path: log values at or below this are probability zero (covers
// LOGZERO=-1e100, which does not fit fp32)
#define TEHMM_LOGZERO_CUT (-1e30)

// One chunk of the time partition.  All positions are absolute row indices in
// the concatenated batch.  [t0,t1) is the chunk, [s0,s1) its sequence.
struct TehmmChunk {
    int64_t t0, t1, s0, s1;
    int64_t tile0;   // global index of the chunk's first traceback tile
    int32_t seq;
    int32_t ntiles;
};

// Device-resident model, both spaces, padded to NP = 32*NS states.
struct TehmmModelDev {
    int N, K, S, NS, NP;
    int LD;                     // row stride (elements) of every batched lattice: elog, blin, alpha,
                                // posteriors, delta.  32 for N <= 32 (128-byte rows of float: one
                                // cache line, 16-byte vector / bulk accesses), N otherwise.  Columns
                                // N..LD-1 are padding and always hold zeros.
    int tab_rows;               // rows of the compact transposed table
    int table_in_smem;          // compact table fits the emission kernel's smem
    double normalize;
    const double *log_start;    // [N]      as given
    const double *log_trans;    // [N*N]    as given
    const double *table;        // [K][N][S] as given
    const double *table_t;      // [tab_rows][N] compact, transposed: row = tab_off[k]+symbol
    const int32_t *tab_off;     // [K]
    const int32_t *track_nsym;  // [K]
    const double *lin_start;    // [NP]     exp(log_start), 0 beyond N / below the cut
    const double *lin_trans;    // [NP*NP]  exp(log_trans)
    const double *cut_start;    // [NP]     log_start with <= cut mapped to -inf
    const double *cut_trans;    // [NP*NP]  log_trans with <= cut mapped to -inf
    // Merged emission tables of the fp32 path (emission.cu, emission_merged_kernel):
    // tracks are grouped, a group's table has one row per COMBINATION of its
    // tracks' symbols, holding normalize * sum of the tracks' log-probs, split
    // into the row's maximum over states (gc, float64) and the remainder
    // (gtab, float32, <= 0, NP = 32 * NS floats per row).  G = 0: not available.
    int G, grows;
    const float *gtab;          // [grows][NP]
    const double *gc;           // [grows]
    const int32_t *gdesc;       // [G][TEHMM_GDESC]: ntracks, first row, track[4], stride[4]
    // Merged rows of the emission HISTOGRAMS (stats.cu, emission_stats_merged_kernel): the same
    // kind of grouping under a smaller row budget (a histogram row is 256 bytes of shared memory).
    int SG, srows;
    const int32_t *sgdesc;      // [SG][TEHMM_GDESC]
};
#define TEHMM_GDESC 10
#define TEHMM_GMAX 16           // groups
#define TEHMM_GROWS_MAX 1200    // merged rows (x 128 bytes of shared memory)
#define TEHMM_SROWS_MAX 704     // merged histogram rows (x 256 bytes of shared memory)

struct TehmmBatchDev {
    const void *obs;
    int obs_bytes;
    int64_t nseq, total, nchunks, ntiles;
    const int64_t *seq_off;      // [nseq+1]
    const int64_t *seq_chunk0;   // [nseq+1] first chunk of each sequence
    const TehmmChunk *chunks;    // [nchunks]
    int warmup;
    // [nseq] 1 where the sequence continues one that began before this batch (tehmm_set_boundary:
    // its first row is not a start, so it adds nothing to the start counts), or NULL: none does
    const uint8_t *cont;
};
__device__ __forceinline__ bool tehmm_is_start(const TehmmBatchDev &b, int64_t seq)
{
    return b.cont == nullptr || b.cont[seq] == 0;
}

__device__ __forceinline__ long tehmm_load_sym(const void *obs, int obs_bytes, int64_t idx)
{
    if (obs_bytes == 1) return ((const uint8_t *)obs)[idx];
    if (obs_bytes == 2) return ((const uint16_t *)obs)[idx];
    return ((const int32_t *)obs)[idx];
}

template <typename T> struct TehmmNum;
template <> struct TehmmNum<float> {
    // biased exponent of a non-negative value
    __device__ static __forceinline__ int exponent_bits(float v) { return (int)(__float_as_uint(v) >> 23); }
    __device__ static __forceinline__ unsigned order_bits(float v) { return __float_as_uint(v); }
    // 2^(bias - e): brings a value with biased exponent e into [1,2)
    __device__ static __forceinline__ float inv_scale(int e) { return __uint_as_float((unsigned)(254 - e) << 23); }
    static constexpr int BIAS = 127;
    static constexpr int EMAX = 253;
};
template <> struct TehmmNum<double> {
    __device__ static __forceinline__ int exponent_bits(double v) { return (int)((unsigned)__double2hiint(v) >> 20); }
    __device__ static __forceinline__ unsigned order_bits(double v) { return (unsigned)__double2hiint(v); }
    __device__ static __forceinline__ double inv_scale(int e) { return __hiloint2double((2046 - e) << 20, 0); }
    static constexpr int BIAS = 1023;
    static constexpr int EMAX = 2045;
};
