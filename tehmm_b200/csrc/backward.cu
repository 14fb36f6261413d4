// Chunked parallel-in-time backward pass fused with the posterior glue and the
// Baum-Welch transition counts (hmm.py:715-729,545-568; basehmm.py:265-272,
// 516-517; _hmm.pyx:62-117,160-198).
//
// Same speculate / verify / repair scheme as forward.cu, run right-to-left.
// Lane i owns ROW i of the transition matrix.  At step t the warp holds
//   w[j]    = b_{t+1}[j] * beta_hat_{t+1}[j]            (broadcast through smem)
//   beta'[i]= sum_j A[i][j] w[j]
//   Z       = sum_i alpha_hat_t[i] beta'[i]
//   gamma_t = alpha_hat_t .* beta' / Z                  (posterior, rows sum to 1)
//   xi_t    = alpha_hat_t[i] A[i][j] w[j] / Z           (sums to 1 over i,j)
// so neither the T x N x N lneta tensor nor a T x N beta lattice is ever
// written.  The factor A[i][j] and the reference's 1/N (its beta[T-1] is
// log(1/N), _hmm.pyx:179) are applied once, in the reduction kernel.
//
// Algorithmic HBM bytes per step (fp32): 4N (b) + 4N (alpha) read,
// + 4N written when posteriors are requested, + 1 for MAP states.
#include "scan.cuh"
#include <type_traits>

#define BWD_U 4

// xi accumulators: NP per owned state; packed pairs for float
template <typename T, int NS> struct XiAcc {
    T a[NS][32 * NS];
    T w[32 * NS];       // broadcast vector kept from the mat-vec
    __device__ __forceinline__ void zero()
    {
#pragma unroll
        for (int s = 0; s < NS; ++s)
#pragma unroll
            for (int j = 0; j < 32 * NS; ++j) a[s][j] = (T)0;
    }
    __device__ __forceinline__ void matvec(const T *ws, const MatSlice<T, NS> &A, T (&bp)[NS])
    {
        matvec_sum_keep<T, NS>(ws, A.c, bp, w);
    }
    __device__ __forceinline__ void add(int s, T q)
    {
#pragma unroll
        for (int j = 0; j < 32 * NS; ++j) a[s][j] = fma(q, w[j], a[s][j]);
    }
    __device__ __forceinline__ void store(int s, T *dst) const
    {
#pragma unroll
        for (int j = 0; j < 32 * NS; ++j) dst[j] = a[s][j];
    }
};
template <int NS> struct XiAcc<float, NS> {
    u64 a[NS][16 * NS];
    u64 w[16 * NS];
    __device__ __forceinline__ void zero()
    {
#pragma unroll
        for (int s = 0; s < NS; ++s)
#pragma unroll
            for (int j = 0; j < 16 * NS; ++j) a[s][j] = 0ull;
    }
    __device__ __forceinline__ void matvec(const float *ws, const MatSlice<float, NS> &A, float (&bp)[NS])
    {
        matvec_sum_keep<NS>(ws, A, bp, w);
    }
    __device__ __forceinline__ void add(int s, float q)
    {
        const u64 q2 = pk2(q, q);
#pragma unroll
        for (int j = 0; j < 16 * NS; ++j) a[s][j] = ffma2(q2, w[j], a[s][j]);
    }
    __device__ __forceinline__ void store(int s, float *dst) const
    {
#pragma unroll
        for (int j = 0; j < 16 * NS; j += 2)
            *reinterpret_cast<ulonglong2 *>(dst + 2 * j) = make_ulonglong2(a[s][j], a[s][j + 1]);
    }
};
template <typename T, int NS> struct XiNone {
    __device__ __forceinline__ void zero() {}
};

// OUT = compile-time output selection (TEHMM_BWD_POSTERIORS | TEHMM_BWD_MAP | TEHMM_BWD_TRANS)
template <typename T, int NS, bool RATIO, int OUT>
__global__ void __launch_bounds__(TEHMM_WARPS_PER_CTA * 32, (sizeof(T) == 4 && NS == 1 && !(OUT & TEHMM_BWD_TRANS)) ? 3 : 1)
backward_kernel(TehmmModelDev m, TehmmBatchDev b, int flags, const T *__restrict__ blin,
                const T *__restrict__ alpha, const double *__restrict__ ratios,
                T *__restrict__ post, uint8_t *__restrict__ map_states,
                double *__restrict__ map_part, T *__restrict__ xi_part,
                T *__restrict__ xdiag_part, T *__restrict__ gamma0, T *__restrict__ start_vec,
                T *__restrict__ end_vec, const int *__restrict__ bad, int mode)
{
    constexpr int NP = 32 * NS;
    __shared__ __align__(16) T ws_all[TEHMM_WARPS_PER_CTA][2][NP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T(*ws)[NP] = ws_all[warp];
    const int N = m.N;
    const unsigned Nu = (unsigned)m.LD;      // lattice row stride
    constexpr bool TRANS = (OUT & TEHMM_BWD_TRANS) != 0;
    constexpr bool want_post = (OUT & TEHMM_BWD_POSTERIORS) != 0;
    constexpr bool want_map = (OUT & TEHMM_BWD_MAP) != 0;
    const bool renorm = (flags & TEHMM_BWD_RENORM_EPS) != 0;
    const double eps32 = 1.1920928955078125e-07;
    const double renorm_inv = 1.0 / (1.0 + (double)N * eps32);

    // row i of the transition matrix for each owned state (zero beyond N)
    MatSlice<T, NS> A;
    double dg[NS];
    unsigned jc[NS];
    bool own[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int i = lane + 32 * s;
#pragma unroll
        for (int j = 0; j < NP; ++j) A.set(s, j, (T)m.lin_trans[(int64_t)i * NP + j]);
        dg[s] = RATIO ? m.cut_trans[(int64_t)i * NP + i] : 0.0;
        own[s] = i < N;
        jc[s] = (unsigned)min(i, N - 1);
    }

    for (int64_t ci = (int64_t)blockIdx.x * TEHMM_WARPS_PER_CTA + warp; ci < b.nchunks;
         ci += (int64_t)gridDim.x * TEHMM_WARPS_PER_CTA) {
        if (mode == 1 && !bad[ci]) continue;
        const TehmmChunk ch = b.chunks[ci];
        T u[NS];                 // scaled beta_hat at the step last processed
        int buf = 0;
        typename std::conditional<TRANS, XiAcc<T, NS>, XiNone<T, NS>>::type xi;
        xi.zero();
        T xd[NS];
#pragma unroll
        for (int s = 0; s < NS; ++s) xd[s] = (T)0;
        double mapsum = 0.0;

        // rows are addressed relative to t0 with 32-bit offsets
        const T *__restrict__ bb = blin + ch.t0 * m.LD;
        const T *__restrict__ aa = alpha + ch.t0 * m.LD;
        T *__restrict__ pp = want_post ? post + ch.t0 * m.LD : nullptr;
        uint8_t *__restrict__ mm = want_map ? map_states + ch.t0 : nullptr;
        const double *__restrict__ rr = RATIO ? ratios + ch.t0 : nullptr;

        // w_{t+1} = b_{t+1} .* u [.* g_{t+1}] -> smem ; bp = beta'_t (unscaled).
        // `row1` is the row of t+1 relative to t0.
        auto beta_step = [&](unsigned row1, const T (&bt1)[NS], T (&bp)[NS]) {
            T w[NS];
#pragma unroll
            for (int s = 0; s < NS; ++s) w[s] = bt1[s] * u[s];
            if (RATIO) {
                const double r = rr[row1];
                if (r > 1.0) {
                    double lg[NS], mg = -INFINITY;
#pragma unroll
                    for (int s = 0; s < NS; ++s) { lg[s] = dg[s] * (r - 1.0); mg = fmax(mg, lg[s]); }
                    mg = warp_max(mg);
#pragma unroll
                    for (int s = 0; s < NS; ++s) w[s] = mg > -INFINITY ? w[s] * (T)exp(lg[s] - mg) : (T)0;
                }
            }
#pragma unroll
            for (int s = 0; s < NS; ++s) ws[buf][lane + 32 * s] = w[s];
            __syncwarp();
            if constexpr (TRANS) xi.matvec(ws[buf], A, bp);
            else matvec_sum<NS>(ws[buf], A, bp);
            buf ^= 1;
        };
        auto load_row = [&](const T *base, unsigned row, T (&v)[NS]) {
#pragma unroll
            for (int s = 0; s < NS; ++s) v[s] = base[row * Nu + jc[s]];
        };

        const unsigned nrows = (unsigned)(ch.t1 - ch.t0);
        const unsigned last_row = (unsigned)(ch.s1 - 1 - ch.t0);    // row of the sequence's last step

        // ---- phase A: beta_hat at t1 (speculated), unless the chunk ends its sequence
        if (ch.t1 < ch.s1) {
            if (mode == 0) {
                unsigned rq = nrows + (unsigned)b.warmup;           // row of tq = t1 + warmup
                if (rq > last_row) rq = last_row;
#pragma unroll
                for (int s = 0; s < NS; ++s) u[s] = own[s] ? (T)1 : (T)0;
                for (unsigned r1 = rq; r1 > nrows; --r1) {          // computes beta at row r1-1 >= nrows
                    T bt1[NS], bp[NS];
                    load_row(bb, r1, bt1);
                    // warm-up never accumulates statistics: plain mat-vec
                    {
                        T w[NS];
#pragma unroll
                        for (int s = 0; s < NS; ++s) w[s] = bt1[s] * u[s];
                        if (RATIO) {
                            const double r = rr[r1];
                            if (r > 1.0) {
                                double lg[NS], mg = -INFINITY;
#pragma unroll
                                for (int s = 0; s < NS; ++s) { lg[s] = dg[s] * (r - 1.0); mg = fmax(mg, lg[s]); }
                                mg = warp_max(mg);
#pragma unroll
                                for (int s = 0; s < NS; ++s) w[s] = mg > -INFINITY ? w[s] * (T)exp(lg[s] - mg) : (T)0;
                            }
                        }
#pragma unroll
                        for (int s = 0; s < NS; ++s) ws[buf][lane + 32 * s] = w[s];
                        __syncwarp();
                        matvec_sum<NS>(ws[buf], A, bp);
                        buf ^= 1;
                    }
                    canonicalise<T, NS>(bp);
#pragma unroll
                    for (int s = 0; s < NS; ++s) u[s] = bp[s];
                }
#pragma unroll
                for (int s = 0; s < NS; ++s) start_vec[ci * NP + lane + 32 * s] = u[s];
            } else {
#pragma unroll
                for (int s = 0; s < NS; ++s) u[s] = start_vec[ci * NP + lane + 32 * s];
            }
        }

        // one output step at row r (t = t0 + r): posterior, statistics, then u <- scaled beta_t
        auto out_step = [&](unsigned r, const T (&at)[NS], const T (&bt1)[NS]) {
            T bp[NS];
            const bool last = (r == last_row);
            if (last) {
#pragma unroll
                for (int s = 0; s < NS; ++s) bp[s] = own[s] ? (T)1 : (T)0;
            } else {
                beta_step(r + 1, bt1, bp);
            }
            T p[NS], zl = (T)0;
#pragma unroll
            for (int s = 0; s < NS; ++s) { p[s] = at[s] * bp[s]; zl += p[s]; }
            const T Z = warp_sum(zl);
            T invZ;
            if constexpr (sizeof(T) == 4) invZ = __frcp_rn(Z);
            else invZ = (T)1 / Z;
            T g[NS];
#pragma unroll
            for (int s = 0; s < NS; ++s) g[s] = p[s] * invZ;
            if constexpr (TRANS) {
                if (!last) {
#pragma unroll
                    for (int s = 0; s < NS; ++s) xi.add(s, at[s] * invZ);
                }
                if (RATIO && ch.t0 + r > ch.s0) {
                    // implied self transitions of a long segment (_hmm.pyx:89-96,106-111)
                    const double rt = rr[r];
                    if (rt > 1.0) {
#pragma unroll
                        for (int s = 0; s < NS; ++s) xd[s] += (T)(rt - 1.0) * g[s];
                    }
                }
                if (ch.t0 + r == ch.s0) {
#pragma unroll
                    for (int s = 0; s < NS; ++s) gamma0[(int64_t)ch.seq * NP + lane + 32 * s] = g[s];
                }
            }
            if constexpr (want_post) {
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    if (own[s]) {
                        T gv = g[s];
                        if (renorm) gv = (T)(((double)gv + eps32) * renorm_inv);
                        pp[r * Nu + (unsigned)(lane + 32 * s)] = gv;
                    } else if (lane + 32 * s < m.LD) {
                        pp[r * Nu + (unsigned)(lane + 32 * s)] = (T)0;     // padding column
                    }
                }
            }
            if constexpr (want_map) {
                // argmax with the lowest state winning ties (np.argmax, basehmm.py:357)
                T best;
                int arg;
                if (sizeof(T) == 4) {
                    // posteriors are >= 0: their bit patterns order like the values
                    unsigned bits[NS], mxl = 0u;
#pragma unroll
                    for (int s = 0; s < NS; ++s) {
                        bits[s] = own[s] ? __float_as_uint((float)g[s]) : 0u;
                        mxl = max(mxl, bits[s]);
                    }
                    const unsigned mx = __reduce_max_sync(TEHMM_FULL, mxl);
                    arg = -1;
#pragma unroll
                    for (int s = 0; s < NS; ++s) {       // lowest state among the maxima
                        const unsigned vote = __ballot_sync(TEHMM_FULL, bits[s] == mx);
                        if (arg < 0 && vote) arg = 32 * s + __ffs(vote) - 1;
                    }
                    best = (T)__uint_as_float(mx);
                } else {
                    best = g[0];
                    arg = lane;
#pragma unroll
                    for (int s = 1; s < NS; ++s)
                        if (g[s] > best) { best = g[s]; arg = lane + 32 * s; }
                    if (arg >= N) best = (T)-1;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        T ob = __shfl_xor_sync(TEHMM_FULL, best, o);
                        int oa = __shfl_xor_sync(TEHMM_FULL, arg, o);
                        if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
                    }
                }
                if (lane == 0) {
                    mm[r] = (uint8_t)arg;
                    mapsum += renorm ? ((double)best + eps32) * renorm_inv : (double)best;
                }
            }
            canonicalise<T, NS>(bp);
#pragma unroll
            for (int s = 0; s < NS; ++s) u[s] = bp[s];
        };

        // ---- phase B: rows nrows-1 ... 0, groups of BWD_U with the next group in flight.
        // For row r the step needs alpha[r] and b[r+1]; b of the row after the
        // sequence's last step does not exist and is not used (clamped load).
        T an[BWD_U][NS], bn[BWD_U][NS];
        unsigned left = nrows;            // rows still to do: [0, left)
        auto load_group = [&](unsigned top, T (&a4)[BWD_U][NS], T (&b4)[BWD_U][NS]) {
#pragma unroll
            for (int q = 0; q < BWD_U; ++q) {
                const unsigned r = top - 1 - (unsigned)q;
                load_row(aa, r, a4[q]);
                load_row(bb, min(r + 1, last_row), b4[q]);
            }
        };
        if (left >= BWD_U) load_group(left, an, bn);
        while (left >= 2 * BWD_U) {
            T ac[BWD_U][NS], bc[BWD_U][NS];
#pragma unroll
            for (int q = 0; q < BWD_U; ++q) {
#pragma unroll
                for (int s = 0; s < NS; ++s) { ac[q][s] = an[q][s]; bc[q][s] = bn[q][s]; }
            }
            load_group(left - BWD_U, an, bn);
#pragma unroll
            for (int q = 0; q < BWD_U; ++q) out_step(left - 1 - (unsigned)q, ac[q], bc[q]);
            left -= BWD_U;
        }
        if (left >= BWD_U) {
#pragma unroll
            for (int q = 0; q < BWD_U; ++q) out_step(left - 1 - (unsigned)q, an[q], bn[q]);
            left -= BWD_U;
        }
        for (; left > 0; --left) {
            T at[NS], bt1[NS];
            load_row(aa, left - 1, at);
            load_row(bb, min(left, last_row), bt1);
            out_step(left - 1, at, bt1);
        }
#pragma unroll
        for (int s = 0; s < NS; ++s) end_vec[ci * NP + lane + 32 * s] = u[s];
        if (want_map && lane == 0) map_part[ci] = mapsum;
        if constexpr (TRANS) {
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                xi.store(s, xi_part + ((int64_t)ci * NP + lane + 32 * s) * NP);
                xdiag_part[(int64_t)ci * NP + lane + 32 * s] = xd[s];
            }
        }
    }
}

// start[i] += sum_seq gamma0[seq][i];
// trans[i][j] += (1/N) * ( A[i][j] * sum_chunks xi_part[c][i][j] + [i==j] sum_chunks xdiag_part[c][i] )
// Deterministic: fixed summation order, float64 accumulation.
template <typename T>
__global__ void trans_reduce_kernel(TehmmModelDev m, TehmmBatchDev b, const T *__restrict__ xi_part,
                                    const T *__restrict__ xdiag_part, const T *__restrict__ gamma0,
                                    double *__restrict__ start_trans)
{
    const int N = m.N, NP = m.NP;
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < N) {
        double acc = 0.0;
        for (int64_t s = 0; s < b.nseq; ++s)
            if (b.seq_off[s + 1] > b.seq_off[s] && tehmm_is_start(b, s)) acc += (double)gamma0[s * NP + e];
        start_trans[e] += acc;
    }
    if (e < N * N) {
        int i = e / N, j = e - i * N;
        double acc = 0.0, dacc = 0.0;
        for (int64_t c = 0; c < b.nchunks; ++c) {
            acc += (double)xi_part[(c * NP + i) * NP + j];
            if (i == j) dacc += (double)xdiag_part[c * NP + i];
        }
        start_trans[N + e] += (acc * m.lin_trans[(int64_t)i * NP + j] + dacc) / (double)N;
    }
}

// map_score[seq] = sum over the sequence's chunks (basehmm.py:358)
__global__ void map_reduce_kernel(TehmmBatchDev b, const double *__restrict__ map_part,
                                  double *__restrict__ map_score)
{
    // one block per sequence
    const int64_t s = blockIdx.x;
    double acc = 0.0;
    for (int64_t c = b.seq_chunk0[s] + threadIdx.x; c < b.seq_chunk0[s + 1]; c += blockDim.x) acc += map_part[c];
    acc = block_sum(acc);
    if (threadIdx.x == 0) map_score[s] = acc;
}

template <typename T, int NS>
static cudaError_t launch_bwd(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                              int flags, const T *blin, const T *alpha, const double *ratios,
                              T *post, uint8_t *map_states, double *map_part, T *xi_part,
                              T *xdiag_part, T *gamma0, T *start_vec, T *end_vec, const int *bad,
                              int mode, int grid)
{
    const int th = TEHMM_WARPS_PER_CTA * 32;
    const int out = flags & (TEHMM_BWD_POSTERIORS | TEHMM_BWD_MAP | TEHMM_BWD_TRANS);
#define BWD_GO(R, O) backward_kernel<T, NS, R, O><<<grid, th, 0, st>>>(m, b, flags, blin, alpha, ratios, post, map_states, map_part, xi_part, xdiag_part, gamma0, start_vec, end_vec, bad, mode)
#define BWD_OUT(O) do { if (ratios) BWD_GO(true, O); else BWD_GO(false, O); } while (0)
    switch (out) {
    case 0: BWD_OUT(0); break;
    case 1: BWD_OUT(1); break;
    case 2: BWD_OUT(2); break;
    case 3: BWD_OUT(3); break;
    case 4: BWD_OUT(4); break;
    case 5: BWD_OUT(5); break;
    case 6: BWD_OUT(6); break;
    default: BWD_OUT(7); break;
    }
#undef BWD_OUT
#undef BWD_GO
    return cudaGetLastError();
}

cudaError_t tehmm_launch_backward(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                  int prec, int flags, const void *blin, const void *alpha,
                                  const double *ratios, void *post, uint8_t *map_states,
                                  double *map_part, void *xi_part, void *xdiag_part, void *gamma0,
                                  void *start_vec, void *end_vec, const int *bad, int mode, int grid)
{
    if (prec == TEHMM_F32) {
        if (m.NS == 1) return launch_bwd<float, 1>(st, m, b, flags, (const float *)blin, (const float *)alpha, ratios, (float *)post, map_states, map_part, (float *)xi_part, (float *)xdiag_part, (float *)gamma0, (float *)start_vec, (float *)end_vec, bad, mode, grid);
        return launch_bwd<float, 2>(st, m, b, flags, (const float *)blin, (const float *)alpha, ratios, (float *)post, map_states, map_part, (float *)xi_part, (float *)xdiag_part, (float *)gamma0, (float *)start_vec, (float *)end_vec, bad, mode, grid);
    }
    if (m.NS == 1) return launch_bwd<double, 1>(st, m, b, flags, (const double *)blin, (const double *)alpha, ratios, (double *)post, map_states, map_part, (double *)xi_part, (double *)xdiag_part, (double *)gamma0, (double *)start_vec, (double *)end_vec, bad, mode, grid);
    return launch_bwd<double, 2>(st, m, b, flags, (const double *)blin, (const double *)alpha, ratios, (double *)post, map_states, map_part, (double *)xi_part, (double *)xdiag_part, (double *)gamma0, (double *)start_vec, (double *)end_vec, bad, mode, grid);
}

cudaError_t tehmm_launch_trans_reduce(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                      int prec, const void *xi_part, const void *xdiag_part,
                                      const void *gamma0, double *start_trans)
{
    int cells = m.N * m.N;
    int grid = (cells + 63) / 64;
    if (prec == TEHMM_F32)
        trans_reduce_kernel<float><<<grid, 64, 0, st>>>(m, b, (const float *)xi_part, (const float *)xdiag_part, (const float *)gamma0, start_trans);
    else
        trans_reduce_kernel<double><<<grid, 64, 0, st>>>(m, b, (const double *)xi_part, (const double *)xdiag_part, (const double *)gamma0, start_trans);
    return cudaGetLastError();
}

cudaError_t tehmm_launch_map_reduce(cudaStream_t st, const TehmmBatchDev &b, const double *map_part,
                                    double *map_score)
{
    // one block per sequence; its chunks are read in a strided loop of dependent-latency loads, so long
    // sequences get the widest block (24 us -> a few at 18 944 chunks)
    const int64_t cps = b.nchunks / b.nseq;
    const int th = cps >= 2048 ? 1024 : cps >= 256 ? 256 : 64;
    map_reduce_kernel<<<(int)b.nseq, th, 0, st>>>(b, map_part, map_score);
    return cudaGetLastError();
}
