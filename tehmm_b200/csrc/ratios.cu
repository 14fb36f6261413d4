// Segment ratios on the fast path (VERDICT r1 item 5; _hmm.pyx:140-149,187-188,89-96,106-111).
//
// A segmented table holds one observation per variable-length segment; r_t = segLen_t / effective
// length stands for the r_t - 1 self transitions the segment swallowed.  In the forward and backward
// recursions that is a per-row DIAGONAL factor on the state the chain is in at t:
//     alpha_t[j] = (sum_i alpha_{t-1}[i] A_ij) * A_jj^(r_t - 1) * b_t[j]        (r_t > 1; also t = 0)
//     beta_t[i]  =  sum_j A_ij * A_jj^(r_{t+1} - 1) * b_{t+1}[j] * beta_{t+1}[j]
// i.e. the recursions of an unsegmented table on b'_t[j] = b_t[j] * A_jj^(r_t - 1).  ratio_fold_kernel
// rewrites the linear emission lattice once (the common factor max_j A_jj^(r_t - 1) goes to rowmax, like
// the row maximum of the emission itself), after which forward, backward, posteriors and the xi kernel
// run WITHOUT ratios -- on the tensor-core tile kernels where those apply -- instead of the
// one-chunk-per-warp kernels with an exp() per state per step.  What is left of the ratios in the
// E-step is the diagonal term of _log_sum_lneta (_hmm.pyx:91-96,107-110):
//     trans[j][j] += (1/N) sum_{t > s0, r_t > 1} (r_t - 1) gamma_t[j]                 (ratio_diag_kernel).
// The Viterbi recursion treats from-state 0 differently (_hmm.pyx:234-237) and keeps its own kernels.
#include "scan.cuh"

template <typename T>
__global__ void ratio_fold_kernel(TehmmModelDev m, int64_t total, const double *__restrict__ ratios,
                                  T *__restrict__ blin, double *__restrict__ rowmax)
{
    // lane (and lane + 32) = state
    const int lane = threadIdx.x & 31;
    const int N = m.N, LD = m.LD, NP = m.NP;
    double dg[2], dgmax = -INFINITY;
    for (int u = 0; u < 2; ++u) {
        const int j = lane + 32 * u;
        dg[u] = j < N ? m.cut_trans[(int64_t)j * NP + j] : -INFINITY;
        dgmax = fmax(dgmax, dg[u]);
    }
    dgmax = warp_max(dgmax);
    // a warp takes 32 consecutive rows: one coalesced load of their ratios, then only the rows with r > 1
    const int64_t ngroups = (total + 31) / 32;
    for (int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < ngroups; g += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int64_t tl = g * 32 + lane;
        const double rl = tl < total ? ratios[tl] : 0.0;
        unsigned todo = __ballot_sync(TEHMM_FULL, rl > 1.0);
        while (todo) {
            const int q = __ffs(todo) - 1;
            todo &= todo - 1;
            const int64_t t = g * 32 + q;
            const double r = __shfl_sync(TEHMM_FULL, rl, q);
            for (int u = 0; u < 2; ++u) {
                const int j = lane + 32 * u;
                if (j >= N) continue;
                // (no self transition anywhere: the reference's sum is over impossible paths; zeros, as forward_kernel)
                const double f = dgmax > -INFINITY ? exp((dg[u] - dgmax) * (r - 1.0)) : 0.0;
                blin[t * LD + j] = (T)((double)blin[t * LD + j] * f);
            }
            if (lane == 0 && dgmax > -INFINITY) rowmax[t] += dgmax * (r - 1.0);
        }
    }
}

// part[c][j] = sum over the rows t of coarse chunk c, t > s0, r_t > 1, of (r_t - 1) post[t][j]; one warp per chunk
template <typename T>
__global__ void ratio_diag_kernel(TehmmModelDev m, TehmmBatchDev b, const double *__restrict__ ratios,
                                  const T *__restrict__ post, double *__restrict__ part)
{
    const int lane = threadIdx.x & 31;
    const int N = m.N, LD = m.LD;
    for (int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < b.nchunks; c += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const TehmmChunk ch = b.chunks[c];
        double acc[2] = {0.0, 0.0};
        const int64_t s0 = tehmm_is_start(b, ch.seq) ? ch.s0 : -1;     // a continued sequence has a transition into its first row
        for (int64_t t4 = ch.t0; t4 < ch.t1; t4 += 4) {
            double r[4];                 // four rows in flight: the walk is latency bound
#pragma unroll
            for (int q = 0; q < 4; ++q) r[q] = t4 + q < ch.t1 && t4 + q != s0 ? ratios[t4 + q] : 0.0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (!(r[q] > 1.0)) continue;
                for (int u = 0; u < 2; ++u) {
                    const int j = lane + 32 * u;
                    if (j < N) acc[u] += (r[q] - 1.0) * (double)post[(t4 + q) * LD + j];
                }
            }
        }
        for (int u = 0; u < 2; ++u) part[c * 64 + lane + 32 * u] = acc[u];
    }
}
__global__ void ratio_diag_reduce_kernel(int N, int64_t nchunks, const double *__restrict__ part, double *__restrict__ start_trans)
{
    // one block per state; fixed assignment of chunks to threads and a fixed reduction tree: deterministic
    const int j = blockIdx.x;
    double acc = 0.0;
    for (int64_t c = threadIdx.x; c < nchunks; c += blockDim.x) acc += part[c * 64 + j];
    acc = block_sum(acc);
    if (threadIdx.x == 0) start_trans[N + (int64_t)j * N + j] += acc / (double)N;
}

cudaError_t tehmm_launch_ratio_fold(cudaStream_t st, const TehmmModelDev &m, int64_t total, int prec,
                                    const double *ratios, void *blin, double *rowmax, int sms)
{
    const int grid = (int)std::min<int64_t>((total + 255) / 256, (int64_t)sms * 16);
    if (prec == TEHMM_F32) ratio_fold_kernel<float><<<grid, 256, 0, st>>>(m, total, ratios, (float *)blin, rowmax);
    else ratio_fold_kernel<double><<<grid, 256, 0, st>>>(m, total, ratios, (double *)blin, rowmax);
    return cudaGetLastError();
}
cudaError_t tehmm_launch_ratio_diag(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b, int prec,
                                    const double *ratios, const void *post, double *part, double *start_trans, int sms)
{
    const int grid = (int)std::min<int64_t>((b.nchunks * 32 + 255) / 256, (int64_t)sms * 16);
    if (prec == TEHMM_F32) ratio_diag_kernel<float><<<grid, 256, 0, st>>>(m, b, ratios, (const float *)post, part);
    else ratio_diag_kernel<double><<<grid, 256, 0, st>>>(m, b, ratios, (const double *)post, part);
    ratio_diag_reduce_kernel<<<m.N, 256, 0, st>>>(m.N, b.nchunks, part, start_trans);
    return cudaGetLastError();
}
