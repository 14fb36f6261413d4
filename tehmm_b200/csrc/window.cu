// Boundary conditions of a batch that is one window of longer sequences (tehmm_set_boundary): forward-
// backward over time windows, each window exact given the vectors its neighbours hand it.
//
//   entry vector v (forward): alpha at the step before the sequence's first row, sum 1.  The first chunk
//     is run from it like a repaired chunk (start_vec, mode 1), so the first step is (v A) .* b.
//   exit vector u (backward): b .* beta of the step after the sequence's last row, any positive scale.
//     Every backward kernel ends a sequence with beta = 1; with y = A u the last row's beta is y, which is
//     the same as running those kernels on a last row of alpha .* y and b .* y.  exit_kernel scales those
//     two rows in place (the originals saved) before the backward pass and puts them back after it, so no
//     backward kernel changes and their hot loops stay as they are.
//   the transition pair across a cut: (1/N) v_i A_ij u_j / sum(v A u), with u = gamma ./ (v A) from the
//     first posterior row after the cut (cut_pair_kernel; also returns u, the left window's exit vector).
//
// Viterbi (tehmm_set_viterbi_boundary): the entry delta goes through entry_kernel and the DP's repair mode
// like the forward entry vector; the exit state s of the row after the cut fixes the state of the last row,
// argmax_i (delta_last[i] + A'(i, s)) -- one more step of the traceback walk, with its operands
// (vit_exit_kernel) -- and the last chunk is walked again from it (forced end, as a repaired chunk).
#include "scan.cuh"

// start_vec[first chunk of seq[k]] = v[k] (lattice precision), bad[that chunk] = 1 (bad zeroed before)
template <typename T>
__global__ void entry_kernel(TehmmBatchDev b, int NP, int64_t n, const int64_t *__restrict__ seq,
                             const double *__restrict__ vec, T *__restrict__ start_vec, int *__restrict__ bad)
{
    const int64_t k = blockIdx.x;
    if (k >= n) return;
    const int64_t c = b.seq_chunk0[seq[k]];
    for (int j = threadIdx.x; j < NP; j += blockDim.x) start_vec[c * NP + j] = (T)vec[k * NP + j];
    if (threadIdx.x == 0) bad[c] = 1;
}

// restore = 0: save the last row of alpha and of blin of each exit sequence, then scale both by
// y = A u / max(A u); restore = 1: copy the saved rows back.  One block per exit sequence.
template <typename T>
__global__ void exit_kernel(TehmmModelDev m, TehmmBatchDev b, int64_t n, const int64_t *__restrict__ seq,
                            const double *__restrict__ u, T *__restrict__ alpha, T *__restrict__ blin,
                            T *__restrict__ save, int restore)
{
    __shared__ double y[64];
    __shared__ double ymax;
    const int64_t k = blockIdx.x;
    if (k >= n) return;
    const int NP = m.NP, LD = m.LD, N = m.N;
    const int64_t row = b.seq_off[seq[k] + 1] - 1;
    T *a = alpha + row * LD, *bl = blin + row * LD, *sv = save + k * 2 * LD;
    if (restore) {
        for (int j = threadIdx.x; j < LD; j += blockDim.x) { a[j] = sv[j]; bl[j] = sv[LD + j]; }
        return;
    }
    for (int i = threadIdx.x; i < NP; i += blockDim.x) {
        double acc = 0.0;
        if (i < N)
            for (int j = 0; j < N; ++j) acc += m.lin_trans[(int64_t)i * NP + j] * u[k * NP + j];
        y[i] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double mx = 0.0;
        for (int i = 0; i < N; ++i) mx = fmax(mx, y[i]);
        ymax = mx > 0.0 ? mx : 1.0;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < LD; j += blockDim.x) {
        sv[j] = a[j];
        sv[LD + j] = bl[j];
        if (j < N) {
            const double f = y[j] / ymax;
            a[j] = (T)((double)a[j] * f);
            bl[j] = (T)((double)bl[j] * f);
        }
    }
}

// one block: w = v A, u = g ./ w (0 where w = 0), trans[i][j] += v_i A_ij u_j / (N sum_ij v_i A_ij u_j)
template <typename T>
__global__ void cut_pair_kernel(TehmmModelDev m, const double *__restrict__ v, const T *__restrict__ g,
                                double *__restrict__ trans, double *__restrict__ u_out)
{
    __shared__ double vs[64], us[64], red[256];
    const int N = m.N, NP = m.NP;
    for (int j = threadIdx.x; j < N; j += blockDim.x) vs[j] = v[j];
    __syncthreads();
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        double w = 0.0;
        for (int i = 0; i < N; ++i) w += vs[i] * m.lin_trans[(int64_t)i * NP + j];
        const double gj = (double)g[j];
        us[j] = w > 0.0 ? gj / w : 0.0;
        u_out[j] = us[j];
    }
    __syncthreads();
    double part = 0.0;
    for (int e = threadIdx.x; e < N * N; e += blockDim.x) {
        const int i = e / N, j = e - i * N;
        part += vs[i] * m.lin_trans[(int64_t)i * NP + j] * us[j];
    }
    red[threadIdx.x] = part;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    const double tot = red[0];
    if (trans == nullptr || !(tot > 0.0)) return;
    for (int e = threadIdx.x; e < N * N; e += blockDim.x) {
        const int i = e / N, j = e - i * N;
        trans[e] += vs[i] * m.lin_trans[(int64_t)i * NP + j] * us[j] / tot / (double)N;
    }
}

// (rows, LD) lattice -> (rows, N) float64; renorm: the posterior renormalisation of backward_kernel's
// TEHMM_BWD_RENORM_EPS, applied to the stored value and rounded to T first, as that kernel does
template <typename T>
__global__ void convert_rows_kernel(int N, int LD, const T *__restrict__ in, int64_t rows, int renorm,
                                    double *__restrict__ out)
{
    const double eps32 = 1.1920928955078125e-07;
    const double renorm_inv = 1.0 / (1.0 + (double)N * eps32);
    const int64_t n = rows * N;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / N;
        const int j = (int)(e - r * N);
        T gv = in[r * LD + j];
        if (renorm) gv = (T)(((double)gv + eps32) * renorm_inv);
        out[e] = (double)gv;
    }
}

// The traceback's step from state s at the row after the cut back to the last row, with the operands of
// vit_traceback4_kernel (fp32: log A clamped to <= 0 in float, arg-max = smallest bit pattern, lowest state on
// ties) and of vit_traceback_kernel's back() (float64: strict '>' from state 0 up).  r < 0: no segment ratio.
__device__ int vit_exit_argmax(const TehmmModelDev &m, const float *d, int s, double rd)
{
    const int NP = m.NP;
    const float r = (float)rd;
    unsigned best = 0xffffffffu;
    int arg = 0;
    for (int i = 0; i < NP; ++i) {
        float a = fminf((float)m.cut_trans[(int64_t)i * NP + s], 0.f);
        if (i == 0 && r >= 0.f) {
            const float dgs = fminf((float)m.cut_trans[(int64_t)s * NP + s], 0.f);
            const float a00 = (float)m.cut_trans[0];
            float extra0 = dgs > -INFINITY ? (r > 1.f ? dgs : dgs * r) : 0.f;
            if (s == 0 && a00 > -INFINITY) extra0 -= a00;
            a += extra0;
        }
        const unsigned bits = __float_as_uint(d[i] + a);
        if (bits < best) { best = bits; arg = i; }
    }
    return arg;
}
__device__ int vit_exit_argmax(const TehmmModelDev &m, const double *d, int s, double r)
{
    const int NP = m.NP, N = m.N;
    double best = -INFINITY;
    int arg = 0;
    for (int i = 0; i < NP; ++i) {
        double cand = (i < N ? d[i] : -INFINITY) + m.cut_trans[(int64_t)i * NP + s];
        if (i == 0 && r >= 0.0) {
            const double dgs = m.cut_trans[(int64_t)s * NP + s], a00 = m.cut_trans[0];
            const double common = r > 1.0 ? dgs * (r - 1.0) : 0.0;
            double extra0 = dgs > -INFINITY ? dgs * r - common : 0.0;
            if (s == 0 && a00 > -INFINITY) extra0 -= a00;
            cand += extra0;
        }
        if (i == 0 || cand > best) { best = cand; arg = i; }
    }
    return arg;
}

// one thread per exit sequence: forced[last chunk] = spec_end[last chunk] = the state of its last row, bad = 1
template <typename T>
__global__ void vit_exit_kernel(TehmmModelDev m, TehmmBatchDev b, const T *__restrict__ lattice, int64_t n,
                                const int64_t *__restrict__ seq, const int32_t *__restrict__ state,
                                const double *__restrict__ ratio, uint8_t *__restrict__ spec_end,
                                uint8_t *__restrict__ forced, int *__restrict__ bad)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int64_t q = seq[k];
    const int st = vit_exit_argmax(m, lattice + (b.seq_off[q + 1] - 1) * m.LD, state[k], ratio[k]);
    const int64_t c = b.seq_chunk0[q + 1] - 1;
    forced[c] = spec_end[c] = (uint8_t)st;
    bad[c] = 1;
}

cudaError_t tehmm_launch_vit_exit(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b, int prec,
                                  const void *lattice, int64_t n, const int64_t *seq, const int32_t *state,
                                  const double *ratio, uint8_t *spec_end, uint8_t *forced, int *bad)
{
    const int grid = (int)((n + 127) / 128);
    if (prec == TEHMM_F32) vit_exit_kernel<float><<<grid, 128, 0, st>>>(m, b, (const float *)lattice, n, seq, state, ratio, spec_end, forced, bad);
    else vit_exit_kernel<double><<<grid, 128, 0, st>>>(m, b, (const double *)lattice, n, seq, state, ratio, spec_end, forced, bad);
    return cudaGetLastError();
}

cudaError_t tehmm_launch_entry(cudaStream_t st, const TehmmBatchDev &b, int prec, int NP, int64_t n,
                               const int64_t *seq, const double *vec, void *start_vec, int *bad)
{
    cudaError_t e = cudaMemsetAsync(bad, 0, sizeof(int) * (size_t)b.nchunks, st);
    if (e != cudaSuccess) return e;
    if (prec == TEHMM_F32) entry_kernel<float><<<(int)n, 64, 0, st>>>(b, NP, n, seq, vec, (float *)start_vec, bad);
    else entry_kernel<double><<<(int)n, 64, 0, st>>>(b, NP, n, seq, vec, (double *)start_vec, bad);
    return cudaGetLastError();
}

cudaError_t tehmm_launch_exit(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b, int prec, int64_t n,
                              const int64_t *seq, const double *u, void *alpha, void *blin, void *save, int restore)
{
    if (prec == TEHMM_F32) exit_kernel<float><<<(int)n, 64, 0, st>>>(m, b, n, seq, u, (float *)alpha, (float *)blin, (float *)save, restore);
    else exit_kernel<double><<<(int)n, 64, 0, st>>>(m, b, n, seq, u, (double *)alpha, (double *)blin, (double *)save, restore);
    return cudaGetLastError();
}

cudaError_t tehmm_launch_cut_pair(cudaStream_t st, const TehmmModelDev &m, int prec, const double *v, const void *g,
                                  double *trans, double *u_out)
{
    if (prec == TEHMM_F32) cut_pair_kernel<float><<<1, 256, 0, st>>>(m, v, (const float *)g, trans, u_out);
    else cut_pair_kernel<double><<<1, 256, 0, st>>>(m, v, (const double *)g, trans, u_out);
    return cudaGetLastError();
}

cudaError_t tehmm_launch_convert_rows(cudaStream_t st, int prec, int N, int LD, const void *in, int64_t rows,
                                      int renorm, double *out, int sms)
{
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((rows * N + 255) / 256, (int64_t)sms * 16));
    if (prec == TEHMM_F32) convert_rows_kernel<float><<<grid, 256, 0, st>>>(N, LD, (const float *)in, rows, renorm, out);
    else convert_rows_kernel<double><<<grid, 256, 0, st>>>(N, LD, (const double *)in, rows, renorm, out);
    return cudaGetLastError();
}
