// Chunked parallel-in-time Viterbi with on-device parallel traceback
// (hmm.py:668-676 -> _hmm.pyx:201-259).
//
// DP (viterbi_kernel; viterbi_lean_kernel for the fp32 production case, see there):
// one warp per chunk, lane j owns column j of log A in
// registers, delta is kept max-normalised (max = 0) and broadcast through
// shared memory.  The kernel is issue-bound, so it computes VALUES only:
//     delta_t[j] = max_i(delta_{t-1}[i] + logA[i][j]) + e_t[j]
// with packed FADD2 + 3-input FMNMX3 (one instruction per candidate instead of
// four with an explicit arg-max) and writes the normalised delta lattice.
// Chunks that do not begin a sequence speculate their start vector with
// `warmup` steps from a flat vector and are verified / repaired like forward.cu.
//
// Traceback (vit_traceback_kernel): back-pointers are needed only ALONG the
// best path, so they are recomputed there: with state s at time t,
//     s_{t-1} = lowest i maximising delta_{t-1}[i] + logA[i][s]
// from the stored lattice, lane i evaluating candidate i with exactly the
// operands the DP used (so ties fall as in the reference: strict '>' scanning
// from-states upward = lowest from-state, _hmm.pyx:232-247).  One warp per
// chunk walks its chunk right to left.  The chunk's END state depends on the
// chunk to its right, so it is speculated too (walk in from `warmup` steps
// beyond the chunk end, best paths coalesce), then verified against the state
// the right neighbour really reaches, and repaired where different.
//
// The returned log-probability is a float64 re-score of the returned path
// against the float64 tables, so it does not carry fp32 DP rounding.
//
// Segment ratios (RATIO kernels): a NEGATIVE ratio marks a step of a sequence
// that has no ratios (segRatios=None).  Such a step gets the plain recursion:
// the reference's from-state-0 term (_hmm.pyx:234-237) is applied only where
// ratios are present, so it would be wrong to fill 1.0 for such a sequence in
// a batch that mixes the two (tehmm_decode_host_ratios).  Real ratios are > 0.
//
// Algorithmic HBM bytes per step (fp32): DP 4N read (e) + 4N written (delta);
// traceback 4N read + 1 written; re-score K + 1 read.
#include "scan.cuh"

#define VIT_U 4
#define TB_PF 6    // delta rows in flight ahead of the traceback walk

#ifndef VIT_WIDE_WARPS
#define VIT_WIDE_WARPS 12     // fp32, 33..64 states: warps per CTA (one CTA per SM; <= 168 registers)
#endif
template <typename T, int NS, bool RATIO, int WARPS = TEHMM_WARPS_PER_CTA>
__global__ void __launch_bounds__(WARPS * 32, (sizeof(T) == 4 && NS == 1) ? 3 : 1)
viterbi_kernel(TehmmModelDev m, TehmmBatchDev b, const T *__restrict__ elog,
               const double *__restrict__ ratios, T *__restrict__ lattice,
               T *__restrict__ start_vec, T *__restrict__ end_vec,
               const int *__restrict__ bad, int mode)
{
    constexpr int NP = 32 * NS;
    __shared__ __align__(16) T ds_all[WARPS][2][NP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T(*ds)[NP] = ds_all[warp];
    const int N = m.N;
    const unsigned Nu = (unsigned)m.LD;      // lattice row stride
    const T NEG = (T)-INFINITY;

    MatSlice<T, NS> A;       // column j of log A (-inf beyond N and for zero transitions)
    T ls[NS], dg[NS];
    unsigned jc[NS];
    bool own[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int j = lane + 32 * s;
#pragma unroll
        for (int i = 0; i < NP; ++i) A.set(s, i, (T)m.cut_trans[(int64_t)i * NP + j]);
        ls[s] = (T)m.cut_start[j];
        dg[s] = (T)m.cut_trans[(int64_t)j * NP + j];
        own[s] = j < N;
        jc[s] = (unsigned)min(j, N - 1);
    }
    const T a00 = (T)m.cut_trans[0];

    for (int64_t ci = (int64_t)blockIdx.x * WARPS + warp; ci < b.nchunks;
         ci += (int64_t)gridDim.x * WARPS) {
        if (mode == 1 && !bad[ci]) continue;
        const TehmmChunk ch = b.chunks[ci];
        T d[NS];
        int buf = 0;

        int64_t tw = ch.t0;
        bool from_start = ch.t0 == ch.s0;
        if (mode == 0 && ch.t0 > ch.s0) {
            tw = ch.t0 - b.warmup;
            if (tw <= ch.s0) { tw = ch.s0; from_start = true; }
        }
        const T *__restrict__ ee = elog + tw * m.LD;
        T *__restrict__ ll = lattice + tw * m.LD;
        const double *__restrict__ rr = RATIO ? ratios + tw : nullptr;

        auto load_e = [&](unsigned row, T (&et)[NS]) {
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const T v = ee[row * Nu + jc[s]];
                et[s] = own[s] ? v : NEG;
            }
        };
        auto store_d = [&](unsigned row) {
#pragma unroll
            for (int s = 0; s < NS; ++s)     // padding columns (N..LD-1) carry -inf
                if (lane + 32 * s < m.LD) ll[row * Nu + (unsigned)(lane + 32 * s)] = own[s] ? d[s] : NEG;
        };
        auto init = [&](unsigned row, const T (&et)[NS]) {
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                d[s] = ls[s] + et[s];
                if (RATIO) {
                    const double r = rr[row];
                    if (r > 1.0) d[s] += dg[s] * (T)(r - 1.0);
                }
            }
            log_normalise<T, NS>(d);
        };
        auto step = [&](unsigned row, const T (&et)[NS]) {
#pragma unroll
            for (int s = 0; s < NS; ++s) ds[buf][lane + 32 * s] = d[s];
            __syncwarp();
            T y[NS];
            if (!RATIO) {
                matvec_maxval<NS>(ds[buf], A, y);
            } else {
                // _hmm.pyx:234-237 vs 243-244: from-state 0 always gets A_jj*r (minus A_00
                // when j==0); the other from-states get A_jj*(r-1), and only if r>1.
                const T r = (T)rr[row];
                const bool seg = r >= (T)0;        // negative: a sequence without ratios
                const T x0 = ds[buf][0];
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    const T common = r > (T)1 ? dg[s] * (r - (T)1) : (T)0;
                    // (a zero-probability self transition would give inf-inf here; the
                    //  reference's finite -1e100 sentinel has no fp32 twin, see DESIGN.md)
                    T extra0 = seg && dg[s] > NEG ? dg[s] * r - common : (T)0;
                    if (seg && lane + 32 * s == 0 && a00 > NEG) extra0 -= a00;
                    T rest = NEG;      // max over from-states >= 1
                    T c0 = NEG;
#pragma unroll
                    for (int i = 0; i < NP; ++i) {
                        T c;
                        if constexpr (sizeof(T) == 4) c = (i & 1) ? hi2(A.c[s][i >> 1]) : lo2(A.c[s][i >> 1]);
                        else c = A.c[s][i];
                        if (i == 0) c0 = c;
                        else rest = fmax(rest, ds[buf][i] + c);
                    }
                    y[s] = fmax(rest, x0 + c0 + extra0) + common;
                }
            }
            buf ^= 1;
#pragma unroll
            for (int s = 0; s < NS; ++s) d[s] = y[s] + et[s];
            log_normalise<T, NS>(d);
        };

        unsigned row = 0;
        const unsigned row0 = (unsigned)(ch.t0 - tw), row1 = (unsigned)(ch.t1 - tw);
        if (mode == 1) {
#pragma unroll
            for (int s = 0; s < NS; ++s) d[s] = start_vec[ci * NP + lane + 32 * s];
        } else if (from_start) {
            T et[NS];
            load_e(0, et);
            init(0, et);
            if (row0 == 0) store_d(0);
            row = 1;
        } else {
#pragma unroll
            for (int s = 0; s < NS; ++s) d[s] = own[s] ? (T)0 : NEG;
        }
        if (mode == 0 && row0 > 0) {
            for (; row < row0; ++row) {
                T et[NS];
                load_e(row, et);
                step(row, et);
            }
#pragma unroll
            for (int s = 0; s < NS; ++s) start_vec[ci * NP + lane + 32 * s] = d[s];
        }

        T en[VIT_U][NS];
        if (row + VIT_U <= row1) {
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) load_e(row + u, en[u]);
        }
        while (row + 2 * VIT_U <= row1) {
            T ec[VIT_U][NS];
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) {
#pragma unroll
                for (int s = 0; s < NS; ++s) ec[u][s] = en[u][s];
            }
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) load_e(row + VIT_U + u, en[u]);
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) {
                step(row + u, ec[u]);
                store_d(row + u);
            }
            row += VIT_U;
        }
        if (row + VIT_U <= row1) {
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) {
                step(row + u, en[u]);
                store_d(row + u);
            }
            row += VIT_U;
        }
        for (; row < row1; ++row) {
            T et[NS];
            load_e(row, et);
            step(row, et);
            store_d(row);
        }
#pragma unroll
        for (int s = 0; s < NS; ++s) end_vec[ci * NP + lane + 32 * s] = d[s];
    }
}

// ---------------------------------------------------------------------------
// fp32 production DP (N <= 32, LD == 32, no segment ratios): 16 x 2 layout.
//
// viterbi_kernel above gives lane j the whole column j of log A and reads the
// 32 deltas back with 8 broadcast LDS.128 per step.  A broadcast LDS.128 returns
// 512 bytes to the register file and issues once per 8 cycles per SM
// sub-partition (profiles/r01_ubench_instruction_rates.txt), i.e. 64 cycles per
// step against 32 cycles of FADD2/FMNMX3 work: the kernel was bound by the
// shared-memory return path, not by arithmetic.  Here lane l = 2a + h owns the
// candidates of from-states i in [16h, 16h+16) for the TWO to-states 2a, 2a+1
// (still 32 packed entries of log A in registers), so a step needs only
// delta[16h .. 16h+15] = 4 LDS.128, and one xor-1 shuffle combines the two
// halves: lane l keeps the maximum of to-state 2a+h = l, so e rows, delta rows
// and the normalisation stay one-lane-per-state.  max is exact and the adds see
// the same operands as before, so the lattice is bit-identical to viterbi_kernel's.
// RATIO: segment ratios (_hmm.pyx:222-225,232-247).  Every candidate of to-state j gets
// common_j = [r_t > 1] logA_jj (r_t - 1), folded into e; the from-state-0 candidate gets logA_jj r_t
// instead (minus logA_00 when j = 0) -- the reference's asymmetry -- i.e. a per-step correction
// x0_j = (r_t > 1 ? logA_jj : logA_jj r_t) - [j = 0] logA_00 on ONE of a lane's 32 candidates.
template <bool RATIO>
__global__ void __launch_bounds__(TEHMM_WARPS_PER_CTA * 32, 3)
viterbi_lean_kernel(TehmmModelDev m, TehmmBatchDev b, const float *__restrict__ elog,
                    float *__restrict__ lattice, float *__restrict__ start_vec,
                    float *__restrict__ end_vec, const int *__restrict__ bad, int mode,
                    const double *__restrict__ rowmax, double *__restrict__ score_part,
                    const double *__restrict__ ratios)
{
    // score_part != nullptr: the chunk also returns its share of the Viterbi log-probability,
    //     sum over its rows of (the maximum M_t taken out of the delta row + rowmax[t]),
    // i.e. the reference's viterbi_lattice[T-1, argmax] (_hmm.pyx:252-254) telescoped over the
    // max-normalised rows (the last row's maximum is 0).  M_t is summed in fp32 over VIT_U steps
    // and then in float64; the chunks' shares add up because a verified start vector is the true
    // normalised row (both have maximum 0).  This replaces the float64 re-score pass.
    __shared__ __align__(16) float ds_all[TEHMM_WARPS_PER_CTA][2][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int h = lane & 1, a2 = lane & ~1;
    const bool own = lane < m.N;
    // A2[jj][q] = (logA[16h+2q][2a+jj], logA[16h+2q+1][2a+jj])
    u64 A2[2][8];
#pragma unroll
    for (int jj = 0; jj < 2; ++jj)
#pragma unroll
        for (int q = 0; q < 8; ++q)
            A2[jj][q] = pk2((float)m.cut_trans[(int64_t)(16 * h + 2 * q) * 32 + a2 + jj],
                            (float)m.cut_trans[(int64_t)(16 * h + 2 * q + 1) * 32 + a2 + jj]);
    const float ls = (float)m.cut_start[lane];
    const uint32_t ds_base = (uint32_t)__cvta_generic_to_shared(&ds_all[warp][0][0]);
    const uint32_t ds_rd = ds_base + 64u * (uint32_t)h, ds_wr = ds_base + 4u * (uint32_t)lane;
    // RATIO: diagonal of log A for this lane's state (common term) and for its two to-states (from-0 correction)
    const float dgl = RATIO ? (float)m.cut_trans[(int64_t)lane * 32 + lane] : 0.f;
    const float dg0 = RATIO ? (float)m.cut_trans[(int64_t)a2 * 32 + a2] : 0.f;
    const float dg1 = RATIO ? (float)m.cut_trans[(int64_t)(a2 + 1) * 32 + a2 + 1] : 0.f;
    const float a00 = RATIO ? (float)m.cut_trans[0] : 0.f;

    for (int64_t ci = (int64_t)blockIdx.x * TEHMM_WARPS_PER_CTA + warp; ci < b.nchunks;
         ci += (int64_t)gridDim.x * TEHMM_WARPS_PER_CTA) {
        if (mode == 1 && !bad[ci]) continue;
        const TehmmChunk ch = b.chunks[ci];
        int64_t tw = ch.t0;
        bool from_start = ch.t0 == ch.s0;
        if (mode == 0 && ch.t0 > ch.s0) {
            tw = ch.t0 - b.warmup;
            if (tw <= ch.s0) { tw = ch.s0; from_start = true; }
        }
        const float *ep = elog + tw * 32 + lane;
        float *lp = lattice + tw * 32 + lane;
        const double *rp = RATIO ? ratios + tw : nullptr;
        unsigned row = 0;
        const unsigned row0 = (unsigned)(ch.t0 - tw), row1 = (unsigned)(ch.t1 - tw);
        float dd, msum = 0.f;
        double macc = 0.0;

        // one DP step from dd (all lanes) with emission value et.  wr / rd: shared-space
        // addresses of this lane's slot and of its half of the vector in the buffer used by
        // this step (the two buffers alternate, so a lane may run one step ahead of the others).
        // Lanes >= N need no masking: their columns of log A are -inf and elog padding is 0.
        auto lean_step = [&](float et, uint32_t wr, uint32_t rd, float r = 1.f) {
            asm volatile("st.shared.f32 [%0], %1;" :: "r"(wr), "f"(dd) : "memory");
            __syncwarp();
            u64 x[8];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                asm volatile("ld.shared.v2.u64 {%0,%1}, [%2];" : "=l"(x[2 * q]), "=l"(x[2 * q + 1]) : "r"(rd + 16u * q) : "memory");
            float p0, p1;
            {
                const u64 c0 = fadd2(x[0], A2[0][0]), c1 = fadd2(x[0], A2[1][0]);
                float f0 = lo2(c0), f1 = lo2(c1);          // candidates of from-state 16h
                if (RATIO) {
                    // (a zero-probability self transition would give inf - inf in the reference's terms; guarded to 0
                    //  like viterbi_kernel, DESIGN.md section 6; r < 0: a sequence without ratios, no correction)
                    const bool seg = r >= 0.f;
                    float x0 = seg && dg0 > -INFINITY ? (r > 1.f ? dg0 : dg0 * r) : 0.f;
                    float x1 = seg && dg1 > -INFINITY ? (r > 1.f ? dg1 : dg1 * r) : 0.f;
                    if (seg && a2 == 0 && a00 > -INFINITY) x0 -= a00;
                    if (h == 0) { f0 += x0; f1 += x1; }
                    if (r > 1.f) et += dgl * (r - 1.f);      // -inf for a state without self transition: it cannot hold a long segment
                }
                p0 = fmaxf(f0, hi2(c0));
                p1 = fmaxf(f1, hi2(c1));
            }
#pragma unroll
            for (int q = 1; q < 8; ++q) {
                const u64 c0 = fadd2(x[q], A2[0][q]), c1 = fadd2(x[q], A2[1][q]);
                p0 = fmax3(p0, lo2(c0), hi2(c0));
                p1 = fmax3(p1, lo2(c1), hi2(c1));
            }
            // lane 2a keeps to-state 2a and needs the partner's p0; lane 2a+1 keeps 2a+1
            const float give = h ? p0 : p1, keep = h ? p1 : p0;
            const float v = fmaxf(keep, __shfl_xor_sync(TEHMM_FULL, give, 1)) + et;
            // every delta and log-probability is <= 0: the row maximum is the unsigned MINIMUM
            // of the bit patterns (+0.0 = 0 is the smallest pattern, -inf the largest).  An
            // all -inf row gives -inf - -inf = NaN, which the max turns back into -inf.
            const float M = __uint_as_float(__reduce_min_sync(TEHMM_FULL, __float_as_uint(v)));
            dd = fmaxf(v - M, -INFINITY);
            msum += M;
        };
        uint32_t wrA = ds_wr, wrB = ds_wr + 128u, rdA = ds_rd, rdB = ds_rd + 128u;
        auto step1 = [&](float et, float r = 1.f) {       // single step, then swap the buffers
            lean_step(et, wrA, rdA, r);
            uint32_t t = wrA; wrA = wrB; wrB = t;
            t = rdA; rdA = rdB; rdB = t;
        };

        if (mode == 1) {
            dd = start_vec[ci * 32 + lane];
        } else if (from_start) {
            float v = ls + (own ? *ep : -INFINITY);
            if (RATIO) {                   // _hmm.pyx:222-225
                const float r0 = (float)rp[0];
                if (r0 > 1.f && dgl > -INFINITY) v += dgl * (r0 - 1.f);
                else if (r0 > 1.f) v = -INFINITY;
            }
            const float M = __uint_as_float(__reduce_min_sync(TEHMM_FULL, __float_as_uint(v)));
            dd = v - (M > -INFINITY ? M : 0.f);
            if (row0 == 0) { *lp = dd; macc = (double)M; }
            ep += 32; lp += 32;
            if (RATIO) rp += 1;
            row = 1;
        } else {
            dd = own ? 0.f : -INFINITY;
        }
        if (mode == 0 && row0 > 0) {
            for (; row < row0; ++row) { step1(*ep, RATIO ? (float)*rp : 1.f); ep += 32; lp += 32; if (RATIO) rp += 1; }
            start_vec[ci * 32 + lane] = dd;
            msum = 0.f;                   // warm-up rows belong to the chunk on the left
        }
        // steady state: the next VIT_U rows of e in flight; VIT_U is even, so the buffer
        // parity is the same at the top of every iteration
        float en[VIT_U], rn[VIT_U];
        if (row + VIT_U <= row1) {
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) { en[u] = ep[u * 32]; rn[u] = RATIO ? (float)rp[u] : 1.f; }
        }
        while (row + 2 * VIT_U <= row1) {
            float ec[VIT_U], rc[VIT_U];
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) { ec[u] = en[u]; rc[u] = rn[u]; }
            ep += VIT_U * 32;
            if (RATIO) rp += VIT_U;
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) { en[u] = ep[u * 32]; rn[u] = RATIO ? (float)rp[u] : 1.f; }
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) {
                if (u & 1) lean_step(ec[u], wrB, rdB, rc[u]); else lean_step(ec[u], wrA, rdA, rc[u]);
                lp[u * 32] = dd;
            }
            lp += VIT_U * 32;
            row += VIT_U;
            macc += (double)msum; msum = 0.f;
        }
        if (row + VIT_U <= row1) {
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) {
                if (u & 1) lean_step(en[u], wrB, rdB, rn[u]); else lean_step(en[u], wrA, rdA, rn[u]);
                lp[u * 32] = dd;
            }
            ep += VIT_U * 32; lp += VIT_U * 32;
            if (RATIO) rp += VIT_U;
            row += VIT_U;
        }
        for (; row < row1; ++row) { step1(*ep, RATIO ? (float)*rp : 1.f); *lp = dd; ep += 32; lp += 32; if (RATIO) rp += 1; }
        end_vec[ci * 32 + lane] = dd;
        if (score_part != nullptr) {
            double rs = 0.0;
            for (int64_t t = ch.t0 + lane; t < ch.t1; t += 32) rs += rowmax[t];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(TEHMM_FULL, rs, o);
            if (lane == 0) score_part[ci] = macc + (double)msum + rs;
        }
    }
}

// ---------------------------------------------------------------------------
// fp32 DP for 33..64 states (lattice rows of 64 floats): TWO warps per chunk (round 2).
//
// viterbi_kernel<float, 2> gives a lane two whole columns of log A: 128 registers, so one CTA of 8-12 warps per
// SM whatever the launch bounds, 16 broadcast LDS.128 per step, and (ncu, profiles/r02_notes_wide.md) 46 % issue
// utilisation with the warps waiting on those loads.  Here warp w of a pair owns the to-states 32w .. 32w+31 and
// lane l = 4a + h of it the candidates of sixteen from-states (16q + 4h + r) for the four to-states 32w+4a .. 32w+4a+3
// (64 packed entries of log A = 64 registers, 16 warps per SM): 4 LDS.128 per step, four independent
// FADD2 / FMNMX3 chains, and two xor-shuffle stages leave lane l with to-state 32w + l.  The halves of the row
// meet in shared memory once per step (one 64-thread named barrier per pair).  The row is normalised LAZILY: a
// lane publishes v_t = max_i(v_{t-1,i} + logA_ij) + e_tj - M_{t-1} and its warp's maximum; M_t = max of the two
// is known to everybody behind the barrier, so the next step subtracts it (max_i(x_i - M + a) = max_i(x_i + a) - M)
// and the owner stores delta_t = v_t - M_t one step late.  Same chunk protocol as viterbi_kernel (start_vec /
// end_vec normalised, maximum 0).
// RATIO: segment ratios as in viterbi_lean_kernel.  The common term [r_t > 1] logA_jj (r_t - 1) is folded into the
// lane's e; the from-state-0 correction goes to the first candidate of the lanes of group h = 0, which hold
// from-state 0 for their four to-states.
#define VW_PAIRS 8
#ifndef VW_ENABLED
#define VW_ENABLED 1
#endif
template <bool RATIO>
__global__ void __launch_bounds__(VW_PAIRS * 64, 1)
viterbi_wide_kernel(TehmmModelDev m, TehmmBatchDev b, const float *__restrict__ elog,
                    float *__restrict__ lattice, float *__restrict__ start_vec,
                    float *__restrict__ end_vec, const int *__restrict__ bad, int mode,
                    const double *__restrict__ ratios)
{
    __shared__ __align__(16) float ds_all[VW_PAIRS][2][72];      // 64 values, the two warps' maxima at [64], [65]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, pair = warp >> 1, w = warp & 1;
    const int h = lane & 3, a4 = lane & ~3;
    const int j = 32 * w + lane;                                   // the to-state this lane ends up with
    // from-states of lane group h: 16q + 4h + r (q, r < 4) -- the four groups of one LDS.128 read one contiguous 64-byte
    // span (16 distinct banks); 16h + 4q + r would put groups h and h + 2 on the same banks
    // A2[k][2q + r/2] = (logA[16q+4h+r][32w+4a+k], logA[16q+4h+r+1][32w+4a+k]), r = 0, 2
    u64 A2[4][8];
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int i0 = 16 * (q >> 1) + 4 * h + 2 * (q & 1);
            A2[k][q] = pk2((float)m.cut_trans[(int64_t)i0 * 64 + 32 * w + a4 + k],
                           (float)m.cut_trans[(int64_t)(i0 + 1) * 64 + 32 * w + a4 + k]);
        }
    const float ls = (float)m.cut_start[j];
    const bool own = j < m.N;
    const uint32_t ds_base = (uint32_t)__cvta_generic_to_shared(&ds_all[pair][0][0]);
    const uint32_t BUF = 72u * 4u;
    const int bar_id = 1 + pair;
    const bool h0 = (h & 1) != 0, h1 = (h & 2) != 0;
    // RATIO: diagonal of log A for this lane's state (common term) and, on the lanes of group h = 0, for its four
    // to-states (from-0 correction x0_k = logA_kk min(r, 1) - [k = 0] logA_00, i.e. (r > 1 ? logA_kk : logA_kk r) as
    // viterbi_lean_kernel writes it; 0 on the other lanes, and for a -inf diagonal, DESIGN.md section 6)
    const float dgl = RATIO ? (float)m.cut_trans[(int64_t)j * 64 + j] : 0.f;
    float dgk[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int jk = 32 * w + a4 + k;
        const float d = RATIO ? (float)m.cut_trans[(int64_t)jk * 64 + jk] : 0.f;
        dgk[k] = h == 0 && d > -INFINITY ? d : 0.f;
    }
    const float a00 = RATIO && h == 0 && w == 0 && a4 == 0 && m.cut_trans[0] > -INFINITY ? (float)m.cut_trans[0] : 0.f;

    for (int64_t ci = (int64_t)blockIdx.x * VW_PAIRS + pair; ci < b.nchunks; ci += (int64_t)gridDim.x * VW_PAIRS) {
        if (mode == 1 && !bad[ci]) continue;                       // the same decision in both warps of the pair
        const TehmmChunk ch = b.chunks[ci];
        int64_t tw = ch.t0;
        bool from_start = ch.t0 == ch.s0;
        if (mode == 0 && ch.t0 > ch.s0) {
            tw = ch.t0 - b.warmup;
            if (tw <= ch.s0) { tw = ch.s0; from_start = true; }
        }
        const float *ep = elog + tw * 64 + j;
        float *lp = lattice + tw * 64 + j;
        const double *rp = RATIO ? ratios + tw : nullptr;             // advances with ep
        const int row0 = (int)(ch.t0 - tw), row1 = (int)(ch.t1 - tw);
        int row = 0, cur = 0;
        float vv;                                                  // this lane's published value of row - 1

        // publish v (this lane's state) and the warp's maximum in buffer `buf`, meet the other warp
        auto publish = [&](float v, int buf) {
            const float mw = __uint_as_float(__reduce_min_sync(TEHMM_FULL, __float_as_uint(v)));   // values <= 0: see viterbi_lean_kernel
            asm volatile("st.shared.f32 [%0], %1;" :: "r"(ds_base + (uint32_t)buf * BUF + 4u * (uint32_t)j), "f"(v) : "memory");
            if (lane == 0) asm volatile("st.shared.f32 [%0], %1;" :: "r"(ds_base + (uint32_t)buf * BUF + 256u + 4u * (uint32_t)w), "f"(mw) : "memory");
            asm volatile("bar.sync %0, 64;" :: "r"(bar_id) : "memory");
        };
        // maximum of the row published in `buf`
        auto row_max = [&](int buf) -> float {
            float m0, m1;
            asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(m0), "=f"(m1) : "r"(ds_base + (uint32_t)buf * BUF + 256u) : "memory");
            return fmaxf(m0, m1);
        };
        // one step: row `row` from the row published in `cur`; stores the row before it if it is an output row
        auto step = [&](float et, float r) {
            const uint32_t rd = ds_base + (uint32_t)cur * BUF + 16u * (uint32_t)h;
            u64 x[8];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                asm volatile("ld.shared.v2.u64 {%0,%1}, [%2];" : "=l"(x[2 * q]), "=l"(x[2 * q + 1]) : "r"(rd + 64u * q) : "memory");
            const float M = row_max(cur);
            if (row - 1 >= row0) lp[(int64_t)(row - 1) * 64] = fmaxf(vv - M, -INFINITY);      // all -inf: NaN -> -inf
            float p[4];
            // r < 0: a sequence without ratios, no correction (min(max(r, 0), 1) = 0)
            const float rc = RATIO ? __saturatef(r) : 0.f, a0 = RATIO && r >= 0.f ? a00 : 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const u64 c0 = fadd2(x[0], A2[k][0]);
                float f = lo2(c0);                                 // from-state 4h: from-state 0 in group h = 0
                if (RATIO) {
                    float x0 = dgk[k] * rc;
                    if (k == 0) x0 -= a0;
                    f += x0;
                }
                p[k] = fmaxf(f, hi2(c0));
            }
            if (RATIO && r > 1.f) et += dgl * (r - 1.f);           // -inf for a state without self transition
#pragma unroll
            for (int q = 1; q < 8; ++q) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const u64 c = fadd2(x[q], A2[k][q]);
                    p[k] = fmax3(p[k], lo2(c), hi2(c));
                }
            }
            // from-state groups meet: xor 2 leaves to-states 2*h1, 2*h1+1 of the four, xor 1 leaves 2*h1 + h0 = h
            float k0 = h1 ? p[2] : p[0], k1 = h1 ? p[3] : p[1];
            const float g0 = h1 ? p[0] : p[2], g1 = h1 ? p[1] : p[3];
            k0 = fmaxf(k0, __shfl_xor_sync(TEHMM_FULL, g0, 2));
            k1 = fmaxf(k1, __shfl_xor_sync(TEHMM_FULL, g1, 2));
            const float keep = h0 ? k1 : k0, give = h0 ? k0 : k1;
            const float pj = fmaxf(keep, __shfl_xor_sync(TEHMM_FULL, give, 1));
            vv = fmaxf(pj + et - M, -INFINITY);
            publish(vv, cur ^ 1);
            cur ^= 1;
            row += 1;
        };

        if (mode == 1) {
            vv = start_vec[ci * 64 + j];
            publish(vv, cur);
            row = 0;
        } else if (from_start) {
            vv = ls + (own ? *ep : -INFINITY);                     // _hmm.pyx:214-220
            if (RATIO) {                                           // _hmm.pyx:222-225
                const float r0 = (float)rp[0];
                if (r0 > 1.f) vv += dgl * (r0 - 1.f);
                rp += 1;
            }
            publish(vv, cur);
            ep += 64;
            row = 1;
        } else {
            vv = own ? 0.f : -INFINITY;
            publish(vv, cur);
            row = 0;
        }
        // (a virtual row -1 published by the first and the third branch is never stored: -1 < row0)
        if (mode == 0 && row0 > 0) {
            while (row < row0) { step(*ep, RATIO ? (float)*rp : 1.f); ep += 64; if (RATIO) rp += 1; }
            const float M = row_max(cur);
            start_vec[ci * 64 + j] = fmaxf(vv - M, -INFINITY);
        }
        float en[VIT_U], rn[VIT_U];
        if (row + VIT_U <= row1) {
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) { en[u] = ep[u * 64]; rn[u] = RATIO ? (float)rp[u] : 1.f; }
        }
        while (row + 2 * VIT_U <= row1) {
            float ec[VIT_U], rc[VIT_U];
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) { ec[u] = en[u]; rc[u] = rn[u]; }
            ep += VIT_U * 64;
            if (RATIO) rp += VIT_U;
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) { en[u] = ep[u * 64]; rn[u] = RATIO ? (float)rp[u] : 1.f; }
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) step(ec[u], rc[u]);
        }
        if (row + VIT_U <= row1) {
#pragma unroll
            for (int u = 0; u < VIT_U; ++u) step(en[u], rn[u]);
            ep += VIT_U * 64;
            if (RATIO) rp += VIT_U;
        }
        while (row < row1) { step(*ep, RATIO ? (float)*rp : 1.f); ep += 64; if (RATIO) rp += 1; }
        {
            const float M = row_max(cur);
            const float dlast = fmaxf(vv - M, -INFINITY);
            if (row - 1 >= row0) lp[(int64_t)(row - 1) * 64] = dlast;
            end_vec[ci * 64 + j] = dlast;
        }
        // the pair's buffers are reused by its next chunk: nobody may still be reading this one's last row
        asm volatile("bar.sync %0, 64;" :: "r"(bar_id) : "memory");
    }
}

// order-preserving key of a float for REDUX (larger value -> larger key)
__device__ __forceinline__ unsigned order_key(float v)
{
    const unsigned bts = __float_as_uint(v);
    return bts ^ ((unsigned)((int)bts >> 31) | 0x80000000u);
}

// lowest state index among the maxima of a warp-distributed vector
template <typename T, int NS>
__device__ __forceinline__ int warp_argmax_first(const T (&v)[NS], int lane)
{
    if constexpr (sizeof(T) == 4 && NS == 1) {
        const unsigned key = order_key((float)v[0]);
        const unsigned mx = __reduce_max_sync(TEHMM_FULL, key);
        return __ffs(__ballot_sync(TEHMM_FULL, key == mx)) - 1;
    } else {
        T best = v[0];
        int arg = lane;
#pragma unroll
        for (int s = 1; s < NS; ++s)
            if (v[s] > best) { best = v[s]; arg = lane + 32 * s; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const T ob = __shfl_xor_sync(TEHMM_FULL, best, o);
            const int oa = __shfl_xor_sync(TEHMM_FULL, arg, o);
            if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
        }
        return arg;
    }
}

// One warp per chunk.  mode 0: speculate the chunk's end state, walk the chunk,
// record the state it implies for the left neighbour (pred).  mode 1: redo the
// chunks whose end state was wrong, from the forced end state.
template <typename T, int NS, bool RATIO>
__global__ void __launch_bounds__(TEHMM_WARPS_PER_CTA * 32, (sizeof(T) == 4 && NS == 1) ? 5 : 1)
vit_traceback_kernel(TehmmModelDev m, TehmmBatchDev b, const T *__restrict__ lattice,
                     const double *__restrict__ ratios, uint8_t *__restrict__ states,
                     int64_t *__restrict__ states64, uint8_t *__restrict__ spec_end,
                     uint8_t *__restrict__ pred, const uint8_t *__restrict__ forced_end,
                     const int *__restrict__ bad, int mode)
{
    constexpr int NP = 32 * NS;
    extern __shared__ __align__(16) unsigned char tb_smem[];
    T *AT = reinterpret_cast<T *>(tb_smem);               // AT[s*NP + i] = logA[i][s]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int N = m.N;
    const unsigned Nu = (unsigned)m.LD;      // lattice row stride
    const T NEG = (T)-INFINITY;
    for (int e = threadIdx.x; e < NP * NP; e += blockDim.x) {
        const int s = e / NP, i = e - s * NP;
        AT[e] = (T)m.cut_trans[(int64_t)i * NP + s];
    }
    __syncthreads();
    const T a00 = (T)m.cut_trans[0];
    unsigned jc[NS];
    bool own[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        own[s] = lane + 32 * s < N;
        jc[s] = (unsigned)min(lane + 32 * s, N - 1);
    }

    for (int64_t ci = (int64_t)blockIdx.x * TEHMM_WARPS_PER_CTA + warp; ci < b.nchunks;
         ci += (int64_t)gridDim.x * TEHMM_WARPS_PER_CTA) {
        if (mode == 1 && !bad[ci]) continue;
        const TehmmChunk ch = b.chunks[ci];
        // rows relative to t0 - 1 (row 0 = the left neighbour's last step, if any)
        const int64_t tbase = ch.t0 > ch.s0 ? ch.t0 - 1 : ch.t0;
        const T *__restrict__ ll = lattice + tbase * m.LD;
        const double *__restrict__ rr = RATIO ? ratios + tbase : nullptr;
        const unsigned rfirst = (unsigned)(ch.t0 - tbase);            // row of t0 (0 or 1)
        const unsigned rlast = (unsigned)(ch.t1 - 1 - tbase);         // row of t1-1

        auto load_d = [&](unsigned row, T (&dv)[NS]) {
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const T v = ll[row * Nu + jc[s]];
                dv[s] = own[s] ? v : NEG;
            }
        };
        // state at row-1 given state st at `row`, from delta[row-1] (already loaded)
        auto back = [&](unsigned row, int st, const T (&dprev)[NS]) -> int {
            T cand[NS];
#pragma unroll
            for (int s = 0; s < NS; ++s) cand[s] = dprev[s] + AT[st * NP + lane + 32 * s];
            if (RATIO) {
                // only the from-state-0 candidate differs between from-states (see viterbi_kernel)
                const T r = (T)rr[row];
                if (lane == 0 && r >= (T)0) {           // negative: a sequence without ratios
                    const T dgs = AT[st * NP + st];
                    const T common = r > (T)1 ? dgs * (r - (T)1) : (T)0;
                    T extra0 = dgs > NEG ? dgs * r - common : (T)0;
                    if (st == 0 && a00 > NEG) extra0 -= a00;
                    cand[0] += extra0;
                }
            }
            return warp_argmax_first<T, NS>(cand, lane);
        };

        // Walk rows hi, hi-1, ..., lo+1 (state at `hi` known), calling emit(row, st)
        // for every visited row and finishing with st = state at row `lo`.
        // delta rows are prefetched TB_PF rows ahead of the (latency-bound) walk.
        auto walk = [&](unsigned hi, unsigned lo, int st, bool emit_rows) -> int {
            auto emit = [&](unsigned row, int state) {
                if (emit_rows && lane == 0) {
                    if (states) states[tbase + row] = (uint8_t)state;
                    if (states64) states64[tbase + row] = state;
                }
            };
            unsigned row = hi;
            // full groups of TB_PF rows, unconditional so the ring stays in registers:
            // cur[q] = delta[row-1-q]; the next group's rows are in flight meanwhile
            if (row >= lo + 2 * TB_PF) {
                T nxt[TB_PF][NS];
#pragma unroll
                for (int q = 0; q < TB_PF; ++q) load_d(row - 1 - (unsigned)q, nxt[q]);
                while (row >= lo + 2 * TB_PF) {
                    T cur[TB_PF][NS];
#pragma unroll
                    for (int q = 0; q < TB_PF; ++q) {
#pragma unroll
                        for (int s = 0; s < NS; ++s) cur[q][s] = nxt[q][s];
                    }
#pragma unroll
                    for (int q = 0; q < TB_PF; ++q) load_d(row - 1 - TB_PF - (unsigned)q, nxt[q]);
#pragma unroll
                    for (int q = 0; q < TB_PF; ++q) {
                        emit(row - (unsigned)q, st);
                        st = back(row - (unsigned)q, st, cur[q]);
                    }
                    row -= TB_PF;
                }
                // nxt holds the rows of one more full group
#pragma unroll
                for (int q = 0; q < TB_PF; ++q) {
                    emit(row - (unsigned)q, st);
                    st = back(row - (unsigned)q, st, nxt[q]);
                }
                row -= TB_PF;
            }
            for (; row > lo; --row) {
                T dc[NS];
                load_d(row - 1, dc);
                emit(row, st);
                st = back(row, st, dc);
            }
            return st;
        };

        int st;
        if (mode == 1) {
            st = forced_end[ci];
        } else if (ch.t1 == ch.s1) {
            T dv[NS];
            load_d(rlast, dv);
            st = warp_argmax_first<T, NS>(dv, lane);        // np.argmax of the last row
        } else {
            // speculate: enter from `warmup` steps to the right (or the sequence end)
            unsigned rq = rlast + (unsigned)b.warmup;
            const unsigned rseq = (unsigned)(ch.s1 - 1 - tbase);
            if (rq > rseq) rq = rseq;
            T dv[NS];
            load_d(rq, dv);
            st = warp_argmax_first<T, NS>(dv, lane);
            st = walk(rq, rlast, st, false);
        }
        if (lane == 0) spec_end[ci] = (uint8_t)st;

        // walk the chunk: rows rlast ... rfirst; when the chunk has a left neighbour
        // (rfirst == 1) the walk ends on row 0 = t0-1, whose state goes to `pred`
        st = walk(rlast, 0, st, true);
        if (rfirst == 1) {
            if (lane == 0) pred[ci] = (uint8_t)st;
        } else if (lane == 0) {
            if (states) states[tbase] = (uint8_t)st;
            if (states64) states64[tbase] = st;
        }
    }
}

// Traceback, FOUR chunks per warp (fp32, N <= 32, no segment ratios).
// The one-chunk-per-warp walk above spends ~30 issue slots per step on a
// 32-lane arg-max (REDUX + ballot) of which 30 lanes matter.  Here a chunk gets
// eight lanes, each owning four consecutive states: one LDG.128 + one LDS.128
// per step fetch delta[t-1][4u..4u+3] and logA[4u..4u+3][state], the arg-max is
// a 4-way local minimum of bit patterns (every candidate is <= 0, so the largest
// value has the smallest unsigned pattern), three xor-shuffles and one ballot
// (ties: lowest state, as _hmm.pyx:232-247).  ~11 issue slots per chunk step.
#define TB4_PF 8     // delta rows in flight per chunk

template <int NS>
__device__ __forceinline__ int tb4_argmax(float c0, float c1, float c2, float c3, int u, unsigned segshift, int lane0)
{
    const unsigned b0 = __float_as_uint(c0), b1 = __float_as_uint(c1), b2 = __float_as_uint(c2), b3 = __float_as_uint(c3);
    const unsigned m01 = min(b0, b1), m23 = min(b2, b3);
    const int i01 = b1 < b0 ? 1 : 0, i23 = b3 < b2 ? 3 : 2;
    const unsigned ml = min(m01, m23);
    const int il = m23 < m01 ? i23 : i01;
    unsigned mg = ml;
    mg = min(mg, __shfl_xor_sync(TEHMM_FULL, mg, 1));
    mg = min(mg, __shfl_xor_sync(TEHMM_FULL, mg, 2));
    mg = min(mg, __shfl_xor_sync(TEHMM_FULL, mg, 4));
    if (NS == 2) mg = min(mg, __shfl_xor_sync(TEHMM_FULL, mg, 8));
    const unsigned vote = __ballot_sync(TEHMM_FULL, ml == mg);
    const int ulo = __ffs((vote >> segshift) & ((1u << (8 * NS)) - 1u)) - 1;
    return __shfl_sync(TEHMM_FULL, 4 * u + il, lane0 + ulo);
}

// RATIO: the from-state-0 candidate carries the reference's extra term (see viterbi_lean_kernel); the term
// common to all from-states does not move the arg-max.
// NS = 2 (33..64 states, lattice rows of 64 floats; round 2): a chunk gets SIXTEEN lanes, two chunks per warp.
template <bool RATIO, int NS>
__global__ void __launch_bounds__(TEHMM_WARPS_PER_CTA * 32, 4)
vit_traceback4_kernel(TehmmModelDev m, TehmmBatchDev b, const float *__restrict__ lattice,
                      uint8_t *__restrict__ states, int64_t *__restrict__ states64,
                      uint8_t *__restrict__ spec_end, uint8_t *__restrict__ pred,
                      const uint8_t *__restrict__ forced_end, const int *__restrict__ bad, int mode,
                      const double *__restrict__ ratios)
{
    constexpr int NP = 32 * NS, LPC = 8 * NS, CPW = 32 / LPC;       // columns, lanes per chunk, chunks per warp
    __shared__ __align__(16) float AT[NP * NP];            // AT[s*NP + i] = min(logA[i][s], 0)
    for (int e = threadIdx.x; e < NP * NP; e += blockDim.x) {
        const int s = e / NP, i = e % NP;
        AT[e] = fminf((float)m.cut_trans[(int64_t)i * NP + s], 0.f);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = lane / LPC, u = lane % LPC;
    const unsigned segshift = (unsigned)(LPC * c);
    const int lane0 = LPC * c;
    const uint32_t at_lane = (uint32_t)__cvta_generic_to_shared(AT) + (uint32_t)u * 16u;
    const float a00 = (float)m.cut_trans[0];

    for (int64_t wg = (int64_t)blockIdx.x * TEHMM_WARPS_PER_CTA + warp; wg * CPW < b.nchunks;
         wg += (int64_t)gridDim.x * TEHMM_WARPS_PER_CTA) {
        const int64_t ci = wg * CPW + c;
        bool valid = ci < b.nchunks;
        if (valid && mode == 1) valid = bad[ci] != 0;
        int row = 0, rlast = 0, st = 0;
        bool has_pred = false;
        int64_t tbase = 0;
        if (valid) {
            const TehmmChunk ch = b.chunks[ci];
            has_pred = ch.t0 > ch.s0;
            tbase = has_pred ? ch.t0 - 1 : ch.t0;        // row 0 = the left neighbour's last step, if any
            rlast = (int)(ch.t1 - 1 - tbase);
            row = rlast;
            if (mode == 1) st = forced_end[ci];
            else if (ch.t1 < ch.s1)                      // speculate: enter from `warmup` steps to the right
                row = (int)min((int64_t)rlast + b.warmup, ch.s1 - 1 - tbase);
        }
        const float *__restrict__ ll = lattice + tbase * NP + 4 * u;
        {   // np.argmax of the row the walk starts from (not used by forced / invalid slots)
            const float4 dv = *reinterpret_cast<const float4 *>(ll + (int64_t)row * NP);
            const int s0 = tb4_argmax<NS>(dv.x, dv.y, dv.z, dv.w, u, segshift, lane0);
            if (valid && mode == 0) st = s0;
        }
        int spec = st;
        float4 ring[TB4_PF];
        float rring[TB4_PF];                           // RATIO: the ratio of the row the walk stands on
        const double *__restrict__ rr = RATIO ? ratios + tbase : nullptr;
#pragma unroll
        for (int p = 0; p < TB4_PF; ++p) {
            ring[p] = *reinterpret_cast<const float4 *>(ll + (int64_t)max(row - 1 - p, 0) * NP);
            rring[p] = RATIO ? (float)rr[max(row - p, 0)] : 1.f;
        }
        while (__any_sync(TEHMM_FULL, row >= 1)) {
#pragma unroll
            for (int p = 0; p < TB4_PF; ++p) {
                const bool act = row >= 1;
                if (act && row == rlast) spec = st;
                if (act && row <= rlast && u == 0) {
                    states[tbase + row] = (uint8_t)st;
                    if (states64) states64[tbase + row] = st;
                }
                const float4 dv = ring[p];
                const float r = rring[p];
                ring[p] = *reinterpret_cast<const float4 *>(ll + (int64_t)max(row - 1 - TB4_PF, 0) * NP);
                if (RATIO) rring[p] = (float)rr[max(row - TB4_PF, 0)];
                float4 a;
                asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                             : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(at_lane + (uint32_t)st * (uint32_t)(NP * 4)));
                if (RATIO) {
                    // candidate of from-state 0 (lane u = 0, first element): + logA_ss r - [r > 1] logA_ss (r - 1), - logA_00 for s = 0
                    // (r < 0: a sequence without ratios, no correction)
                    const float dgs = AT[st * NP + st];
                    float extra0 = r >= 0.f && dgs > -INFINITY ? (r > 1.f ? dgs : dgs * r) : 0.f;
                    if (r >= 0.f && st == 0 && a00 > -INFINITY) extra0 -= a00;
                    if (u == 0) a.x += extra0;
                }
                const int sn = tb4_argmax<NS>(dv.x + a.x, dv.y + a.y, dv.z + a.z, dv.w + a.w, u, segshift, lane0);
                if (act) { st = sn; row -= 1; }
            }
        }
        if (valid && u == 0) {
            if (rlast == 0) spec = st;
            spec_end[ci] = (uint8_t)spec;
            if (has_pred) pred[ci] = (uint8_t)st;        // the state the left neighbour must end in
            else {
                states[tbase] = (uint8_t)st;
                if (states64) states64[tbase] = st;
            }
        }
    }
}

// bad[c-1] = the end state chunk c-1 assumed differs from the state its right
// neighbour c really reaches at t0-1; the true state is handed to the repair pass.
__global__ void vit_tb_verify_kernel(TehmmBatchDev b, uint8_t *spec_end, const uint8_t *pred,
                                     uint8_t *forced_end, int *bad, int *nbad)
{
    int64_t ci = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= b.nchunks) return;
    const TehmmChunk ch = b.chunks[ci];
    if (ch.t0 > ch.s0) {
        const int flag = spec_end[ci - 1] != pred[ci];
        bad[ci - 1] = flag;
        if (flag) {
            forced_end[ci - 1] = pred[ci];
            spec_end[ci - 1] = pred[ci];
            atomicAdd(nbad, 1);
        }
    }
    if (ch.t1 == ch.s1) bad[ci] = 0;      // last chunk of a sequence: exact by construction
}

// float64 score of the returned path, in the reference's terms
// (_hmm.pyx:222-225, 232-248): one warp per chunk, lanes over time.
template <typename OBS>
__global__ void vit_rescore_kernel(TehmmModelDev m, TehmmBatchDev b, const OBS *__restrict__ obs,
                                   const uint8_t *__restrict__ states,
                                   const double *__restrict__ ratios_em,
                                   const double *__restrict__ ratios_dp,
                                   double *__restrict__ score_part, int64_t lo, int64_t hi)
{
    int64_t ci = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (ci >= b.nchunks) return;
    const TehmmChunk ch = b.chunks[ci];
    const int N = m.N;
    double acc = 0.0;
    // [lo, hi): the rows whose terms are wanted (the whole batch for decode; a core range
    // when one long sequence is sharded in time across ranks, parallel.py)
    for (int64_t t = max(ch.t0, lo) + lane; t < min(ch.t1, hi); t += 32) {
        const int j = states[t];
        double e = 0.0;
        for (int k = 0; k < m.K; ++k)
            e += m.table[((int64_t)k * N + j) * m.S + (int64_t)obs[t * m.K + k]];
        e *= m.normalize;
        if (ratios_em) e *= ratios_em[t];
        const double ajj = m.log_trans[(int64_t)j * N + j];
        double term;
        if (t == ch.s0) {
            term = m.log_start[j] + e;
            if (ratios_dp && ratios_dp[t] > 1.) term += ajj * (ratios_dp[t] - 1.);
        } else {
            const int i = states[t - 1];
            term = m.log_trans[(int64_t)i * N + j] + e;
            if (ratios_dp && ratios_dp[t] >= 0.) {      // negative: a sequence without ratios
                const double r = ratios_dp[t];
                if (i == 0) {
                    term += ajj * r;
                    if (j == 0) term -= m.log_trans[0];
                } else if (r > 1.) {
                    term += ajj * (r - 1.);
                }
            }
        }
        acc += term;
    }
    acc = warp_sum(acc);
    if (lane == 0) score_part[ci] = acc;
}

__global__ void vit_score_reduce_kernel(TehmmBatchDev b, const double *__restrict__ score_part,
                                        double *__restrict__ logprob)
{
    // one block per sequence
    const int64_t s = blockIdx.x;
    double acc = 0.0;
    for (int64_t c = b.seq_chunk0[s] + threadIdx.x; c < b.seq_chunk0[s + 1]; c += blockDim.x) acc += score_part[c];
    acc = block_sum(acc);
    if (threadIdx.x == 0) logprob[s] = acc;
}

template <typename T, int NS>
static cudaError_t launch_vit(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                              const T *elog, const double *ratios, T *lattice, T *start_vec,
                              T *end_vec, const int *bad, int mode, int grid)
{
    if (ratios)
        viterbi_kernel<T, NS, true><<<grid, TEHMM_WARPS_PER_CTA * 32, 0, st>>>(m, b, elog, ratios, lattice, start_vec, end_vec, bad, mode);
    else if (sizeof(T) == 4 && NS == 2) {
        // one CTA per SM either way (the transition matrix alone is 128 registers per lane): twelve warps at <= 168 registers
        const int64_t need = (b.nchunks + VIT_WIDE_WARPS - 1) / VIT_WIDE_WARPS;
        const int g = (int)(need < grid ? need : grid);
        viterbi_kernel<T, NS, false, VIT_WIDE_WARPS><<<g, VIT_WIDE_WARPS * 32, 0, st>>>(m, b, elog, ratios, lattice, start_vec, end_vec, bad, mode);
    } else
        viterbi_kernel<T, NS, false><<<grid, TEHMM_WARPS_PER_CTA * 32, 0, st>>>(m, b, elog, ratios, lattice, start_vec, end_vec, bad, mode);
    return cudaGetLastError();
}

// the DP that can return the log-probability itself (viterbi_lean_kernel's score_part)
bool tehmm_viterbi_dp_scores(const TehmmModelDev &m, int prec, const double *ratios)
{
    return prec == TEHMM_F32 && m.NS == 1 && m.LD == 32 && !ratios;
}

cudaError_t tehmm_launch_viterbi(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                 int prec, const void *elog, const double *ratios, void *lattice,
                                 void *start_vec, void *end_vec, const int *bad, int mode, int grid,
                                 const double *rowmax, double *score_part)
{
    if (prec == TEHMM_F32) {
        if (m.NS == 1 && m.LD == 32) {
            if (ratios)
                viterbi_lean_kernel<true><<<grid, TEHMM_WARPS_PER_CTA * 32, 0, st>>>(m, b, (const float *)elog, (float *)lattice, (float *)start_vec, (float *)end_vec, bad, mode, nullptr, nullptr, ratios);
            else
                viterbi_lean_kernel<false><<<grid, TEHMM_WARPS_PER_CTA * 32, 0, st>>>(m, b, (const float *)elog, (float *)lattice, (float *)start_vec, (float *)end_vec, bad, mode, rowmax, rowmax ? score_part : nullptr, nullptr);
            return cudaGetLastError();
        }
        if (m.NS == 1) return launch_vit<float, 1>(st, m, b, (const float *)elog, ratios, (float *)lattice, (float *)start_vec, (float *)end_vec, bad, mode, grid);
        if (m.LD == 64 && VW_ENABLED) {
            const int64_t need = (b.nchunks + VW_PAIRS - 1) / VW_PAIRS;
            const int g = (int)(need < grid ? need : grid);
            if (ratios)
                viterbi_wide_kernel<true><<<g, VW_PAIRS * 64, 0, st>>>(m, b, (const float *)elog, (float *)lattice, (float *)start_vec, (float *)end_vec, bad, mode, ratios);
            else
                viterbi_wide_kernel<false><<<g, VW_PAIRS * 64, 0, st>>>(m, b, (const float *)elog, (float *)lattice, (float *)start_vec, (float *)end_vec, bad, mode, nullptr);
            return cudaGetLastError();
        }
        return launch_vit<float, 2>(st, m, b, (const float *)elog, ratios, (float *)lattice, (float *)start_vec, (float *)end_vec, bad, mode, grid);
    }
    if (m.NS == 1) return launch_vit<double, 1>(st, m, b, (const double *)elog, ratios, (double *)lattice, (double *)start_vec, (double *)end_vec, bad, mode, grid);
    return launch_vit<double, 2>(st, m, b, (const double *)elog, ratios, (double *)lattice, (double *)start_vec, (double *)end_vec, bad, mode, grid);
}

template <typename T, int NS>
static cudaError_t launch_tb(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                             const T *lattice, const double *ratios, uint8_t *states,
                             int64_t *states64, uint8_t *spec_end, uint8_t *pred,
                             const uint8_t *forced_end, const int *bad, int mode, int grid)
{
    const size_t smem = (size_t)m.NP * m.NP * sizeof(T);
    if (ratios) {
        auto k = vit_traceback_kernel<T, NS, true>;
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k<<<grid, TEHMM_WARPS_PER_CTA * 32, smem, st>>>(m, b, lattice, ratios, states, states64, spec_end, pred, forced_end, bad, mode);
    } else {
        auto k = vit_traceback_kernel<T, NS, false>;
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k<<<grid, TEHMM_WARPS_PER_CTA * 32, smem, st>>>(m, b, lattice, ratios, states, states64, spec_end, pred, forced_end, bad, mode);
    }
    return cudaGetLastError();
}

cudaError_t tehmm_launch_traceback(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                   int prec, const void *lattice, const double *ratios,
                                   uint8_t *states, int64_t *states64, uint8_t *spec_end,
                                   uint8_t *pred, const uint8_t *forced_end, const int *bad,
                                   int mode, int grid)
{
    if (prec == TEHMM_F32) {
        if (m.LD == 32 * m.NS) {
            const int cpw = m.NS == 1 ? 4 : 2;
            const int64_t need = ((b.nchunks + cpw - 1) / cpw + TEHMM_WARPS_PER_CTA - 1) / TEHMM_WARPS_PER_CTA;
            const int g4 = (int)(need < grid ? (need < 1 ? 1 : need) : grid);
            if (m.NS == 1) {
                if (ratios)
                    vit_traceback4_kernel<true, 1><<<g4, TEHMM_WARPS_PER_CTA * 32, 0, st>>>(m, b, (const float *)lattice, states, states64, spec_end, pred, forced_end, bad, mode, ratios);
                else
                    vit_traceback4_kernel<false, 1><<<g4, TEHMM_WARPS_PER_CTA * 32, 0, st>>>(m, b, (const float *)lattice, states, states64, spec_end, pred, forced_end, bad, mode, nullptr);
            } else {
                if (ratios)
                    vit_traceback4_kernel<true, 2><<<g4, TEHMM_WARPS_PER_CTA * 32, 0, st>>>(m, b, (const float *)lattice, states, states64, spec_end, pred, forced_end, bad, mode, ratios);
                else
                    vit_traceback4_kernel<false, 2><<<g4, TEHMM_WARPS_PER_CTA * 32, 0, st>>>(m, b, (const float *)lattice, states, states64, spec_end, pred, forced_end, bad, mode, nullptr);
            }
            return cudaGetLastError();
        }
        if (m.NS == 1) return launch_tb<float, 1>(st, m, b, (const float *)lattice, ratios, states, states64, spec_end, pred, forced_end, bad, mode, grid);
        return launch_tb<float, 2>(st, m, b, (const float *)lattice, ratios, states, states64, spec_end, pred, forced_end, bad, mode, grid);
    }
    if (m.NS == 1) return launch_tb<double, 1>(st, m, b, (const double *)lattice, ratios, states, states64, spec_end, pred, forced_end, bad, mode, grid);
    return launch_tb<double, 2>(st, m, b, (const double *)lattice, ratios, states, states64, spec_end, pred, forced_end, bad, mode, grid);
}

cudaError_t tehmm_launch_tb_verify(cudaStream_t st, const TehmmBatchDev &b, uint8_t *spec_end,
                                   const uint8_t *pred, uint8_t *forced_end, int *bad, int *nbad)
{
    cudaError_t e = cudaMemsetAsync(nbad, 0, sizeof(int), st);
    if (e != cudaSuccess) return e;
    vit_tb_verify_kernel<<<(int)((b.nchunks + 127) / 128), 128, 0, st>>>(b, spec_end, pred, forced_end, bad, nbad);
    return cudaGetLastError();
}

// per-sequence sum of the chunks' shares of the log-probability (viterbi_lean_kernel's score_part)
cudaError_t tehmm_launch_vit_score_reduce(cudaStream_t st, const TehmmBatchDev &b, const double *score_part,
                                          double *logprob)
{
    const int64_t cps = b.nchunks / b.nseq;
    vit_score_reduce_kernel<<<(int)b.nseq, cps >= 2048 ? 1024 : cps >= 256 ? 256 : 64, 0, st>>>(b, score_part, logprob);
    return cudaGetLastError();
}

// float64 re-score of the path: 2 launches
cudaError_t tehmm_launch_rescore(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                 const uint8_t *states, const double *ratios_em,
                                 const double *ratios_dp, double *score_part, double *logprob,
                                 int64_t lo, int64_t hi)
{
    int warps = 4;
    int rgrid = (int)((b.nchunks + warps - 1) / warps);
    if (b.obs_bytes == 1) vit_rescore_kernel<uint8_t><<<rgrid, warps * 32, 0, st>>>(m, b, (const uint8_t *)b.obs, states, ratios_em, ratios_dp, score_part, lo, hi);
    else if (b.obs_bytes == 2) vit_rescore_kernel<uint16_t><<<rgrid, warps * 32, 0, st>>>(m, b, (const uint16_t *)b.obs, states, ratios_em, ratios_dp, score_part, lo, hi);
    else vit_rescore_kernel<int32_t><<<rgrid, warps * 32, 0, st>>>(m, b, (const int32_t *)b.obs, states, ratios_em, ratios_dp, score_part, lo, hi);
    const int64_t cps = b.nchunks / b.nseq;
    vit_score_reduce_kernel<<<(int)b.nseq, cps >= 2048 ? 1024 : cps >= 256 ? 256 : 64, 0, st>>>(b, score_part, logprob);
    return cudaGetLastError();
}
