// Forward and backward passes at 33..64 states on the 5th-generation tensor cores: tcgen05.mma
// with the accumulator AND the state operand in tensor memory (hmm.py:678-729 -> _hmm.pyx:120-198).
//
// At 33..64 states the one-chunk-per-warp kernels (forward.cu, backward.cu) hold 128 registers of
// transition matrix per lane and are issue bound on the mat-vec.  Here a CTA of eight warps advances
// ONE TILE OF 128 CHUNKS (chunk = TMEM lane) per step, TWO threads per chunk:
//
//     D[128 x 64] = X_lo A_hi + X_hi A_lo + X_hi A_hi        24 tcgen05.mma (M128 N64 K8, kind::tf32),
//                                                             issued by one thread, D and X in TMEM,
//                                                             A (hi / lo parts) in shared memory
//     x' = D .* b_t * 2^-shift                                epilogue: tcgen05.ld of the thread's 32 columns,
//                                                             the row maximum from both halves, power-of-two
//                                                             scale with a one-step lag, split into hi / lo,
//                                                             tcgen05.st back as the next X
//
// Warps 0-3 take columns 0-31 of the rows, warps 4-7 columns 32-63 (a warp reaches the 32 tensor-memory
// lanes of its index modulo 4), which halves the serial epilogue between two tensor-core steps; the halves
// of a row exchange their maxima through shared memory behind the step's one CTA barrier.  b rows arrive and
// alpha rows leave as pairs of 3-D tensor-map boxes {32 floats, 1 step, 128 chunks} side by side (SWIZZLE_128B,
// so that a thread reading "its" 128-byte row does not collide with its neighbours), double buffered, one
// elected thread issuing.  Same chunk partition, same speculate / verify / repair protocol, same start_vec /
// end_vec / cscale conventions as forward_kernel, whose alpha lattice this one's is interchangeable with
// (everything downstream is scale free).  Used for the first pass over a batch that is ONE sequence; repairs
// and everything else take the one-chunk-per-warp kernels.
//
// Measured on B200, 10 M steps of one sequence: 1.26 ms against 2.30 ms for forward_kernel at 33, 50 and
// 64 states (DESIGN.md §5, where the measured reason is also given why <= 32 states stay on fwd_tile_kernel).
#include "scan.cuh"
#include <cuda.h>
#include <cstring>
#include <cstdio>

#define UM_ROWS 128
#define UM_NLD 2                      // load buffers
#define UM_NST 2                      // store buffers
// A lattice row is 64 floats: two boxes {32 floats, 1 step, 128 chunks} with the 128-byte swizzle side by side.
constexpr int UM_NP = 64;                                    // lattice row stride, columns of D / X
constexpr int UM_BOX = UM_ROWS * 128;                        // bytes of one box
constexpr int UM_BLK = 2 * UM_BOX;                           // bytes of one block buffer (one step of the tile)
constexpr int UM_BMAT = UM_NP * UM_NP * 4;                   // one part (hi or lo) of the transition matrix
constexpr unsigned UM_TMEM_COLS = 256u;                      // D, X hi, X lo
constexpr int UM_FWD_SMEM = 1024 + (UM_NLD + UM_NST) * UM_BLK + 2 * UM_BMAT + 256 + 2048;

__device__ __forceinline__ void um_mbar_init(uint32_t bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void um_mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
// bounded wait: a protocol error must not hang the GPU.  After ~0.1 s without the phase
// completing the kernel-wide fault flag is raised; once it is up every wait returns at once, so
// all threads keep walking the same barrier sequence to the end and the host reports the error.
__device__ __forceinline__ void um_mbar_wait(uint32_t bar, uint32_t parity, volatile int *fault)
{
    for (unsigned spin = 0; spin < (1u << 22); ++spin) {
        unsigned ok;
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
        if ((spin & 1023u) == 1023u && *fault) return;
    }
    *fault = 1;
}
__device__ __forceinline__ void um_tensor_load3(uint32_t dst, const CUtensorMap *tm, int x, int y, int z, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 :: "r"(dst), "l"(tm), "r"(x), "r"(y), "r"(z), "r"(bar) : "memory");
}
__device__ __forceinline__ void um_tensor_store3(const CUtensorMap *tm, int x, int y, int z, uint32_t src)
{
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];"
                 :: "l"(tm), "r"(x), "r"(y), "r"(z), "r"(src) : "memory");
}
__device__ __forceinline__ void um_tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32"
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void um_tmem_st32(uint32_t taddr, const uint32_t (&v)[32])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0],"
                 "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16,"
                 "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n"
                 :: "r"(taddr),
                    "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
                    "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
                    "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
                    "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
                 : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem descriptor]; one thread issues on behalf of the CTA
__device__ __forceinline__ void um_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %6, %7, %8}, p;\n\t}"
                 :: "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u) : "memory");
}
__device__ __forceinline__ u64 um_fmul2(u64 a, u64 b)
{
    u64 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
// K-major, no swizzle: core matrices of 8 rows x 16 bytes; LBO = bytes between the two 16-byte
// K-chunks of one instruction, SBO = bytes between 8-row groups (cute/atom/mma_traits_sm100.hpp)
__device__ __forceinline__ uint64_t um_smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo)
{
    return (uint64_t)((addr >> 4) & 0x3fff) | ((uint64_t)((lbo >> 4) & 0x3fff) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3fff) << 32) | (1ull << 46);
}

__global__ void __launch_bounds__(UM_ROWS * 2, 1)
fwd_umma_kernel(TehmmModelDev m, TehmmBatchDev b, const float *__restrict__ blin,
                const double *__restrict__ rowmax, float *__restrict__ alpha,
                float *__restrict__ start_vec, float *__restrict__ end_vec, double *__restrict__ cscale,
                const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_a,
                int lf, int nfull, int *__restrict__ fault)
{
    constexpr int NP = UM_NP;
    constexpr uint32_t UMBOX = UM_BOX, UMBLK = UM_BLK, BMAT = UM_BMAT;
    extern __shared__ unsigned char um_raw[];
    const uint32_t raw = (uint32_t)__cvta_generic_to_shared(um_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;                 // SWIZZLE_128B boxes: 1024-byte aligned
    unsigned char *gbase = um_raw + (base - raw);
    const uint32_t ldbuf = base, stbuf = base + UM_NLD * UMBLK, bhi = stbuf + UM_NST * UMBLK, blo = bhi + BMAT;
    const uint32_t bars = blo + BMAT;                             // ld[UM_NLD], mma
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(gbase + (UM_NLD + UM_NST) * UMBLK + 2 * BMAT + 64);
    int *esum_s = reinterpret_cast<int *>(gbase);                 // reused after the main loop (load buffer 0)
    float *mxs = reinterpret_cast<float *>(gbase + (UM_NLD + UM_NST) * UMBLK + 2 * BMAT + 256);   // [parity][half][row]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row = tid % UM_ROWS, hh = tid / UM_ROWS;           // this thread's chunk of the tile and its column half
    constexpr int NTHR = UM_ROWS * 2;
    const int col0 = 32 * hh;                                     // its first column
    const uint32_t boxoff = (uint32_t)hh * UMBOX;                 // the box its columns are in
    const int N = m.N, W = b.warmup;

    // ---- transition matrix, hi / lo TF32 parts, canonical K-major layout: B[n = j][k = i] = A[i][j]
    // (per 16-byte K-chunk: NP rows of 16 bytes; LBO = NP * 16 between the two chunks of one K = 8 instruction,
    //  SBO = 128 between 8-row groups)
    for (int e = tid; e < NP * NP; e += NTHR) {
        const int n = e / NP, k = e % NP;
        const double v = m.lin_trans[(int64_t)k * NP + n];
        uint32_t h;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"((float)v));
        uint32_t l;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"((float)(v - (double)__uint_as_float(h))));
        const uint32_t off = (uint32_t)((k >> 2) * (NP * 16) + (n >> 3) * 128 + (n & 7) * 16 + (k & 3) * 4);
        *reinterpret_cast<uint32_t *>(gbase + (UM_NLD + UM_NST) * UMBLK + off) = h;
        *reinterpret_cast<uint32_t *>(gbase + (UM_NLD + UM_NST) * UMBLK + BMAT + off) = l;
    }
    if (tid == 0) {
        for (int i = 0; i < UM_NLD + 1; ++i) um_mbar_init(bars + 8 * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"((uint32_t)__cvta_generic_to_shared(tmem_slot)), "r"(UM_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // B parts (generic writes) -> tensor core (async proxy)
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    const uint32_t t_d = tmem, t_hi = tmem + NP, t_lo = tmem + 2 * NP;          // column offsets
    const uint32_t my_lane = (uint32_t)((warp & 3) * 32) << 16;                  // this warp's TMEM lanes
    const uint32_t bar_mma = bars + 8 * UM_NLD;
    // kind::tf32, F32 accumulate, A and B K-major, N = NP, M = 128
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (((uint32_t)NP >> 3) << 17) | ((128u >> 4) << 24);

    uint32_t mma_phase = 0, ld_phase = 0;                         // bit i of ld_phase: parity of load barrier i
    volatile int *vfault = fault;
    for (int64_t tile = blockIdx.x; tile * UM_ROWS < b.nchunks; tile += gridDim.x) {
        // ---- this thread's chunk
        const int64_t c = tile * UM_ROWS + row;
        const bool valid = c < b.nchunks;
        TehmmChunk ch = b.chunks[valid ? c : b.nchunks - 1];
        const int64_t dist = ch.t0 - ch.s0;
        const bool first = valid && dist == 0, pred = valid && dist > 0;
        const int len = valid ? (int)(ch.t1 - ch.t0) : 0;
        const int ks = first ? W : 0, ke = W + len;
        const bool boxed = valid && len == lf && c < nfull;      // its rows travel in the boxes
        const int kmax = W + lf;
        const int c0 = (int)(tile * UM_ROWS);
        const float *brow0 = blin + (ch.t0 - W) * NP;            // row of clock 0 (direct path only)
        float *arow0 = alpha ? alpha + (ch.t0 - W) * NP : nullptr;
        const uint32_t line = (uint32_t)row;                      // 128-byte line of this thread's row in a box

        auto issue_load = [&](int k) {                           // thread 0: the b rows of clock k
            const bool warm = k < W;
            const uint32_t bar = bars + 8 * (k % UM_NLD);
            um_mbar_expect_tx(bar, UMBLK);
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2)
                um_tensor_load3(ldbuf + (k % UM_NLD) * UMBLK + h2 * UMBOX, &tmap_b, 32 * h2, warm ? lf - W + k : k - W, c0 - (warm ? 1 : 0), bar);
        };
        if (tid == 0)
            for (int k = 0; k < UM_NLD && k < kmax; ++k) issue_load(k);

        // ---- initial operand: a flat vector (a row that starts its sequence stays empty until clock W)
        uint32_t xh[32], xl[32];
        {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                xh[i] = (valid && !first && col0 + i < N) ? __float_as_uint(1.f) : 0u;
                xl[i] = 0u;
            }
            um_tmem_st32(t_hi + col0 + my_lane, xh);
            um_tmem_st32(t_lo + col0 + my_lane, xl);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        float scp = 1.f;
        int shp = 0, esum = 0;

        auto issue_mma = [&]() {                                 // thread 0, after the CTA barrier
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            constexpr uint32_t LBO = NP * 16, KSTEP = 2 * LBO;
#pragma unroll
            for (int kk = 0; kk < NP / 8; ++kk)
                um_mma_tf32_ts(t_d, t_lo + kk * 8, um_smem_desc(bhi + kk * KSTEP, LBO, 128), idesc, kk > 0);
#pragma unroll
            for (int kk = 0; kk < NP / 8; ++kk)
                um_mma_tf32_ts(t_d, t_hi + kk * 8, um_smem_desc(blo + kk * KSTEP, LBO, 128), idesc, 1);
#pragma unroll
            for (int kk = 0; kk < NP / 8; ++kk)
                um_mma_tf32_ts(t_d, t_hi + kk * 8, um_smem_desc(bhi + kk * KSTEP, LBO, 128), idesc, 1);
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar_mma) : "memory");
        };
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) issue_mma();

        for (int k = 0; k < kmax; ++k) {
            const uint32_t lb = ldbuf + (k % UM_NLD) * UMBLK, sb = stbuf + (k % UM_NST) * UMBLK;
            um_mbar_wait(bars + 8 * (k % UM_NLD), (ld_phase >> (k % UM_NLD)) & 1u, vfault);
            ld_phase ^= 1u << (k % UM_NLD);
            const bool storing = alpha != nullptr && k >= W;
            if (storing && k >= UM_NST) {                        // the store that last used this buffer has read it
                if (tid == 0) asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(UM_NST - 1) : "memory");
                __syncthreads();
            }
            const bool on = valid && k >= ks && k < ke;
            const bool start_here = first && k == ks;
            // D of this clock
            um_mbar_wait(bar_mma, mma_phase, vfault);
            mma_phase ^= 1u;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const u64 sc2 = pk2(scp, scp);
            const int sh_now = start_here ? 0 : shp;
            float mx = 0.f;
            {
                // b row half of this clock: from the box (16-byte chunks XOR-swizzled) or direct
                float bt[32];
                if (boxed) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                                     : "=f"(bt[4 * q]), "=f"(bt[4 * q + 1]), "=f"(bt[4 * q + 2]), "=f"(bt[4 * q + 3])
                                     : "r"(lb + boxoff + line * 128u + (((uint32_t)q ^ (line & 7u)) << 4)) : "memory");
                } else {
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const float4 v = on ? *reinterpret_cast<const float4 *>(brow0 + (int64_t)k * NP + col0 + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
                        bt[4 * q] = v.x; bt[4 * q + 1] = v.y; bt[4 * q + 2] = v.z; bt[4 * q + 3] = v.w;
                    }
                }
                uint32_t dv[32];
                um_tmem_ld32(t_d + col0 + my_lane, dv);
                // x' = D .* b * scale in packed fp32 (FMUL2), maximum as a 3-input tree
                u64 a2[16];
                float m0 = 0.f, m1 = 0.f;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const u64 d2 = ((u64)dv[2 * i + 1] << 32) | (u64)dv[2 * i];
                    a2[i] = um_fmul2(d2, um_fmul2(pk2(bt[2 * i], bt[2 * i + 1]), sc2));
                    if (i & 1) m1 = fmax3(m1, lo2(a2[i]), hi2(a2[i])); else m0 = fmax3(m0, lo2(a2[i]), hi2(a2[i]));
                }
                float mh = fmaxf(m0, m1);
                if (start_here) {                            // alpha_0 = pi .* b_0
                    mh = 0.f;
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const float p0 = (float)m.lin_start[col0 + 2 * i] * bt[2 * i], p1 = (float)m.lin_start[col0 + 2 * i + 1] * bt[2 * i + 1];
                        a2[i] = pk2(p0, p1);
                        mh = fmax3(mh, p0, p1);
                    }
                }
                if (!valid || k < ks) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) a2[i] = 0ull;
                    mh = 0.f;
                }
                mx = fmaxf(mx, mh);
                if (k >= W) {
                    if (alpha) {
                        if (boxed) {
#pragma unroll
                            for (int q = 0; q < 8; ++q)
                                asm volatile("st.shared.v2.u64 [%0], {%1,%2};"
                                             :: "r"(sb + boxoff + line * 128u + (((uint32_t)q ^ (line & 7u)) << 4)), "l"(a2[2 * q]), "l"(a2[2 * q + 1]) : "memory");
                        } else if (valid && k < ke) {
#pragma unroll
                            for (int q = 0; q < 8; ++q)
                                *reinterpret_cast<ulonglong2 *>(arow0 + (int64_t)k * NP + col0 + 4 * q) = make_ulonglong2(a2[2 * q], a2[2 * q + 1]);
                        }
                    }
                } else if (k == W - 1 && pred) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<ulonglong2 *>(start_vec + c * NP + col0 + 4 * q) = make_ulonglong2(a2[2 * q], a2[2 * q + 1]);
                }
                if (valid && k + 1 == ke) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<ulonglong2 *>(end_vec + c * NP + col0 + 4 * q) = make_ulonglong2(a2[2 * q], a2[2 * q + 1]);
                }
                // next operand: hi = the 11 leading bits (a TF32 number), lo = the rest, exactly (FFMA2: a - hi)
                const u64 neg1 = pk2(-1.f, -1.f);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const u64 h2 = a2[i] & 0xffffe000ffffe000ull;
                    const u64 l2 = ffma2(h2, neg1, a2[i]);
                    xh[2 * i] = (uint32_t)h2; xh[2 * i + 1] = (uint32_t)(h2 >> 32);
                    xl[2 * i] = (uint32_t)l2; xl[2 * i + 1] = (uint32_t)(l2 >> 32);
                }
                um_tmem_st32(t_hi + col0 + my_lane, xh);
                um_tmem_st32(t_lo + col0 + my_lane, xl);
            }
            mxs[((k & 1) * 2 + hh) * UM_ROWS + row] = mx;       // the other half of the row reads it behind the barrier
            if (k >= W) esum += k < ke ? sh_now : 0;
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // alpha rows -> TMA store
            __syncthreads();
            mx = fmaxf(mx, mxs[((k & 1) * 2 + (hh ^ 1)) * UM_ROWS + row]);
            {   // exact power-of-two scale for the NEXT step (scale_of in tile.cu)
                const unsigned mb = __float_as_uint(mx);
                scp = __uint_as_float(0x7f000000u - (mb & 0x7f800000u));
                shp = (int)(mb >> 23) - 127;
            }
            if (tid == 0 && k + 1 < kmax) issue_mma();
            if (tid == 0) {
                if (storing) {
#pragma unroll
                    for (int h2 = 0; h2 < 2; ++h2)
                        um_tensor_store3(&tmap_a, 32 * h2, k - W, c0, sb + h2 * UMBOX);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
                if (k + UM_NLD < kmax) issue_load(k + UM_NLD);           // every thread has passed the barrier after reading lb
            }
        }
        if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __syncthreads();

        // ---- log of everything taken out of each chunk: exponents and row maxima
        if (hh == 0) esum_s[row] = esum;
        __syncthreads();
        for (int rr = warp; rr < UM_ROWS; rr += NTHR / 32) {
            const int64_t cc = tile * UM_ROWS + rr;
            if (cc >= b.nchunks) break;
            const TehmmChunk c2 = b.chunks[cc];
            double ms = 0.0;
            for (int64_t tt = c2.t0 + lane; tt < c2.t1; tt += 32) ms += rowmax[tt];
            ms = warp_sum(ms);
            if (lane == 0) cscale[cc] = (double)esum_s[rr] * 0.6931471805599453094 + ms;
        }
        __syncthreads();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(UM_TMEM_COLS) : "memory");
}

// [chunk][step][64 floats] view, boxes {32, 1, 128}, 128-byte swizzle
static bool um_make_tmap(CUtensorMap *tm, const float *base, int64_t lf, int64_t nfull)
{
    typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static encode_fn encode = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            encode = (encode_fn)fn;
        else
            cudaGetLastError();
    }
    if (!encode || nfull < 1 || lf < 1) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)UM_NP, (cuuint64_t)lf, (cuuint64_t)nfull};
    const cuuint64_t strides[2] = {(cuuint64_t)(4 * UM_NP), (cuuint64_t)lf * 4 * UM_NP};
    const cuuint32_t box[3] = {32, 1, UM_ROWS}, estr[3] = {1, 1, 1};
    return encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void *)base, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// whether this batch / pass can take the tcgen05 forward kernel: 33..64 states, one sequence, first pass
bool tehmm_forward_umma_ok(const TehmmModelDev &m, const TehmmBatchDev &b, int mode, int64_t fine_len)
{
    return m.NS == 2 && b.nseq == 1 && mode == 0 && fine_len >= b.warmup && b.total / fine_len >= 1;
}

// ------------------------------------------------------------------ backward twin (33..64 states)
// The backward recursion in the same shape, run right to left (hmm.py:715-729 -> _hmm.pyx:160-198, the
// posterior glue basehmm.py:265-272,357).  With X the operand row (b_{t+1} .* beta'_{t+1}, scaled) the
// accumulator of a clock IS beta'_t = X A^T (the transition matrix is staged transposed), so the epilogue of
// clock k (time t = t1 - 1 + W - k) reads D, b_t and alpha_t of the SAME row:
//     next X   = D .* b_t * 2^-shift                         (exactly fwd_umma_kernel's epilogue)
//     p        = D .* alpha_t,  Z = sum p                    posterior = p / Z, MAP state = argmax p
// Two threads per chunk (column halves) exchange their partial Z / best / arg-max through shared memory across
// the step's one CTA barrier, next to the row maximum; the normalisation, the MAP byte and the posterior rows
// are written BEHIND the barrier, while the tensor core runs the next clock.  The posterior rows overwrite the
// alpha box they were computed from (same thread, same addresses) and leave as one tensor-map store per
// clock; alpha buffers cycle load -> read -> overwrite -> store -> reload (three of them).  First pass of a
// single-sequence batch only; repairs and transition counts stay with backward_kernel (backward.cu), whose
// start_vec / end_vec / map_part conventions these are.
#define UM_NA 3
constexpr int UM_XCH = 4 * 2 * 2 * UM_ROWS * 4;          // row maximum, Z, best, arg-max: [parity][half][row]
constexpr int UM_BWD_SMEM = 1024 + (UM_NLD + UM_NA) * UM_BLK + 2 * UM_BMAT + 256 + UM_XCH;

__global__ void __launch_bounds__(UM_ROWS * 2, 1)
bwd_umma_kernel(TehmmModelDev m, TehmmBatchDev b, int flags, const float *__restrict__ blin,
                const float *__restrict__ alpha, float *__restrict__ post, uint8_t *__restrict__ map_states,
                double *__restrict__ map_part, float *__restrict__ start_vec, float *__restrict__ end_vec,
                const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_a,
                const __grid_constant__ CUtensorMap tmap_p, int lf, int nfull, int *fault)
{
    constexpr int NP = UM_NP, NH = 2;                             // NH: column halves of a row, one thread each
    constexpr uint32_t UMBOX = UM_BOX, UMBLK = UM_BLK, BMAT = UM_BMAT;
    constexpr int OFF_MAT = (UM_NLD + UM_NA) * UM_BLK, OFF_BAR = OFF_MAT + 2 * UM_BMAT;
    extern __shared__ unsigned char um_raw[];
    const uint32_t raw = (uint32_t)__cvta_generic_to_shared(um_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char *gbase = um_raw + (base - raw);
    const uint32_t bbuf = base, abuf = base + UM_NLD * UMBLK, bhi = base + OFF_MAT, blo = bhi + BMAT;
    const uint32_t bars = base + OFF_BAR;                         // b[UM_NLD], alpha[UM_NA], mma
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(gbase + OFF_BAR + 64);
    float *mxs = reinterpret_cast<float *>(gbase + OFF_BAR + 256);
    float *zs = mxs + 2 * NH * UM_ROWS, *bests = zs + 2 * NH * UM_ROWS;
    int *idxs = reinterpret_cast<int *>(bests + 2 * NH * UM_ROWS);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int row = tid % UM_ROWS, hh = tid / UM_ROWS;
    constexpr int NTHR = UM_ROWS * NH;
    const int N = m.N, W = b.warmup;
    const bool want_post = (flags & TEHMM_BWD_POSTERIORS) != 0 && post != nullptr;
    const bool want_map = (flags & TEHMM_BWD_MAP) != 0 && map_states != nullptr;
    const bool renorm = (flags & TEHMM_BWD_RENORM_EPS) != 0;
    const float eps32 = 1.1920928955078125e-07f;
    const double renorm_inv = 1.0 / (1.0 + (double)N * 1.1920928955078125e-07);
    const float renorm_invf = (float)renorm_inv;

    // ---- transition matrix TRANSPOSED, hi / lo TF32 parts, canonical K-major layout: B[n = i][k = j] = A[i][j]
    for (int e = tid; e < NP * NP; e += NTHR) {
        const int n = e / NP, k = e % NP;
        const double v = m.lin_trans[(int64_t)n * NP + k];
        uint32_t h;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"((float)v));
        uint32_t l;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"((float)(v - (double)__uint_as_float(h))));
        const uint32_t off = (uint32_t)((k >> 2) * (NP * 16) + (n >> 3) * 128 + (n & 7) * 16 + (k & 3) * 4);
        *reinterpret_cast<uint32_t *>(gbase + OFF_MAT + off) = h;
        *reinterpret_cast<uint32_t *>(gbase + OFF_MAT + BMAT + off) = l;
    }
    if (tid == 0) {
        for (int i = 0; i < UM_NLD + UM_NA + 1; ++i) um_mbar_init(bars + 8 * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"((uint32_t)__cvta_generic_to_shared(tmem_slot)), "r"(UM_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    const uint32_t t_d = tmem, t_hi = tmem + NP, t_lo = tmem + 2 * NP;
    const uint32_t my_lane = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t bar_a0 = bars + 8 * UM_NLD, bar_mma = bars + 8 * (UM_NLD + UM_NA);
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (((uint32_t)NP >> 3) << 17) | ((128u >> 4) << 24);

    uint32_t mma_phase = 0, b_phase = 0, a_phase = 0;
    volatile int *vfault = fault;
    for (int64_t tile = blockIdx.x; tile * UM_ROWS < b.nchunks; tile += gridDim.x) {
        const int64_t c = tile * UM_ROWS + row;
        const bool valid = c < b.nchunks;
        const TehmmChunk ch = b.chunks[valid ? c : b.nchunks - 1];
        const int64_t rem = ch.s1 - ch.t1;                        // steps of the sequence to the right of the chunk
        const bool succ = valid && rem > 0;
        const bool exact = valid && rem <= (int64_t)W;            // beta_{T-1} = 1 is within reach (_hmm.pyx:179)
        const int len = valid ? (int)(ch.t1 - ch.t0) : 0;
        const int ks = exact ? W - (int)rem : 0, ke = W + len;
        const bool own_boxed = valid && c < nfull;                // its own rows travel in the boxes
        const bool warm_boxed = valid && c + 1 < nfull;           // and so do the warm-up rows (chunk c + 1)
        const int kmax = W + lf;
        const int c0 = (int)(tile * UM_ROWS);
        const int64_t trow = ch.t1 - 1 + W;                       // time of clock 0
        const float *bclk0 = blin + trow * NP + 32 * hh;
        const float *aclk0 = alpha + trow * NP + 32 * hh;
        float *pclk0 = want_post ? post + trow * NP + 32 * hh : nullptr;
        uint8_t *mclk0 = want_map ? map_states + trow : nullptr;
        double mapsum = 0.0;

        auto issue_b = [&](int j) {                               // thread 0: b rows of clock j
            const uint32_t bar = bars + 8 * (j % UM_NLD);
            um_mbar_expect_tx(bar, UMBLK);
#pragma unroll
            for (int h2 = 0; h2 < NH; ++h2)
                um_tensor_load3(bbuf + (j % UM_NLD) * UMBLK + h2 * UMBOX, &tmap_b, 32 * h2, j < W ? W - 1 - j : lf - 1 - (j - W),
                                j < W ? c0 + 1 : c0, bar);
        };
        auto issue_a = [&](int ja) {                              // thread 0: alpha rows of clock W + ja
            const uint32_t bar = bar_a0 + 8 * (ja % UM_NA);
            um_mbar_expect_tx(bar, UMBLK);
#pragma unroll
            for (int h2 = 0; h2 < NH; ++h2)
                um_tensor_load3(abuf + (ja % UM_NA) * UMBLK + h2 * UMBOX, &tmap_a, 32 * h2, lf - 1 - ja, c0, bar);
        };
        if (tid == 0) {
            for (int j = 0; j < UM_NLD && j < kmax; ++j) issue_b(j);
            for (int ja = 0; ja < UM_NA && ja < lf; ++ja) issue_a(ja);
        }

        uint32_t xh[32], xl[32];
        {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                xh[i] = (valid && !exact && 32 * hh + i < N) ? __float_as_uint(1.f) : 0u;     // speculate from a flat vector
                xl[i] = 0u;
            }
            um_tmem_st32(t_hi + 32 * hh + my_lane, xh);
            um_tmem_st32(t_lo + 32 * hh + my_lane, xl);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        float scp = 1.f;

        auto issue_mma = [&]() {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            constexpr uint32_t LBO = NP * 16, KSTEP = 2 * LBO;
#pragma unroll
            for (int kk = 0; kk < NP / 8; ++kk)
                um_mma_tf32_ts(t_d, t_lo + kk * 8, um_smem_desc(bhi + kk * KSTEP, LBO, 128), idesc, kk > 0);
#pragma unroll
            for (int kk = 0; kk < NP / 8; ++kk)
                um_mma_tf32_ts(t_d, t_hi + kk * 8, um_smem_desc(blo + kk * KSTEP, LBO, 128), idesc, 1);
#pragma unroll
            for (int kk = 0; kk < NP / 8; ++kk)
                um_mma_tf32_ts(t_d, t_hi + kk * 8, um_smem_desc(bhi + kk * KSTEP, LBO, 128), idesc, 1);
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar_mma) : "memory");
        };
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) issue_mma();

        for (int k = 0; k < kmax; ++k) {
            const bool warm = k < W;
            const int ja = k - W;
            const uint32_t lb = bbuf + (k % UM_NLD) * UMBLK + hh * UMBOX;
            const uint32_t ab = abuf + ((ja < 0 ? 0 : ja) % UM_NA) * UMBLK + hh * UMBOX;
            um_mbar_wait(bars + 8 * (k % UM_NLD), (b_phase >> (k % UM_NLD)) & 1u, vfault);
            b_phase ^= 1u << (k % UM_NLD);
            if (!warm) {
                um_mbar_wait(bar_a0 + 8 * (ja % UM_NA), (a_phase >> (ja % UM_NA)) & 1u, vfault);
                a_phase ^= 1u << (ja % UM_NA);
            }
            const uint32_t line = (uint32_t)row;
            const bool on = valid && k >= ks && k < ke;
            const bool start_here = exact && k == ks;
            const bool boxed = warm ? warm_boxed : own_boxed;
            const int par = k & 1;
            float bt[32];
            if (boxed) {
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                                 : "=f"(bt[4 * q]), "=f"(bt[4 * q + 1]), "=f"(bt[4 * q + 2]), "=f"(bt[4 * q + 3])
                                 : "r"(lb + line * 128u + (((uint32_t)q ^ (line & 7u)) << 4)) : "memory");
            } else {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 v = on ? *reinterpret_cast<const float4 *>(bclk0 - (int64_t)k * NP + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
                    bt[4 * q] = v.x; bt[4 * q + 1] = v.y; bt[4 * q + 2] = v.z; bt[4 * q + 3] = v.w;
                }
            }
            um_mbar_wait(bar_mma, mma_phase, vfault);
            mma_phase ^= 1u;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t dv[32];
            um_tmem_ld32(t_d + 32 * hh + my_lane, dv);            // beta'_t, this thread's half of the row
            if (start_here) {                                     // the sequence's last step: beta = 1
#pragma unroll
                for (int i = 0; i < 32; ++i) dv[i] = 32 * hh + i < N ? __float_as_uint(1.f) : 0u;
            }
            const float scn = start_here ? 1.f : scp;
            const u64 sc2 = pk2(scn, scn);
            u64 a2[16];
            float m0 = 0.f, m1 = 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const u64 d2 = ((u64)dv[2 * i + 1] << 32) | (u64)dv[2 * i];
                a2[i] = um_fmul2(d2, um_fmul2(pk2(bt[2 * i], bt[2 * i + 1]), sc2));
                if (i & 1) m1 = fmax3(m1, lo2(a2[i]), hi2(a2[i])); else m0 = fmax3(m0, lo2(a2[i]), hi2(a2[i]));
            }
            float mx = fmaxf(m0, m1);
            if (!valid || k < ks) {
#pragma unroll
                for (int i = 0; i < 16; ++i) a2[i] = 0ull;
                mx = 0.f;
            }
            {
                const u64 neg1 = pk2(-1.f, -1.f);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const u64 h2 = a2[i] & 0xffffe000ffffe000ull;
                    const u64 l2 = ffma2(h2, neg1, a2[i]);
                    xh[2 * i] = (uint32_t)h2; xh[2 * i + 1] = (uint32_t)(h2 >> 32);
                    xl[2 * i] = (uint32_t)l2; xl[2 * i + 1] = (uint32_t)(l2 >> 32);
                }
                um_tmem_st32(t_hi + 32 * hh + my_lane, xh);
                um_tmem_st32(t_lo + 32 * hh + my_lane, xl);
            }
            mxs[(par * NH + hh) * UM_ROWS + row] = mx;
            // chunk boundary vectors (beta' itself, any scale: the verification is ratio based)
            if (k == W - 1 && succ && k >= ks) {
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    *reinterpret_cast<uint4 *>(start_vec + c * NP + 32 * hh + 4 * q) = make_uint4(dv[4 * q], dv[4 * q + 1], dv[4 * q + 2], dv[4 * q + 3]);
            }
            if (valid && k + 1 == ke) {
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    *reinterpret_cast<uint4 *>(end_vec + c * NP + 32 * hh + 4 * q) = make_uint4(dv[4 * q], dv[4 * q + 1], dv[4 * q + 2], dv[4 * q + 3]);
            }
            // products with alpha_t: this half's share of Z, its best state
            float p[32];
            float zown = 0.f, bown = 0.f;
            int iown = 99;
            const bool outp = valid && !warm && k < ke;
            if (!warm) {
                float at[32];
                if (own_boxed) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                                     : "=f"(at[4 * q]), "=f"(at[4 * q + 1]), "=f"(at[4 * q + 2]), "=f"(at[4 * q + 3])
                                     : "r"(ab + line * 128u + (((uint32_t)q ^ (line & 7u)) << 4)) : "memory");
                } else {
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const float4 v = outp ? *reinterpret_cast<const float4 *>(aclk0 - (int64_t)k * NP + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
                        at[4 * q] = v.x; at[4 * q + 1] = v.y; at[4 * q + 2] = v.z; at[4 * q + 3] = v.w;
                    }
                }
                float z0 = 0.f, z1 = 0.f, b0 = 0.f, b1 = 0.f;
#pragma unroll
                for (int i = 0; i < 32; i += 2) {
                    p[i] = __uint_as_float(dv[i]) * at[i];
                    p[i + 1] = __uint_as_float(dv[i + 1]) * at[i + 1];
                    z0 += p[i]; z1 += p[i + 1];
                    if (i & 2) b1 = fmax3(b1, p[i], p[i + 1]); else b0 = fmax3(b0, p[i], p[i + 1]);
                }
                const float best = fmaxf(b0, b1);
                int idx = 99;
                if (want_map) {
#pragma unroll
                    for (int i = 31; i >= 0; --i)
                        if (p[i] == best) idx = 32 * hh + i;       // lowest state among the maxima (np.argmax, basehmm.py:357)
                }
                zs[(par * NH + hh) * UM_ROWS + row] = z0 + z1;
                bests[(par * NH + hh) * UM_ROWS + row] = best;
                idxs[(par * NH + hh) * UM_ROWS + row] = idx;
                zown = z0 + z1; bown = best; iown = idx;
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            mx = fmaxf(mx, mxs[(par * NH + (hh ^ 1)) * UM_ROWS + row]);
            {
                const unsigned mb = __float_as_uint(mx);
                scp = __uint_as_float(0x7f000000u - (mb & 0x7f800000u));
            }
            if (tid == 0 && k + 1 < kmax) issue_mma();
            if (!warm) {
                int idx = iown;
                float Z = zown, best = bown;
                const float zo = zs[(par * NH + (hh ^ 1)) * UM_ROWS + row];
                const float bo = bests[(par * NH + (hh ^ 1)) * UM_ROWS + row];
                const int io = idxs[(par * NH + (hh ^ 1)) * UM_ROWS + row];
                Z = hh == 0 ? Z + zo : zo + Z;                // the same sum in both halves
                if (bo > best || (bo == best && io < idx)) { best = bo; idx = io; }
                const float invZ = __frcp_rn(Z);
                if (want_map && hh == 0 && outp) {
                    mclk0[-(int64_t)k] = (uint8_t)(idx < N ? idx : 0);
                    const float bg = best * invZ;
                    mapsum += renorm ? ((double)bg + (double)eps32) * renorm_inv : (double)bg;
                }
                if (want_post) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        p[i] *= invZ;
                        if (renorm) p[i] = 32 * hh + i < N ? (p[i] + eps32) * renorm_invf : 0.f;      // padding stays zero
                    }
                    if (own_boxed) {
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};"
                                         :: "r"(ab + line * 128u + (((uint32_t)q ^ (line & 7u)) << 4)),
                                            "f"(p[4 * q]), "f"(p[4 * q + 1]), "f"(p[4 * q + 2]), "f"(p[4 * q + 3]) : "memory");
                    } else if (outp) {
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            *reinterpret_cast<float4 *>(pclk0 - (int64_t)k * NP + 4 * q) = make_float4(p[4 * q], p[4 * q + 1], p[4 * q + 2], p[4 * q + 3]);
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // posterior rows -> TMA store (behind the next barrier)
                }
            }
            if (tid == 0) {
                if (k + UM_NLD < kmax) issue_b(k + UM_NLD);      // every thread has read this clock's b rows before the barrier
                if (!warm) {
                    if (want_post) {
                        if (ja >= 1) {
                            if (ja >= 2) {
                                // the store of clock ja - 2 (issued a whole clock ago) has read its buffer: reload it
                                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                                if (ja + 1 < lf) issue_a(ja + 1);
                            }
#pragma unroll
                            for (int h2 = 0; h2 < NH; ++h2)
                                um_tensor_store3(&tmap_p, 32 * h2, lf - ja, c0, abuf + ((ja - 1) % UM_NA) * UMBLK + h2 * UMBOX);
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                    } else if (ja + UM_NA < lf) {
                        issue_a(ja + UM_NA);                      // nothing overwrites the alpha rows: reload at once
                    }
                }
            }
        }
        if (want_post) {
            __syncthreads();                                       // the last clock's rows are in shared memory
            if (tid == 0) {
#pragma unroll
                for (int h2 = 0; h2 < NH; ++h2)
                    um_tensor_store3(&tmap_p, 32 * h2, 0, c0, abuf + ((lf - 1) % UM_NA) * UMBLK + h2 * UMBOX);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            }
        }
        if (want_map && hh == 0 && valid) map_part[c] = mapsum;
        __syncthreads();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(UM_TMEM_COLS) : "memory");
}

bool tehmm_backward_umma_ok(const TehmmModelDev &m, const TehmmBatchDev &b, int flags, int mode, int64_t fine_len)
{
    return m.NS == 2 && b.nseq == 1 && mode == 0 && !(flags & TEHMM_BWD_TRANS) && fine_len >= b.warmup &&
           b.total / fine_len >= 1;
}

cudaError_t tehmm_launch_backward_umma(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b, int flags,
                                       const float *blin, const float *alpha, float *post, uint8_t *map_states,
                                       double *map_part, float *start_vec, float *end_vec, int sms,
                                       int64_t fine_len, int *fault)
{
    CUtensorMap tb, ta, tp;
    memset(&tb, 0, sizeof tb);
    memset(&ta, 0, sizeof ta);
    memset(&tp, 0, sizeof tp);
    const int64_t nfull = b.total / fine_len;
    const bool want_post = (flags & TEHMM_BWD_POSTERIORS) != 0 && post != nullptr;
    if (!um_make_tmap(&tb, blin, fine_len, nfull) || !um_make_tmap(&ta, alpha, fine_len, nfull) ||
        (want_post && !um_make_tmap(&tp, post, fine_len, nfull)))
        return cudaErrorNotSupported;
    cudaError_t e = cudaFuncSetAttribute(bwd_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_BWD_SMEM);
    if (e != cudaSuccess) return e;
    const int64_t tiles = (b.nchunks + UM_ROWS - 1) / UM_ROWS;
    const int grid = (int)(tiles < (int64_t)sms ? tiles : (int64_t)sms);
    bwd_umma_kernel<<<grid, UM_ROWS * 2, UM_BWD_SMEM, st>>>(m, b, flags, blin, alpha, post, map_states, map_part, start_vec, end_vec,
                                                        tb, ta, tp, (int)fine_len, (int)nfull, fault);
    return cudaGetLastError();
}

cudaError_t tehmm_launch_forward_umma(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                      const float *blin, const double *rowmax, float *alpha,
                                      float *start_vec, float *end_vec, double *cscale, int sms,
                                      int64_t fine_len, int *fault)
{
    CUtensorMap tb, ta;
    memset(&tb, 0, sizeof tb);
    memset(&ta, 0, sizeof ta);
    const int64_t nfull = b.total / fine_len;
    if (!um_make_tmap(&tb, blin, fine_len, nfull) || (alpha && !um_make_tmap(&ta, alpha, fine_len, nfull)))
        return cudaErrorNotSupported;
    cudaError_t e = cudaFuncSetAttribute(fwd_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, UM_FWD_SMEM);
    if (e != cudaSuccess) return e;
    const int64_t tiles = (b.nchunks + UM_ROWS - 1) / UM_ROWS;
    const int grid = (int)(tiles < (int64_t)sms ? tiles : (int64_t)sms);
    fwd_umma_kernel<<<grid, UM_ROWS * 2, UM_FWD_SMEM, st>>>(m, b, blin, rowmax, alpha, start_vec, end_vec, cscale, tb, ta,
                                                            (int)fine_len, (int)nfull, fault);
    return cudaGetLastError();
}
