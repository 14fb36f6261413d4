// Tensor-core forward / backward passes: SIXTEEN chunks per warp.
// (hmm.py:678-729 -> _hmm.pyx:120-198; basehmm.py:265-272,357-358)
//
// forward.cu / backward.cu give one chunk of the time axis to one warp and do
// the N x N mat-vec with 16 FFMA2 + 8 LDS.128 per step: ~70-100 issue slots per
// time step, which is what bounds them.  Here a warp owns a TILE of 16 chunks
// and advances all of them one time step with one 16 x 32 x 32 matrix product
//     X'[chunk][j] = sum_i X[chunk][i] A[i][j]
// on the tensor cores (mma.sync.m16n8k8 TF32, fp32 accumulate).  TF32 alone
// (10-bit mantissa) is far outside the 1e-5 contract, so every product is the
// usual three-term split  x_hi A_hi + x_lo A_hi + x_hi A_lo  with x = x_hi + x_lo
// exactly (Veltkamp split, packed fp32): 48 MMAs per tile step = 3 per chunk
// step, ~2^-21 relative error per step, and the filter does not accumulate it.
//
// Register layout (g = lane/4, q = lane%4): the lane holds, for tile rows g and
// g+8, the EIGHT CONSECUTIVE states 8q .. 8q+7.  The accumulator fragment of
// n-tile nt (columns n = 2q, 2q+1) is mapped to states 8q+2nt, 8q+2nt+1, so
//   * a row of b / alpha / posteriors (LD = 32 floats = one 128-byte line) is
//     read and written as two 16-byte accesses per lane, a quad covering the row;
//   * the accumulator fragment of n-tile kt IS the A-operand fragment of
//     k-tile kt of the next step (k-slot q <-> state 8q+2kt, slot q+4 <-> state
//     8q+2kt+1): the recursion never leaves registers, no shuffles, no smem.
// The state vector is kept as packed (row g, row g+8) pairs per state, which is
// both the A-operand register order and the operand shape of FFMA2 / FMUL2.
// The transition matrix lives in registers as B-operand fragments permuted
// accordingly (64 registers: hi and lo parts).
//
// Rows of b (and alpha) are staged global -> shared with cp.async, several time
// steps ahead of the recursion; each lane stages and reads back only its own
// values, so no barrier is involved.
//
// Chunks of one tile run in lock step on a common clock k: row r processes
// time t0_r - W + k (forward) or t1_r - 1 + W - k (backward), W = warm-up
// length, so the speculative warm-up is k < W for every row and outputs start
// at k = W.  Rows that start late (sequence start inside the warm-up window),
// end early (ragged chunks) or are not selected by a repair pass are masked:
// their loads are zero-filled and their stores predicated off.  Row starts and
// ends are handled as rare, warp-uniform "events" outside the steady-state step.
//
// Scaling is by exact powers of two like canonicalise() in scan.cuh, but LAGGED
// by one step: step k multiplies by the scale derived from the row maximum of
// step k-1 (folded into b), which takes the max-reduction off the critical
// path.  The stored vectors are then normalised to within one step's shrinkage
// of [1,2) instead of exactly; everything downstream (posteriors, verify_kernel,
// forward_logprob_kernel) is scale free or carries the exponent explicitly, so
// either implementation can consume the other's alpha lattice.
//
// Speculate / verify / repair and the start_vec / end_vec / cscale conventions
// are those of forward.cu and backward.cu.
//
// Requires fp32, N <= 32 (lattice row stride LD = 32), no segment ratios;
// everything else takes the one-chunk-per-warp kernels.
// Algorithmic HBM bytes per step: forward 4N read + 4N written, backward 8N read
// (+4N posteriors, +1 MAP state).
#include "scan.cuh"
#include <type_traits>
#include <cuda.h>
#include <cstring>

#define TILE_WARPS 8
#define TEHMM_TILE_TENSOR 1     // 3-D tensor-map block loads where the batch is one regularly chunked sequence
// Measured on B200 (10 M x 30, forward with / without the alpha store, ms):
//   per-lane LDGSTS + STG.128 0.887 / 0.525;  TB=2,NBL=4,NBS=2 0.845 / 0.738;
//   TB=4,NBL=2,NBS=1 0.668 / 0.542  -- small bulk copies are TMA issue bound.
#define FWD_NBL 2       // forward: bulk-load block buffers (TB time steps each)
#define FWD_NBS 1       // forward: bulk-store block buffers
#define BWD_STAGES 5    // time steps of b and alpha staged ahead
#define TILE_STAGE_BYTES 2048   // per warp per stage: 16 rows x 128 bytes
#define TILE_NEVER 0x7fffffff

struct TransFrag {
    uint32_t hi[4][4][2];   // [k-tile][n-tile][b0,b1]
    uint32_t lo[4][4][2];
};

__device__ __forceinline__ uint32_t tf32_rna(float x)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ u64 fmul2(u64 a, u64 b)
{
    u64 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint32_t lo32(u64 v) { return (uint32_t)v; }
__device__ __forceinline__ uint32_t hi32(u64 v) { return (uint32_t)(v >> 32); }

__device__ __forceinline__ void mma_tf32(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2,
                                         uint32_t a3, uint32_t b0, uint32_t b1)
{
    asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// B-operand fragments of the (zero padded, 32 x 32) linear transition matrix.
// forward:  D[r][j] = sum_i X[r][i] A[i][j]   -> B[k = i][n = j] = A[i][j]
// backward: D[r][i] = sum_j W[r][j] A[i][j]   -> B[k = j][n = i] = A[i][j]
template <bool BACKWARD>
__device__ __forceinline__ void load_trans(const TehmmModelDev &m, int g, int q, TransFrag &A)
{
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            const int sn = 8 * (g >> 1) + 2 * nt + (g & 1);   // state of output column n = g
            const int sk = 8 * q + 2 * kt;                    // state of k-slot q (slot q+4: sk+1)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const double v = BACKWARD ? m.lin_trans[(int64_t)sn * 32 + sk + e]
                                          : m.lin_trans[(int64_t)(sk + e) * 32 + sn];
                const uint32_t h = tf32_rna((float)v);
                A.hi[kt][nt][e] = h;
                A.lo[kt][nt][e] = tf32_rna((float)(v - (double)__uint_as_float(h)));
            }
        }
    }
}

// The tile's state: xp[c] = (row g, row g+8) values of state 8q + c, packed.
// acc[nt] = accumulator fragment of n-tile nt = (row g: states 8q+2nt, +1; row g+8: same).
__device__ __forceinline__ void tile_matmul(const u64 (&xp)[8], const TransFrag &A, float (&acc)[4][4])
{
    // Veltkamp split, two rows at a time: hi has 11 significant bits (a TF32
    // number), lo = x - hi exactly; the tensor core drops lo's last two bits.
    const u64 C = pk2(8193.f, 8193.f), M1 = pk2(-1.f, -1.f);
    u64 xh[8], xl[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const u64 t = fmul2(xp[c], C);
        const u64 d = ffma2(xp[c], M1, t);      // t - x
        xh[c] = ffma2(d, M1, t);                // t - (t - x)
        xl[c] = ffma2(xh[c], M1, xp[c]);        // x - hi
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
    // small terms first; the four n-tiles are independent accumulator chains
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
            mma_tf32(acc[nt], lo32(xl[2 * kt]), hi32(xl[2 * kt]), lo32(xl[2 * kt + 1]), hi32(xl[2 * kt + 1]),
                     A.hi[kt][nt][0], A.hi[kt][nt][1]);
    }
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
            mma_tf32(acc[nt], lo32(xh[2 * kt]), hi32(xh[2 * kt]), lo32(xh[2 * kt + 1]), hi32(xh[2 * kt + 1]),
                     A.lo[kt][nt][0], A.lo[kt][nt][1]);
    }
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
            mma_tf32(acc[nt], lo32(xh[2 * kt]), hi32(xh[2 * kt]), lo32(xh[2 * kt + 1]), hi32(xh[2 * kt + 1]),
                     A.hi[kt][nt][0], A.hi[kt][nt][1]);
    }
}

// maximum / sum over the 32 states of a tile row (the four lanes of a quad)
__device__ __forceinline__ float quad_max(float v)
{
    v = fmaxf(v, __shfl_xor_sync(TEHMM_FULL, v, 1));
    return fmaxf(v, __shfl_xor_sync(TEHMM_FULL, v, 2));
}
__device__ __forceinline__ float quad_sum(float v)
{
    v += __shfl_xor_sync(TEHMM_FULL, v, 1);
    return v + __shfl_xor_sync(TEHMM_FULL, v, 2);
}

// Exact power-of-two scale that would put a (positive, finite) row maximum m
// into [1,2): sc = 2^-(e-127), sh = e-127 with e the biased exponent.  A zero or
// subnormal maximum gets 2^127 (lifts subnormals, keeps zeros); the exponent of
// a masked row is never used.
__device__ __forceinline__ void scale_of(float m, float &sc, int &sh)
{
    const unsigned mb = __float_as_uint(m);
    sc = __uint_as_float(0x7f000000u - (mb & 0x7f800000u));
    sh = (int)(mb >> 23) - 127;
}

__device__ __forceinline__ void load_vec32(const float *p, float (&v)[8])
{
    const float4 a = *reinterpret_cast<const float4 *>(p);
    const float4 c = *reinterpret_cast<const float4 *>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
}
// row h (0: tile row g, 1: tile row g+8) of the packed state
__device__ __forceinline__ void store_row_vec32(float *p, const u64 (&xp)[8], int h)
{
    float v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) v[c] = h ? hi2(xp[c]) : lo2(xp[c]);
    *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4 *>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void set_row(u64 (&xp)[8], int h, const float (&v)[8])
{
#pragma unroll
    for (int c = 0; c < 8; ++c) xp[c] = h ? pk2(lo2(xp[c]), v[c]) : pk2(v[c], hi2(xp[c]));
}

// Row staging: global -> shared with cp.async (LDGSTS), 16 bytes per lane (rows
// are LD = 32 floats = one 128-byte line, so a quad reads half a row per
// instruction).  Register prefetch rings do not work here: the loads of several
// steps share hardware scoreboards, so waiting for the oldest waits for the
// newest (ncu: 70% of the stall samples were long-scoreboard on the first use);
// cp.async completion is tracked per commit group instead.  Slot layout
// [row][half][lane] x 16 bytes: every LDGSTS.128 and every read-back LDS.128
// covers 512 consecutive bytes (no bank conflicts).  Masked rows are zero-filled
// (src-size 0: the address is not accessed); padding columns hold zeros in HBM.
__device__ __forceinline__ void stage_row(uint32_t slot, const float *src, bool on)
{
    const int nbytes = on ? 16 : 0;
#pragma unroll
    for (int h = 0; h < 2; ++h)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                     :: "r"(slot + (uint32_t)(h * 512)), "l"(src + 4 * h), "r"(nbytes) : "memory");
}
__device__ __forceinline__ void stage_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_> __device__ __forceinline__ void stage_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N_) : "memory"); }
__device__ __forceinline__ void stage_read(uint32_t slot, float (&v)[8])
{
#pragma unroll
    for (int h = 0; h < 2; ++h)
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(v[4 * h]), "=f"(v[4 * h + 1]), "=f"(v[4 * h + 2]), "=f"(v[4 * h + 3])
                     : "r"(slot + (uint32_t)(h * 512)) : "memory");
}
// a lattice row slice (states 8q..8q+7, padding included) as two 16-byte stores
__device__ __forceinline__ void store_row8(float *p, bool on, const float (&v)[8])
{
    if (on) {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4 *>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
}

// ---- bulk asynchronous copies (TMA, 1-D) and mbarriers, per warp ----------------
// A tile row's lattice rows of consecutive time steps are consecutive in HBM
// (LD = 32 floats = 128 bytes each, 16-byte aligned), so one cp.async.bulk moves
// a row's next TB steps into shared memory; 16 lanes issue the 16 rows of a
// block, completion is counted in bytes on a per-warp mbarrier.  Outputs go the
// other way (st.shared, then cp.async.bulk shared -> global).  Compared with
// per-lane LDGSTS / STG (8 cache lines per instruction, address registers held
// until the LSU has read them) this takes the global traffic off the LSU queue:
// the per-lane path spent two thirds of its time in mio_throttle / scoreboard
// stalls (profiles/).
#define TB 4                          // time steps per bulk block
#define TMA_RS (TB * 128 + 16)        // bytes between tile rows of a block (pad: conflict-free LDS.128)
#define TMA_BUF (16 * TMA_RS)         // bytes of one block buffer
#define FWD_WARP_BYTES ((((FWD_NBL + FWD_NBS) * TMA_BUF + 64) + 127) & ~127)   // per warp, 128-byte aligned (tensor copies)

__device__ __forceinline__ void mbar_init(uint32_t bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "WAIT_%=:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE_%=;\n\t"
                 "bra WAIT_%=;\n\t"
                 "DONE_%=:\n\t}" :: "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// One 3-D tensor-map copy moves a whole block: box {32 floats, TB steps, 16 chunks} of the lattice
// seen as [chunk][step][32] (a single sequence cut into equal chunks IS that array).  One lane,
// one instruction, instead of sixteen per-row bulk copies whose uniform-register operands are
// set up in a sixteen-trip loop (40 % of this kernel's stall samples, profiles/r01_notes_v3.md).
__device__ __forceinline__ void tensor_load3(uint32_t dst, const CUtensorMap *tm, int x, int y, int z, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 :: "r"(dst), "l"(tm), "r"(x), "r"(y), "r"(z), "r"(bar) : "memory");
}
__device__ __forceinline__ void tensor_store3(const CUtensorMap *tm, int x, int y, int z, uint32_t src)
{
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];"
                 :: "l"(tm), "r"(x), "r"(y), "r"(z), "r"(src) : "memory");
}
__device__ __forceinline__ void bulk_store(void *dst, uint32_t src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N_> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(N_) : "memory"); }
template <int N_> __device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" :: "n"(N_) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void lds128(uint32_t a, float (&v)[8], int o)
{
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v[o]), "=f"(v[o + 1]), "=f"(v[o + 2]), "=f"(v[o + 3]) : "r"(a) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, float x, float y, float z, float w)
{
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" :: "r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}

// ------------------------------------------------------------------ forward
__global__ void __launch_bounds__(TILE_WARPS * 32, 1)
fwd_tile_kernel(TehmmModelDev m, TehmmBatchDev b, const float *__restrict__ blin,
                const double *__restrict__ rowmax, float *__restrict__ alpha,
                float *__restrict__ start_vec, float *__restrict__ end_vec,
                double *__restrict__ cscale, const int *__restrict__ bad, int mode,
                const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_a,
                int tm_lf, int tm_nfull)
{
    // tm_lf > 0: blin is also described by tmap_b as [tm_nfull chunks][tm_lf steps][32] (one sequence,
    // full-length chunks only); tiles inside that range load their blocks with one tensor copy
    extern __shared__ __align__(128) unsigned char tile_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int N = m.N, W = b.warmup;
    constexpr int LD = 32;                        // lattice row stride (TehmmModelDev::LD for N <= 32)
    // per warp: FWD_NBL load buffers, FWD_NBS store buffers, FWD_NBL mbarriers
    constexpr int WARP_BYTES = FWD_WARP_BYTES;
    const uint32_t wbase = (uint32_t)__cvta_generic_to_shared(tile_smem) + (uint32_t)(warp * WARP_BYTES);
    const uint32_t sbase = wbase + FWD_NBL * TMA_BUF;
    const uint32_t bars = sbase + FWD_NBS * TMA_BUF;
    // where this lane reads / writes its tile rows g and g+8 inside a block buffer
    const uint32_t myoff = (uint32_t)(g * TMA_RS + 32 * q);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < FWD_NBL; ++i) mbar_init(bars + 8 * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    __syncwarp();
    uint32_t nblk_done = 0;                       // load blocks consumed so far by this warp (barrier phases)

    TransFrag A;
    load_trans<false>(m, g, q, A);
    float pi[8], ones[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        pi[i] = (float)m.lin_start[8 * q + i];
        ones[i] = 8 * q + i < N ? 1.f : 0.f;
    }

    const int64_t ngroups = (b.nchunks + 15) / 16;
    for (int64_t gi = (int64_t)blockIdx.x * TILE_WARPS + warp; gi < ngroups;
         gi += (int64_t)gridDim.x * TILE_WARPS) {
        // ---- schedule of the lane's two tile rows
        int ks[2], ke[2];
        int64_t cid[2];
        bool first[2], pred[2];
        int kb = TILE_NEVER, kmax = 0;
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int64_t c = gi * 16 + g + 8 * r;
            cid[r] = c;
            bool valid = c < b.nchunks;
            if (valid && mode == 1) valid = bad[c] != 0;
            ks[r] = TILE_NEVER; ke[r] = 0; first[r] = false; pred[r] = false;
            if (valid) {
                const TehmmChunk ch = b.chunks[c];
                const int64_t dist = ch.t0 - ch.s0;
                pred[r] = dist > 0;
                // mode 1 takes a sequence's first chunk only when the sequence continues one before the batch
                // (tehmm_set_boundary): it starts from the entry vector in start_vec like any repaired chunk
                if (dist == 0 && mode == 0) { ks[r] = W; first[r] = true; }
                else if (mode == 1) ks[r] = W;                       // from the true vector at t0-1
                else if (dist <= W) { ks[r] = W - (int)dist; first[r] = true; }
                else ks[r] = 0;                                      // speculate from a flat vector
                ke[r] = W + (int)(ch.t1 - ch.t0);
                kb = min(kb, ks[r]);
                kmax = max(kmax, ke[r]);
            }
        }
        kb = __reduce_min_sync(TEHMM_FULL, kb);
        kmax = __reduce_max_sync(TEHMM_FULL, kmax);
        if (kmax <= 0) continue;

        // ---- the tile row this lane moves with bulk copies (lanes 0..15: row = lane)
        int oks = TILE_NEVER, oke = 0;
        int64_t ooff = 0;                          // element offset of the row of clock 0
        {
            const int64_t c = gi * 16 + lane;
            bool valid = lane < 16 && c < b.nchunks;
            if (valid && mode == 1) valid = bad[c] != 0;
            if (valid) {
                const TehmmChunk ch = b.chunks[c];
                const int64_t dist = ch.t0 - ch.s0;
                if (dist == 0 || mode == 1) oks = W;
                else if (dist <= W) oks = W - (int)dist;
                else oks = 0;
                oke = W + (int)(ch.t1 - ch.t0);
                ooff = (ch.t0 - W) * LD;
            }
        }
        const int nblk = (kmax - kb + TB - 1) / TB;
        // a tile of sixteen full-length chunks of the one sequence, first pass: tensor copies
        const bool tens = tm_lf > 0 && mode == 0 && kb == 0 && (W % TB) == 0 && W <= tm_lf && gi * 16 + 15 < (int64_t)tm_nfull;   // W <= lf: the warm-up lies in ONE chunk to the left
        const uint32_t rs = tens ? (uint32_t)(TB * 128) : (uint32_t)TMA_RS;      // bytes between tile rows in a load buffer
        // bulk-load the b rows of block j (clocks kb + j*TB ...) into buffer (nblk_done + j) % FWD_NBL
        auto issue_load = [&](int j) {
            const uint32_t slot = (nblk_done + (uint32_t)j) % FWD_NBL;
            const int k0 = kb + j * TB;
            if (tens) {
                // clocks before W read the tail of the chunk to the left: the same box one chunk up
                // (chunk -1, left of the first tile, is out of bounds: zero fill for a row that has not started)
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    mbar_expect_tx(bars + 8 * slot, 16u * TB * 128u);
                    const bool warm = k0 < W;
                    tensor_load3(wbase + slot * TMA_BUF, &tmap_b, 0, warm ? tm_lf - W + k0 : k0 - W,
                                 (int)(gi * 16) - (warm ? 1 : 0), bars + 8 * slot);
                }
                return;
            }
            const int a = max(k0, oks), e = min(k0 + TB, oke);
            const uint32_t bytes = e > a ? (uint32_t)(e - a) * 128u : 0u;
            const uint32_t total = __reduce_add_sync(TEHMM_FULL, bytes);
            fence_async_smem();                   // earlier reads of this buffer are done (WAR across proxies)
            if (lane == 0) mbar_expect_tx(bars + 8 * slot, total);
            __syncwarp();
            if (bytes)
                bulk_load(wbase + slot * TMA_BUF + (uint32_t)(lane * TMA_RS + (a - k0) * 128),
                          blin + ooff + (int64_t)a * LD, bytes, bars + 8 * slot);
        };
        // bulk-store the alpha rows of block j from store buffer j % FWD_NBS
        auto issue_store = [&](int j) {
            const int k0 = kb + j * TB;
            const int a = max(k0, W), e = min(min(k0 + TB, oke), kmax);
            fence_async_smem();                   // st.shared above -> visible to the async proxy
            __syncwarp();
            if (tens) {                           // every row of a regular tile is live for W <= k < W + lf:
                if (lane == 0) {                  // one box; steps beyond the chunk are clipped by the map
                    tensor_store3(&tmap_a, 0, k0 - W, (int)(gi * 16), sbase + (uint32_t)((j % FWD_NBS) * TMA_BUF));
                    bulk_commit();
                }
                return;
            }
            if (lane < 16) {
                if (e > a)
                    bulk_store(alpha + ooff + (int64_t)a * LD,
                               sbase + (uint32_t)((j % FWD_NBS) * TMA_BUF + lane * TMA_RS + (a - k0) * 128),
                               (uint32_t)(e - a) * 128u);
                bulk_commit();
            }
        };

        // next clock >= k at which some row of the tile starts or ends
        auto next_event = [&](int k) -> int {
            int e = TILE_NEVER;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (ks[r] >= k) e = min(e, ks[r]);
                if (ke[r] - 1 >= k) e = min(e, ke[r] - 1);
            }
            return __reduce_min_sync(TEHMM_FULL, e);
        };

        u64 xp[8];                      // state, packed (row g, row g+8)
        float scp[2] = {1.f, 1.f};      // scale to apply at the next step
        int shp[2] = {0, 0}, esum[2] = {0, 0};
#pragma unroll
        for (int c = 0; c < 8; ++c) xp[c] = 0ull;

        for (int j = 0; j < FWD_NBL - 1 && j < nblk; ++j) issue_load(j);
        int kev = next_event(kb);
        // One block of TB clocks.  EVC (compile time): a row may start or end inside this block; the
        // blocks in between run the copy without that code (see bwd_tile_kernel's clock_step).
        auto block_step = [&](const int j, auto evtag) {
            constexpr bool EVC = decltype(evtag)::value;
            if (j + FWD_NBL - 1 < nblk) issue_load(j + FWD_NBL - 1);
            const uint32_t slot = (nblk_done + (uint32_t)j) % FWD_NBL;
            mbar_wait(bars + 8 * slot, ((nblk_done + (uint32_t)j) / FWD_NBL) & 1u);
            const uint32_t lbuf = wbase + slot * TMA_BUF + (tens ? (uint32_t)(g * TB * 128 + 32 * q) : myoff);
            const uint32_t sbuf = sbase + (uint32_t)((j % FWD_NBS) * TMA_BUF) + (tens ? (uint32_t)(g * TB * 128 + 32 * q) : myoff);
            const bool storing = alpha != nullptr && kb + j * TB + TB > W;
            if (storing && j >= FWD_NBS) {         // the bulk store that last used this buffer has read it
                if (lane < 16) bulk_wait_read<FWD_NBS - 1>();
                __syncwarp();
            }
#pragma unroll
            for (int s = 0; s < TB; ++s) {
                const int k = kb + j * TB + s;
                if (k >= kmax) break;
                float bt[2][8];
                lds128(lbuf + s * 128, bt[0], 0);
                lds128(lbuf + s * 128 + 16, bt[0], 4);
                lds128(lbuf + s * 128 + 8 * rs, bt[1], 0);
                lds128(lbuf + s * 128 + 8 * rs + 16, bt[1], 4);
                const bool ev = EVC && k == kev;      // warp uniform, rare
                if (ev) {
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        if (k == ks[r]) {             // the row starts here
                            float v[8];
                            if (mode == 1 && !first[r]) load_vec32(start_vec + cid[r] * 32 + 8 * q, v);
                            else {
#pragma unroll
                                for (int i = 0; i < 8; ++i) v[i] = ones[i];
                            }
                            set_row(xp, r, v);
                            scp[r] = 1.f; shp[r] = 0;
                        }
                    }
                }
                // ---- the step: x <- (x A) .* (b * 2^-shp)
                u64 bs[2][4];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    const u64 s2 = pk2(scp[r], scp[r]);
#pragma unroll
                    for (int p = 0; p < 4; ++p) bs[r][p] = fmul2(pk2(bt[r][2 * p], bt[r][2 * p + 1]), s2);
                }
                float acc[4][4];
                tile_matmul(xp, A, acc);
                float m0 = 0.f, m1 = 0.f;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const float a0 = acc[nt][0] * lo2(bs[0][nt]), a1 = acc[nt][1] * hi2(bs[0][nt]);
                    const float c0 = acc[nt][2] * lo2(bs[1][nt]), c1 = acc[nt][3] * hi2(bs[1][nt]);
                    xp[2 * nt] = pk2(a0, c0);
                    xp[2 * nt + 1] = pk2(a1, c1);
                    m0 = fmax3(m0, a0, a1);
                    m1 = fmax3(m1, c0, c1);
                }
                int sh_now[2] = {shp[0], shp[1]};     // exponents applied in this step
                if (ev) {
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        if (k == ks[r] && first[r]) {  // alpha_0 = pi .* b_0
                            float v[8];
                            float mm = 0.f;
#pragma unroll
                            for (int i = 0; i < 8; ++i) { v[i] = pi[i] * bt[r][i]; mm = fmaxf(mm, v[i]); }
                            set_row(xp, r, v);
                            if (r == 0) m0 = mm; else m1 = mm;
                            sh_now[r] = 0;
                        }
                    }
                }
                scale_of(quad_max(m0), scp[0], shp[0]);
                scale_of(quad_max(m1), scp[1], shp[1]);
                if (k >= W) {
                    esum[0] += k < ke[0] ? sh_now[0] : 0;
                    esum[1] += k < ke[1] ? sh_now[1] : 0;
                    if (alpha) {                       // masked rows stage garbage that is never copied out
                        sts128(sbuf + s * 128, lo2(xp[0]), lo2(xp[1]), lo2(xp[2]), lo2(xp[3]));
                        sts128(sbuf + s * 128 + 16, lo2(xp[4]), lo2(xp[5]), lo2(xp[6]), lo2(xp[7]));
                        sts128(sbuf + s * 128 + 8 * rs, hi2(xp[0]), hi2(xp[1]), hi2(xp[2]), hi2(xp[3]));
                        sts128(sbuf + s * 128 + 8 * rs + 16, hi2(xp[4]), hi2(xp[5]), hi2(xp[6]), hi2(xp[7]));
                    }
                } else if (k == W - 1 && mode == 0) {
#pragma unroll
                    for (int r = 0; r < 2; ++r)
                        if (pred[r] && k >= ks[r] && k < ke[r]) store_row_vec32(start_vec + cid[r] * 32 + 8 * q, xp, r);
                }
                if (ev) {
#pragma unroll
                    for (int r = 0; r < 2; ++r)
                        if (k + 1 == ke[r]) store_row_vec32(end_vec + cid[r] * 32 + 8 * q, xp, r);
                    kev = next_event(k + 1);
                }
            }
            if (storing) issue_store(j);
        };
        for (int j = 0; j < nblk; ++j) {
            if (kev < kb + (j + 1) * TB) block_step(j, std::true_type());
            else block_step(j, std::false_type());
        }
        nblk_done += (uint32_t)nblk;
        if (alpha) {
            if (lane < 16) bulk_wait<0>();         // the stores have left shared memory and are complete
            __syncwarp();
        }

        // log of everything taken out of each chunk: exponents and row maxima
        for (int rr = 0; rr < 16; ++rr) {
            const int64_t c = gi * 16 + rr;
            if (c >= b.nchunks) break;
            if (mode == 1 && !bad[c]) continue;
            const TehmmChunk ch = b.chunks[c];
            double ms = 0.0;
            for (int64_t tt = ch.t0 + lane; tt < ch.t1; tt += 32) ms += rowmax[tt];
            ms = warp_sum(ms);
            const int e = __shfl_sync(TEHMM_FULL, (rr & 8) ? esum[1] : esum[0], (rr & 7) * 4);
            if (lane == 0) cscale[c] = (double)e * 0.6931471805599453094 + ms;
        }
    }
}

// ------------------------------------------------------------------ backward
// OUT = TEHMM_BWD_POSTERIORS | TEHMM_BWD_MAP (compile time)
template <int OUT>
__global__ void __launch_bounds__(TILE_WARPS * 32, 1)
bwd_tile_kernel(TehmmModelDev m, TehmmBatchDev b, int flags, const float *__restrict__ blin,
                const float *__restrict__ alpha, float *__restrict__ post,
                uint8_t *__restrict__ map_states, double *__restrict__ map_part,
                float *__restrict__ start_vec, float *__restrict__ end_vec,
                const int *__restrict__ bad, int mode)
{
    constexpr bool want_post = (OUT & TEHMM_BWD_POSTERIORS) != 0;
    constexpr bool want_map = (OUT & TEHMM_BWD_MAP) != 0;
    extern __shared__ __align__(128) unsigned char tile_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int N = m.N, W = b.warmup;
    constexpr int LD = 32;
    // per stage: b rows then alpha rows
    const uint32_t slot0 = (uint32_t)__cvta_generic_to_shared(tile_smem) +
                           (uint32_t)(warp * BWD_STAGES * 2 * TILE_STAGE_BYTES + lane * 16);
    constexpr bool renorm = (OUT & TEHMM_BWD_RENORM_EPS) != 0;      // compile time: no branch in the posterior epilogue
    const float eps32 = 1.1920928955078125e-07f;
    const double renorm_inv = 1.0 / (1.0 + (double)N * 1.1920928955078125e-07);
    const float renorm_invf = (float)renorm_inv;

    TransFrag A;
    load_trans<true>(m, g, q, A);
    float ones[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) ones[i] = 8 * q + i < N ? 1.f : 0.f;

    const int64_t ngroups = (b.nchunks + 15) / 16;
    for (int64_t gi = (int64_t)blockIdx.x * TILE_WARPS + warp; gi < ngroups;
         gi += (int64_t)gridDim.x * TILE_WARPS) {
        // ---- schedule: at clock k the row is at time t1 - 1 + W - k
        int ks[2], ke[2], kbv[2];      // kbv: first clock whose b_{t+1} exists
        int64_t off[2], trow[2], cid[2];
        bool exact[2], succ[2];
        int kb = TILE_NEVER, kmax = 0;
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int64_t c = gi * 16 + g + 8 * r;
            cid[r] = c;
            bool valid = c < b.nchunks;
            if (valid && mode == 1) valid = bad[c] != 0;
            ks[r] = TILE_NEVER; ke[r] = 0; kbv[r] = TILE_NEVER; off[r] = 0; trow[r] = 0;
            exact[r] = false; succ[r] = false;
            if (valid) {
                const TehmmChunk ch = b.chunks[c];
                const int64_t rem = ch.s1 - ch.t1;                   // steps of the sequence after the chunk
                succ[r] = rem > 0;
                if (rem == 0) { ks[r] = W; exact[r] = true; }        // beta_{T-1}: _hmm.pyx:179 (1/N applied later)
                else if (mode == 1) ks[r] = W;                       // from the true vector at t1
                else if (rem <= W) { ks[r] = W - (int)rem; exact[r] = true; }
                else ks[r] = 0;                                      // speculate from a flat vector
                kbv[r] = exact[r] ? ks[r] + 1 : ks[r];
                ke[r] = W + (int)(ch.t1 - ch.t0);
                trow[r] = ch.t1 - 1 + W;
                off[r] = trow[r] * LD + 8 * q;
                kb = min(kb, ks[r]);
                kmax = max(kmax, ke[r]);
            }
        }
        kb = __reduce_min_sync(TEHMM_FULL, kb);
        kmax = __reduce_max_sync(TEHMM_FULL, kmax);
        if (kmax <= 0) continue;

        auto next_event = [&](int k) -> int {
            int e = TILE_NEVER;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (ks[r] >= k) e = min(e, ks[r]);
                if (ke[r] - 1 >= k) e = min(e, ke[r] - 1);
            }
            return __reduce_min_sync(TEHMM_FULL, e);
        };

        u64 up[8];                      // beta'_{t+1}, packed (row g, row g+8), scaled with a one-step lag
        float scp[2] = {1.f, 1.f};
        double mapsum[2] = {0.0, 0.0};
#pragma unroll
        for (int c = 0; c < 8; ++c) up[c] = 0ull;

        const float *lb[2], *la[2];     // rows b_{t+1} and alpha_t of the next clock to stage
        float *pp_[2];                  // posterior row of the current clock
        uint8_t *mp_[2];                // MAP state of the current clock
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            lb[r] = blin + off[r] + LD - (int64_t)kb * LD;
            la[r] = alpha + off[r] - (int64_t)kb * LD;
            pp_[r] = want_post ? post + off[r] - (int64_t)kb * LD : nullptr;
            mp_[r] = want_map ? map_states + trow[r] - kb : nullptr;
        }
        auto issue = [&](int k, int stage) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const uint32_t sl = slot0 + (uint32_t)(stage * 2 * TILE_STAGE_BYTES + r * 1024);
                stage_row(sl, lb[r], k >= kbv[r] && k < ke[r]);
                stage_row(sl + TILE_STAGE_BYTES, la[r], k >= W && k < ke[r]);
                lb[r] -= LD;
                la[r] -= LD;
            }
            stage_commit();
        };

        // Posterior output of ONE clock from its products pr = alpha_t .* beta'_t (both tile rows packed).
        // Called one clock late (`back` = 1: the output pointers have moved on by one row), between the
        // issue of the next clock's MMAs and the first use of their accumulators: the shuffles, the
        // reciprocal, the arg-max and the stores then overlap the tensor-core latency instead of adding to it.
        u64 prq[8];
        bool actq[2] = {false, false}, pend = false;
        auto post_out = [&](const u64 (&pr)[8], const bool (&actr)[2], int back) {
            u64 zs = 0ull;
#pragma unroll
            for (int c = 0; c < 8; ++c) zs = fadd2(zs, pr[c]);
            const float Z0 = quad_sum(lo2(zs)), Z1 = quad_sum(hi2(zs));
            const float invZ[2] = {__frcp_rn(Z0), __frcp_rn(Z1)};
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const bool act = actr[r];
                float p[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) p[c] = r ? hi2(pr[c]) : lo2(pr[c]);
                if constexpr (want_map) {
                    // argmax with the lowest state winning ties (np.argmax, basehmm.py:357)
                    const float best = quad_max(fmaxf(fmax3(fmax3(p[0], p[1], p[2]), p[3], p[4]), fmax3(p[5], p[6], p[7])));
                    int idx = 99;
#pragma unroll
                    for (int i = 7; i >= 0; --i)
                        if (p[i] == best) idx = 8 * q + i;
                    idx = min(idx, __shfl_xor_sync(TEHMM_FULL, idx, 1));
                    idx = min(idx, __shfl_xor_sync(TEHMM_FULL, idx, 2));
                    // every lane of the quad keeps the (identical) running score: no divergent branch
                    const float bg = act ? best * invZ[r] : 0.f;
                    mapsum[r] += renorm ? (act ? ((double)bg + (double)eps32) * renorm_inv : 0.0) : (double)bg;
                    if (act && q == 0) mp_[r][back] = (uint8_t)(idx < N ? idx : 0);
                }
                if constexpr (want_post) {
                    float gv[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        gv[i] = p[i] * invZ[r];
                        if (renorm) gv[i] = (gv[i] + eps32) * renorm_invf * ones[i];   // padding stays zero
                    }
                    store_row8(pp_[r] + (int64_t)back * LD, act, gv);
                }
            }
        };

#pragma unroll
        for (int v = 0; v < BWD_STAGES - 1; ++v) issue(kb + v, v);
        int rs = 0, ws = BWD_STAGES - 1;
        int kev = next_event(kb);
        // One clock.  EV (compile time): this clock may start or end a row.  The clocks between two
        // events run the EV = false copy, which has no conditional update of `up` in it: with the
        // event code inside the hot loop the compiler re-materialised `up` every clock (ncu: ~50 of
        // 390 instructions per clock were moves and predicated-off event code).
        auto clock_step = [&](const int k, auto evtag) {
            constexpr bool EVC = decltype(evtag)::value;
            issue(k + BWD_STAGES - 1, ws);
            stage_wait<BWD_STAGES - 1>();
            float at[2][8], bt[2][8];
            const uint32_t sl = slot0 + (uint32_t)(rs * 2 * TILE_STAGE_BYTES);
            stage_read(sl, bt[0]);
            stage_read(sl + 1024, bt[1]);
            stage_read(sl + TILE_STAGE_BYTES, at[0]);
            stage_read(sl + TILE_STAGE_BYTES + 1024, at[1]);
            const bool ev = EVC;
            if constexpr (EVC) {
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    if (k == ks[r] && !exact[r]) {
                        float v[8];
                        if (mode == 1) load_vec32(start_vec + cid[r] * 32 + 8 * q, v);
                        else {
#pragma unroll
                            for (int i = 0; i < 8; ++i) v[i] = ones[i];
                        }
                        set_row(up, r, v);
                        scp[r] = 1.f;
                    }
                }
            }
            // ---- w = (b_{t+1} 2^-sh) .* beta'_{t+1};  beta'_t = w A^T
            u64 wp[8];
            {
                u64 bs[2][4];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    const u64 s2 = pk2(scp[r], scp[r]);
#pragma unroll
                    for (int p = 0; p < 4; ++p) bs[r][p] = fmul2(pk2(bt[r][2 * p], bt[r][2 * p + 1]), s2);
                }
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    // scalar multiplies: their operands sit in an MMA accumulator quad and an LDS.128 quad,
                    // neither pairs up as (row g, row g+8) without moves (ncu: 70 IMAD.MOV per clock before)
                    wp[2 * p] = pk2(lo2(up[2 * p]) * lo2(bs[0][p]), hi2(up[2 * p]) * lo2(bs[1][p]));
                    wp[2 * p + 1] = pk2(lo2(up[2 * p + 1]) * hi2(bs[0][p]), hi2(up[2 * p + 1]) * hi2(bs[1][p]));
                }
            }
            float acc[4][4];
            tile_matmul(wp, A, acc);
            if (pend) post_out(prq, actq, 1);        // the previous clock's posterior, behind this clock's MMAs
            float m0 = 0.f, m1 = 0.f;
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                up[2 * nt] = pk2(acc[nt][0], acc[nt][2]);
                up[2 * nt + 1] = pk2(acc[nt][1], acc[nt][3]);
                m0 = fmax3(m0, acc[nt][0], acc[nt][1]);
                m1 = fmax3(m1, acc[nt][2], acc[nt][3]);
            }
            if constexpr (EVC) {
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    if (k == ks[r] && exact[r]) {    // the sequence's last step: beta = 1
                        set_row(up, r, ones);
                        if (r == 0) m0 = 1.f; else m1 = 1.f;
                    }
                }
            }
            {
                int dummy;
                scale_of(quad_max(m0), scp[0], dummy);
                scale_of(quad_max(m1), scp[1], dummy);
            }
            if (k >= W) {
                // posterior of time t: gamma = alpha_t .* beta'_t / Z.  Only the products are formed
                // here; the reductions, the arg-max and the stores of this clock are issued behind
                // the NEXT clock's MMAs (post_out above), off the recursion's critical path.
#pragma unroll
                for (int c = 0; c < 8; ++c) prq[c] = pk2(lo2(up[c]) * at[0][c], hi2(up[c]) * at[1][c]);
                actq[0] = k < ke[0];
                actq[1] = k < ke[1];
                pend = true;
            } else if (k == W - 1 && mode == 0) {
#pragma unroll
                for (int r = 0; r < 2; ++r)
                    if (succ[r] && k >= ks[r] && k < ke[r]) store_row_vec32(start_vec + cid[r] * 32 + 8 * q, up, r);
            }
            if constexpr (EVC) {
#pragma unroll
                for (int r = 0; r < 2; ++r)
                    if (k + 1 == ke[r]) store_row_vec32(end_vec + cid[r] * 32 + 8 * q, up, r);
                kev = next_event(k + 1);
            }
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if constexpr (want_post) pp_[r] -= LD;
                if constexpr (want_map) mp_[r] -= 1;
            }
            rs = rs + 1 == BWD_STAGES ? 0 : rs + 1;
            ws = ws + 1 == BWD_STAGES ? 0 : ws + 1;
        };
        for (int k = kb; k < kmax;) {
            clock_step(k, std::true_type());          // k == kev: kb is an event, and so is every clock the inner loop stops at
            ++k;
            const int stop = min(kmax, kev);
            for (; k < stop; ++k) clock_step(k, std::false_type());
        }
        stage_wait<0>();
        if (pend) post_out(prq, actq, 1);            // the last clock's posterior
        if constexpr (want_map) {
#pragma unroll
            for (int r = 0; r < 2; ++r)
                if (q == 0 && ke[r] > 0) map_part[cid[r]] = mapsum[r];
        }
    }
}

// ------------------------------------------------------------------ transition counts (xi)
// Expected transition counts of Baum-Welch (hmm.py:545-568 -> _hmm.pyx:62-117) as two
// dense products per tile of 16 CONSECUTIVE time steps, from the lattices the E-step keeps
// anyway (alpha from fwd_tile_kernel, the posteriors gamma from bwd_tile_kernel):
//     pred_{t+1} = alpha_t A                       (16 x 32) (32 x 32)     -- tile_matmul
//     W'_{t+1}   = gamma_{t+1} ./ pred_{t+1}
//     xi[i][j]  += sum_t alpha_t[i] W'_{t+1}[j]    (32 x 16) (16 x 32)     -- contraction over time
// and xi[i][j] * A[i][j] is the summed two-slice marginal: sum_i xi_t[i][j] A[i][j] =
// gamma_{t+1}[j] exactly, whatever power-of-two scale alpha_t carries (it cancels), so no
// recursion, no normaliser and no T x N x N tensor are needed -- every tile is independent.
// The second product contracts over the tile's ROWS, so both operands are needed transposed
// with respect to how lanes hold them: they take one trip through shared memory ([time][40]
// floats: fragment reads hit 32 distinct banks).  Both products are 3xTF32.  Accumulators are
// flushed into a per-warp float64 partial every XI_FLUSH tiles (tensor-core accumulation may
// truncate; 48 accumulations bound the bias near 3e-6 relative, far below it in practice).
#define XI_LDS 40
#define XI_FLUSH 8

__device__ __forceinline__ void tf32_split(float x, uint32_t &hi, uint32_t &lo)
{
    hi = tf32_rna(x);
    lo = tf32_rna(x - __uint_as_float(hi));
}

__global__ void __launch_bounds__(TILE_WARPS * 32, 1)
xi_mma_kernel(TehmmModelDev m, TehmmBatchDev b, const float *__restrict__ alpha,
               const float *__restrict__ post, double *__restrict__ xi_part, float *__restrict__ gamma0)
{
    extern __shared__ __align__(128) unsigned char tile_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    float *Xs = reinterpret_cast<float *>(tile_smem) + (size_t)warp * (2 * 16 * XI_LDS);
    float *Ws = Xs + 16 * XI_LDS;
    TransFrag A;
    load_trans<false>(m, g, q, A);
    float cacc[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) cacc[mt][nt][0] = cacc[mt][nt][1] = cacc[mt][nt][2] = cacc[mt][nt][3] = 0.f;
    const int64_t wid = (int64_t)blockIdx.x * TILE_WARPS + warp, nw = (int64_t)gridDim.x * TILE_WARPS;
    double *mine = xi_part + wid * 1024;
    for (int e = lane; e < 1024; e += 32) mine[e] = 0.0;
    __syncwarp();
    int pending = 0;
    auto flush = [&]() {
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                const int i0 = 16 * mt + g, j0 = 8 * nt + 2 * q;
                mine[i0 * 32 + j0] += (double)cacc[mt][nt][0];
                mine[i0 * 32 + j0 + 1] += (double)cacc[mt][nt][1];
                mine[(i0 + 8) * 32 + j0] += (double)cacc[mt][nt][2];
                mine[(i0 + 8) * 32 + j0 + 1] += (double)cacc[mt][nt][3];
                cacc[mt][nt][0] = cacc[mt][nt][1] = cacc[mt][nt][2] = cacc[mt][nt][3] = 0.f;
            }
        pending = 0;
    };

    for (int64_t ci = wid; ci < b.nchunks; ci += nw) {
        const TehmmChunk ch = b.chunks[ci];
        if (ch.t0 == ch.s0 && ch.t1 > ch.t0) gamma0[(int64_t)ch.seq * 32 + lane] = post[ch.t0 * 32 + lane];
        // rows g and g+8 of a tile: alpha_t and gamma_{t+1}; a row without a successor in its
        // sequence (or beyond the chunk) is zero and contributes nothing.  The next tile's rows
        // are in flight while this one is multiplied.
        auto load_tile = [&](int64_t t, float (&xv)[2][8], float (&gv)[2][8]) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int64_t tr = t + g + 8 * r;
                if (tr < ch.t1 && tr + 1 < ch.s1) {
                    load_vec32(alpha + tr * 32 + 8 * q, xv[r]);
                    load_vec32(post + (tr + 1) * 32 + 8 * q, gv[r]);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) { xv[r][i] = 0.f; gv[r][i] = 0.f; }
                }
            }
        };
        float nx[2][8], ng[2][8];
        load_tile(ch.t0, nx, ng);
        for (int64_t t = ch.t0; t < ch.t1; t += 16) {
            float xv[2][8], gv[2][8];
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int i = 0; i < 8; ++i) { xv[r][i] = nx[r][i]; gv[r][i] = ng[r][i]; }
            load_tile(t + 16, nx, ng);                 // beyond the chunk: zeros, no access
            u64 xp[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) xp[c] = pk2(xv[0][c], xv[1][c]);
            float acc[4][4];
            tile_matmul(xp, A, acc);
            __syncwarp();                              // the previous tile's fragment reads are done
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                float wv[8];
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const float p0 = acc[nt][2 * r], p1 = acc[nt][2 * r + 1];
                    wv[2 * nt] = p0 > 0.f ? __fdividef(gv[r][2 * nt], p0) : 0.f;
                    wv[2 * nt + 1] = p1 > 0.f ? __fdividef(gv[r][2 * nt + 1], p1) : 0.f;
                }
                float *xr = Xs + (g + 8 * r) * XI_LDS + 8 * q, *wr = Ws + (g + 8 * r) * XI_LDS + 8 * q;
                *reinterpret_cast<float4 *>(xr) = make_float4(xv[r][0], xv[r][1], xv[r][2], xv[r][3]);
                *reinterpret_cast<float4 *>(xr + 4) = make_float4(xv[r][4], xv[r][5], xv[r][6], xv[r][7]);
                *reinterpret_cast<float4 *>(wr) = make_float4(wv[0], wv[1], wv[2], wv[3]);
                *reinterpret_cast<float4 *>(wr + 4) = make_float4(wv[4], wv[5], wv[6], wv[7]);
            }
            __syncwarp();
            // xi += X^T W': M = from-state i, N = to-state j, K = time row of the tile
#pragma unroll
            for (int kt = 0; kt < 2; ++kt) {
                uint32_t ah[2][4], al[2][4], bh[4][2], bl[4][2];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    const float *base = Xs + (8 * kt + q) * XI_LDS + 16 * mt + g;
                    tf32_split(base[0], ah[mt][0], al[mt][0]);
                    tf32_split(base[8], ah[mt][1], al[mt][1]);
                    tf32_split(base[4 * XI_LDS], ah[mt][2], al[mt][2]);
                    tf32_split(base[4 * XI_LDS + 8], ah[mt][3], al[mt][3]);
                }
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const float *base = Ws + (8 * kt + q) * XI_LDS + 8 * nt + g;
                    tf32_split(base[0], bh[nt][0], bl[nt][0]);
                    tf32_split(base[4 * XI_LDS], bh[nt][1], bl[nt][1]);
                }
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 4; ++nt) {
                        mma_tf32(cacc[mt][nt], al[mt][0], al[mt][1], al[mt][2], al[mt][3], bh[nt][0], bh[nt][1]);
                        mma_tf32(cacc[mt][nt], ah[mt][0], ah[mt][1], ah[mt][2], ah[mt][3], bl[nt][0], bl[nt][1]);
                        mma_tf32(cacc[mt][nt], ah[mt][0], ah[mt][1], ah[mt][2], ah[mt][3], bh[nt][0], bh[nt][1]);
                    }
            }
            if (++pending == XI_FLUSH) flush();
        }
    }
    flush();
}

// start[i] += sum_seq gamma0[seq][i];  trans[i][j] += (1/N) A[i][j] sum_warps xi_part[w][i][j]
// (the 1/N is the reference's beta[T-1] = log(1/N), _hmm.pyx:179).  Fixed order, float64.
__global__ void xi_reduce_kernel(TehmmModelDev m, TehmmBatchDev b, const double *__restrict__ xi_part,
                                 int nparts, const float *__restrict__ gamma0, double *__restrict__ start_trans)
{
    const int N = m.N;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < N) {
        double acc = 0.0;
        for (int64_t s = 0; s < b.nseq; ++s)
            if (b.seq_off[s + 1] > b.seq_off[s] && tehmm_is_start(b, s)) acc += (double)gamma0[s * 32 + e];
        start_trans[e] += acc;
    }
    if (e < N * N) {
        const int i = e / N, j = e - i * N;
        double acc = 0.0;
        for (int p = 0; p < nparts; ++p) acc += xi_part[(int64_t)p * 1024 + i * 32 + j];
        start_trans[N + e] += acc * m.lin_trans[(int64_t)i * 32 + j] / (double)N;
    }
}

// ------------------------------------------------------------------ launchers
static int tile_grid(const TehmmBatchDev &b, int sms)
{
    const int64_t ngroups = (b.nchunks + 15) / 16;
    const int64_t need = (ngroups + TILE_WARPS - 1) / TILE_WARPS;
    return (int)(need < 1 ? 1 : (need < sms ? need : sms));
}

// [chunk][step][32 floats] view of a lattice holding ONE sequence cut into chunks of `lf` steps
// (full-length chunks only), boxes of TB steps x 16 chunks.  false: no tensor map (driver entry
// point missing, odd shape).
static bool make_lattice_tmap(CUtensorMap *tm, const float *base, int64_t lf, int64_t nfull)
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
    if (!encode || nfull < 1 || lf < TB || lf > (1 << 30) || nfull > (1 << 30)) return false;
    const cuuint64_t dims[3] = {32, (cuuint64_t)lf, (cuuint64_t)nfull};
    const cuuint64_t strides[2] = {128, (cuuint64_t)lf * 128};
    const cuuint32_t box[3] = {32, (cuuint32_t)TB, 16}, estr[3] = {1, 1, 1};
    return encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void *)base, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

cudaError_t tehmm_launch_forward_tile(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                      const float *blin, const double *rowmax, float *alpha,
                                      float *start_vec, float *end_vec, double *cscale,
                                      const int *bad, int mode, int sms, int64_t fine_len)
{
    const int smem = TILE_WARPS * FWD_WARP_BYTES;
    cudaError_t e = cudaFuncSetAttribute(fwd_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    CUtensorMap tm, tma;
    memset(&tm, 0, sizeof tm);
    memset(&tma, 0, sizeof tma);
    int lf = 0, nfull = 0;
    if (TEHMM_TILE_TENSOR && b.nseq == 1 && fine_len > 0 && mode == 0 &&
        make_lattice_tmap(&tm, blin, fine_len, b.total / fine_len) &&
        (!alpha || make_lattice_tmap(&tma, alpha, fine_len, b.total / fine_len))) {
        lf = (int)fine_len;
        nfull = (int)(b.total / fine_len);
    }
    fwd_tile_kernel<<<tile_grid(b, sms), TILE_WARPS * 32, smem, st>>>(m, b, blin, rowmax, alpha, start_vec,
                                                                      end_vec, cscale, bad, mode, tm, tma, lf, nfull);
    return cudaGetLastError();
}

cudaError_t tehmm_launch_backward_tile(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                       int flags, const float *blin, const float *alpha, float *post,
                                       uint8_t *map_states, double *map_part, float *start_vec,
                                       float *end_vec, const int *bad, int mode, int sms)
{
    const int th = TILE_WARPS * 32;
    const int smem = TILE_WARPS * BWD_STAGES * 2 * TILE_STAGE_BYTES;
    const int outr = flags & (TEHMM_BWD_POSTERIORS | TEHMM_BWD_MAP | TEHMM_BWD_RENORM_EPS);
    const int grid = tile_grid(b, sms);
#define BWD_TILE(O) do { cudaError_t e = cudaFuncSetAttribute(bwd_tile_kernel<O>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); \
                         if (e != cudaSuccess) return e; \
                         bwd_tile_kernel<O><<<grid, th, smem, st>>>(m, b, flags, blin, alpha, post, map_states, map_part, start_vec, end_vec, bad, mode); } while (0)
    switch (outr) {
    case 0: BWD_TILE(0); break;
    case TEHMM_BWD_POSTERIORS: BWD_TILE(TEHMM_BWD_POSTERIORS); break;
    case TEHMM_BWD_MAP: BWD_TILE(TEHMM_BWD_MAP); break;
    case TEHMM_BWD_POSTERIORS | TEHMM_BWD_MAP: BWD_TILE(TEHMM_BWD_POSTERIORS | TEHMM_BWD_MAP); break;
    case TEHMM_BWD_RENORM_EPS: BWD_TILE(0); break;                 // nothing to renormalise without an output
    case TEHMM_BWD_POSTERIORS | TEHMM_BWD_RENORM_EPS: BWD_TILE(TEHMM_BWD_POSTERIORS | TEHMM_BWD_RENORM_EPS); break;
    case TEHMM_BWD_MAP | TEHMM_BWD_RENORM_EPS: BWD_TILE(TEHMM_BWD_MAP | TEHMM_BWD_RENORM_EPS); break;
    default: BWD_TILE(TEHMM_BWD_POSTERIORS | TEHMM_BWD_MAP | TEHMM_BWD_RENORM_EPS); break;
    }
#undef BWD_TILE
    return cudaGetLastError();
}

int tehmm_tile_warps(void) { return TILE_WARPS; }

// expected start / transition counts from the alpha and posterior lattices (fine partition b);
// xi_part: sms * TILE_WARPS * 1024 doubles, gamma0: nseq * 32 floats.  2 launches.
cudaError_t tehmm_launch_xi_mma(cudaStream_t st, const TehmmModelDev &m, const TehmmBatchDev &b,
                                 const float *alpha, const float *post, double *xi_part, float *gamma0,
                                 double *start_trans, int sms)
{
    const int smem = TILE_WARPS * 2 * 16 * XI_LDS * 4;
    const int64_t need = (b.nchunks + TILE_WARPS - 1) / TILE_WARPS;       // a chunk at a time per warp
    const int grid = (int)(need < 1 ? 1 : (need < sms ? need : sms));
    cudaError_t e = cudaFuncSetAttribute(xi_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    xi_mma_kernel<<<grid, TILE_WARPS * 32, smem, st>>>(m, b, alpha, post, xi_part, gamma0);
    xi_reduce_kernel<<<(m.N * m.N + 127) / 128, 128, 0, st>>>(m, b, xi_part, grid * TILE_WARPS, gamma0, start_trans);
    return cudaGetLastError();
}
size_t tehmm_xi_mma_scratch_bytes(int sms) { return (size_t)sms * TILE_WARPS * 1024 * sizeof(double); }
