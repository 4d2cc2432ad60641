// gemv2.cu -- K3 v2: small-M (M <= 8) Linear on a packed Q4_K / Q5_K weight, bound by reading the packed bytes once.
//
//   Y[m, n] = sum_k X[m, k] * W[n, k] (+ bias),   W[n, k] = D[n, sb] * q[n, k] - Mn[n, sb],   sb = k / 32
//
// Round 1's kernel (gemv.cu, kept as the reference-exact route) materialises every weight in the activation dtype before the
// dot product: ~125 instructions per 16 weights, issue-bound at 0.25 of the HBM peak.  This kernel never forms W:
//   * the 4/5-bit integers go to the tensor core AS INTEGERS: the byte 0x43 (bf16) / 0x64 (fp16) over a quant byte is the exact
//     number 128 + q / 1024 + q, two PRMTs make four of them -- no integer-to-float conversion, no multiply, no cast;
//   * one mma.sync.m16n8k16 sums q-pattern * x over 16 k of ONE sub-block for 16 weight rows x 8 activation rows, fp32
//     accumulate; two of them cover a 32-element sub-block;
//   * the sub-block scale is applied to the 16 x 8 partial sums, not to the weights:
//         acc += D * S - (BIAS * D + Mn) * Xs,      S = sum (BIAS + q) x,   Xs = sum x   over the sub-block (precomputed per CTA)
//     as packed fp32x2 FMAs (FFMA2), with D = fp16(d * sc) and Mn = fp16(dmin * mn) the reference's own sub-block products.
// Per weight that is ~2 instructions (unpack 0.8, scale decode + exchange 0.5, scale application 0.3, MMA + loads 0.4).
// Numerics: the integer unpack and the sub-block products are the reference's; W itself is never rounded, so the result is
// closer to the exact product than the reference's (which rounds W three times in fp16 and once more to bf16) -- this is the
// `fast` contract (DESIGN.md section 3): within 1e-3 of the reference for fp16 activations, 8e-3 for bf16.
//
// Data movement: a CTA owns 16 consecutive weight rows per row tile (persistent grid).  A dedicated producer warp streams
// their packed bytes K-chunk by K-chunk (6 super-blocks = 1536 k per row) through a ring of 3..8 shared-memory stages with ONE
// 3-D tensor-map copy per stage (box = [16 rows][6 blocks][144 | 176 bytes]; a ragged K or N tail is zero-filled by the TMA
// engine), full / empty mbarriers per stage, no CTA-wide barrier in the K loop.  The 8 consumer warps take the 128-k units of
// a stage round-robin (the rotation carries over from stage to stage, so the load is even whatever K is); their 16 x 8 partial
// tiles are reduced through a double-buffered shared-memory tile at the end of a row tile (one named barrier per tile).  The
// activations (<= 8 rows) are staged once per CTA by bulk copies, their sub-block sums computed once per CTA from that copy.
#include "blocks.cuh"
#include "umma.cuh"

namespace ggufb200 {

constexpr int kV2Warps = 8;                   // consumer warps
constexpr int kV2Threads = 32 * (kV2Warps + 1);   // + the producer warp
constexpr int kV2ChunkBlocks = 6;             // super-blocks per stage and row: 864 / 1056 bytes == 96 / 32 (mod 128), so the four rows of a half-warp's 8-byte loads hit disjoint banks
constexpr int kV2MaxStages = 8;

int g_gemv2_ctas = 0;                         // bench A/B switch (ggufb200_set_tuning key 2, inert without GGUFB200_ALLOW_TUNING=1): CTAs per SM, 0 = pick

template <int TS> struct V2Cfg {
    static constexpr int PITCH = kV2ChunkBlocks * TS;               // row pitch inside a stage (dense TMA box)
    static constexpr int STAGE = 16 * PITCH;                         // 13824 / 16896 bytes, multiples of 128
};
constexpr int kV2PartBytes = 2 * kV2Warps * 16 * 9 * 4;             // double-buffered [8 warps][16][9] fp32 partial tiles
constexpr int kV2BarBytes = 256;

__device__ __forceinline__ void v2_tma_load_3d(uint32_t dst, const CUtensorMap *tm, uint64_t *bar, int c0, int c1, int c2)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
                 "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void v2_bar_consumers() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__device__ __forceinline__ unsigned long long v2_fma2(unsigned long long a, unsigned long long b, unsigned long long c)
{
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ unsigned long long v2_pack(float lo, float hi)
{
    return (unsigned long long)__float_as_uint(lo) | ((unsigned long long)__float_as_uint(hi) << 32);
}
template <int ACT> __device__ __forceinline__ void v2_mma(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1)
{
    if constexpr (ACT == kBF16) {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    } else {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    }
}
// first MMA of a sub-block: zero accumulator input
template <int ACT> __device__ __forceinline__ void v2_mma0(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1)
{
    if constexpr (ACT == kBF16) {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
                     : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(0.f));
    } else {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
                     : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(0.f));
    }
}
__device__ __forceinline__ uint32_t v2_lds32(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint2 v2_lds64(uint32_t a)
{
    uint2 v;
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 v2_lds128(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}

// QK = 4: Q4_K (144-byte super-blocks, qs at +16);  QK = 5: Q5_K (176 bytes, qh at +16, qs at +48)
template <int QK, int ACT, bool XSM>
__global__ void __launch_bounds__(kV2Threads) gemv2_kernel(const __grid_constant__ CUtensorMap tmW, long long N, long long K, const uint8_t *__restrict__ X,
                                                           long long ldx, int M, const void *__restrict__ bias, int bias_dtype,
                                                           uint8_t *__restrict__ Y, long long ldy, int NS, int w_stable)
{
    constexpr int TS = QK == 4 ? 144 : 176;
    constexpr int QS_OFF = QK == 4 ? 16 : 48;
    using Cfg = V2Cfg<TS>;
    // pattern byte and its value: fp16 0x64 -> 1024 + u (and 0x54 -> 64 + q for a high nibble kept in place, Q4_K only); bf16 0x43 -> 128 + u
    constexpr uint32_t MAGIC = ACT == kBF16 ? 0x43434343u : 0x64646464u;
    constexpr float BIAS_LO = ACT == kBF16 ? 128.f : 1024.f;
    constexpr bool INPLACE_HI = (ACT == kF16 && QK == 4);
    constexpr float BIAS_HI = INPLACE_HI ? 64.f : BIAS_LO;

    extern __shared__ __align__(128) uint8_t v2_smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(v2_smem);                 // [NS]
    uint64_t *empty = full + kV2MaxStages;                                   // [NS]
    uint64_t *xbar = empty + kV2MaxStages;
    float *part = reinterpret_cast<float *>(v2_smem + kV2BarBytes);         // [2][8 warps][16][9]
    uint8_t *ring = v2_smem + kV2BarBytes + kV2PartBytes;                   // NS x STAGE (128-byte aligned)
    float *xs = reinterpret_cast<float *>(ring + (size_t)NS * Cfg::STAGE);  // [K / 32][8]
    // XSM: the activations themselves are staged once per (persistent) CTA: M rows, pitch 2K + 64 bytes (the two rows of a
    // quarter-warp's 16-byte loads then fall into disjoint banks).  From global memory every B-fragment load is 8 L1 wavefronts
    // at M = 8 (8 different rows) and the kernel slows down with M; from shared memory it is one.
    uint8_t *xsm = reinterpret_cast<uint8_t *>(xs) + (K / 32) * 8 * 4;
    const uint32_t xpitch = (uint32_t)(2 * K + 64);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, c = lane & 3;
    const int n_blocks = (int)(K / 256);
    const int n_chunks = (n_blocks + kV2ChunkBlocks - 1) / kV2ChunkBlocks;
    const int n_tiles = (int)((N + 15) / 16);
    const int my_tiles = (int)blockIdx.x < n_tiles ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

    if (tid == 0) {
        for (int s = 0; s < NS; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kV2Warps);
        }
        mbar_init(xbar, 1);
        fence_mbar_init();
    }
    if (warp == kV2Warps && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW)) : "memory");
    __syncthreads();
    // Programmatic dependent launch: the set-up above overlaps the tail of the previous kernel in the stream; nothing below may
    // touch global memory before that kernel's writes are visible.  W_STABLE (the caller's promise that no kernel still in
    // flight writes the packed weight): the producer starts filling the ring at once -- the whole ring is in flight while the
    // previous kernel drains -- and only the consumers (activations, bias, Y) wait.
    if (w_stable) {
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (warp != kV2Warps) asm volatile("griddepcontrol.wait;" ::: "memory");
    } else {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }

    if (warp == kV2Warps) {
        // ===================== producer: one tensor-map copy per (row tile, K chunk) stage
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 1;                                     // parity to wait for on empty[s]: the first pass finds every stage free
            for (int t = 0; t < my_tiles; ++t) {
                const int row0 = ((int)blockIdx.x + t * (int)gridDim.x) * 16;
                for (int ch = 0; ch < n_chunks; ++ch) {
                    mbar_wait(&empty[s], ph);
                    mbar_arrive_expect_tx(&full[s], (uint32_t)Cfg::STAGE);          // out-of-range rows / blocks are zero-filled and count
                    v2_tma_load_3d(smem_u32(ring + (size_t)s * Cfg::STAGE), &tmW, &full[s], 0, ch * kV2ChunkBlocks, row0);
                    if (++s == NS) { s = 0; ph ^= 1u; }
                }
            }
        }
        return;
    }

    // ===================== consumers (256 threads)
    if constexpr (XSM) {
        if (tid == 0) {
            mbar_arrive_expect_tx(xbar, (uint32_t)(M * 2 * K));
            for (int m = 0; m < M; ++m) bulk_g2s(xsm + (size_t)m * xpitch, X + (long long)m * ldx * 2, (uint32_t)(2 * K), xbar);
        }
        mbar_wait(xbar, 0);
    }
    // sub-block sums of the activations: xs[sb][m] = sum of X[m, 32 sb .. 32 sb + 31] (fp32, fixed order).  Columns m >= M are
    // never written: they only ever feed output columns that are not stored.
    for (int i = tid; i < (int)(K / 32) * M; i += 32 * kV2Warps) {
        const int sb = i / M, m = i - sb * M;
        float s = 0.f;
        uint4 v[4];
        if constexpr (XSM) {
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = v2_lds128(smem_u32(xsm) + (uint32_t)m * xpitch + (uint32_t)(64 * sb + 16 * q));
        } else {
            const uint4 *p = reinterpret_cast<const uint4 *>(X + ((long long)m * ldx + 32ll * sb) * 2);
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = p[q];
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t wv[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if constexpr (ACT == kBF16) s += __uint_as_float(wv[j] << 16) + __uint_as_float(wv[j] & 0xFFFF0000u);
                else {
                    const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&wv[j]));
                    s += f.x + f.y;
                }
            }
        }
        xs[sb * 8 + m] = s;
    }
    v2_bar_consumers();

    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    // B-fragment column g = activation row g.  A column of B only feeds the same column of D, so lanes whose row does not
    // exist (g >= M) simply read the last valid row: their results are never stored -- no masking in the inner loop.
    const int gm = g < M ? g : M - 1;
    const uint8_t *xrow = X + (long long)gm * ldx * 2;
    const uint32_t xrow_s = smem_u32(xsm) + (uint32_t)gm * xpitch;
    const uint32_t xs_base = smem_u32(xs) + (uint32_t)(2 * c) * 4;
    const uint32_t quad_base = (uint32_t)(lane & ~3);

    int s = 0, rot = 0;
    uint32_t ph = 0;
    for (int t = 0; t < my_tiles; ++t) {
        for (int ch = 0; ch < n_chunks; ++ch) {
            const int cb = min(kV2ChunkBlocks, n_blocks - ch * kV2ChunkBlocks);
            const int u0 = (warp - rot) & (kV2Warps - 1);
            rot = (rot + 2 * cb) & (kV2Warps - 1);
            if (u0 < 2 * cb) {
                mbar_wait(&full[s], ph);
                const uint32_t buf = smem_u32(ring + (size_t)s * Cfg::STAGE);
                const uint32_t rg = buf + (uint32_t)(g * Cfg::PITCH), rg8 = buf + (uint32_t)((g + 8) * Cfg::PITCH);
#pragma unroll 1
                for (int u = u0; u < 2 * cb; u += kV2Warps) {
                    const int bl = u >> 1, h = u & 1;                       // super-block inside the chunk, 128-element half
                    const uint32_t bg = rg + (uint32_t)(bl * TS), bg8 = rg8 + (uint32_t)(bl * TS);
                    const int kblk = (ch * kV2ChunkBlocks + bl) * 256;
                    // ---- sub-block scales: thread c of a quad decodes sub-block j = 4h + c for both rows, the quad exchanges by shuffle
                    float Dg, Eg, Dg8, Eg8;
                    {
                        const uint4 hg = v2_lds128(bg), hg8 = v2_lds128(bg8);
                        const int j = 4 * h + c;
                        const int sh = 8 * (j & 3);
                        auto dec = [&](const uint4 &hd, float &D, float &E) {
                            const uint32_t a = (hd.y >> sh) & 0xFFu, b = (hd.z >> sh) & 0xFFu, cc = (hd.w >> sh) & 0xFFu;
                            const uint32_t sc = h ? ((cc & 0x0Fu) | ((a >> 6) << 4)) : (a & 63u);
                            const uint32_t mn = h ? ((cc >> 4) | ((b >> 6) << 4)) : (b & 63u);
                            uint32_t scm = sc | (mn << 16) | 0x64006400u;
                            const __half2 k1024 = __half2half2(__ushort_as_half((unsigned short)0x6400u));
                            const __half2 v = __hsub2_rn(*reinterpret_cast<__half2 *>(&scm), k1024);
                            uint32_t dm = hd.x;
                            const float2 DM = __half22float2(__hmul2_rn(*reinterpret_cast<__half2 *>(&dm), v));     // fp16(d*sc), fp16(dmin*mn): the reference's products
                            D = DM.x;
                            E = -fmaf((c & 1) ? BIAS_HI : BIAS_LO, DM.x, DM.y);         // stored negated: the update is acc += D * S + E * Xs
                        };
                        dec(hg, Dg, Eg);
                        dec(hg8, Dg8, Eg8);
                    }
                    uint32_t qhg[2] = {0, 0}, qhg8[2] = {0, 0};
                    if constexpr (QK == 5) {
                        const uint2 a = v2_lds64(bg + 16 + 8 * c), b = v2_lds64(bg8 + 16 + 8 * c);
                        qhg[0] = a.x; qhg[1] = a.y; qhg8[0] = b.x; qhg8[1] = b.y;
                    }
#pragma unroll
                    for (int p = 0; p < 2; ++p) {
                        const uint2 wg = v2_lds64(bg + QS_OFF + 32 * (2 * h + p) + 8 * c), wg8 = v2_lds64(bg8 + QS_OFF + 32 * (2 * h + p) + 8 * c);
#pragma unroll
                        for (int odd = 0; odd < 2; ++odd) {
                            const int s = 2 * p + odd;                      // sub-block 4h + s
                            const int sb = (int)(kblk >> 5) + 4 * h + s;
                            const uint32_t src = quad_base | (uint32_t)s;
                            const float D0 = __shfl_sync(0xffffffffu, Dg, src), E0 = __shfl_sync(0xffffffffu, Eg, src);
                            const float D8 = __shfl_sync(0xffffffffu, Dg8, src), E8 = __shfl_sync(0xffffffffu, Eg8, src);
                            uint4 xv;
                            if constexpr (XSM) xv = v2_lds128(xrow_s + (uint32_t)((kblk + 32 * (4 * h + s) + 8 * c) * 2));
                            else xv = *reinterpret_cast<const uint4 *>(xrow + (kblk + 32 * (4 * h + s) + 8 * c) * 2);
                            float d[4];
#pragma unroll
                            for (int i = 0; i < 2; ++i) {
                                uint32_t ug = i ? wg.y : wg.x, ug8 = i ? wg8.y : wg8.x;
                                uint32_t magic = MAGIC;
                                if (odd) {
                                    if constexpr (INPLACE_HI) {
                                        ug &= 0xF0F0F0F0u; ug8 &= 0xF0F0F0F0u;
                                        magic = 0x54545454u;
                                    } else {
                                        ug = (ug >> 4) & 0x0F0F0F0Fu; ug8 = (ug8 >> 4) & 0x0F0F0F0Fu;
                                    }
                                } else {
                                    ug &= 0x0F0F0F0Fu; ug8 &= 0x0F0F0F0Fu;
                                }
                                if constexpr (QK == 5) {
                                    const int jj = 4 * h + s;
                                    ug |= ((qhg[i] >> jj) & 0x01010101u) << 4;
                                    ug8 |= ((qhg8[i] >> jj) & 0x01010101u) << 4;
                                }
                                if (i == 0)
                                    v2_mma0<ACT>(d, prmt(ug, magic, 0x4140u), prmt(ug8, magic, 0x4140u), prmt(ug, magic, 0x4342u), prmt(ug8, magic, 0x4342u), xv.x, xv.y);
                                else
                                    v2_mma<ACT>(d, prmt(ug, magic, 0x4140u), prmt(ug8, magic, 0x4140u), prmt(ug, magic, 0x4342u), prmt(ug8, magic, 0x4342u), xv.z, xv.w);
                            }
                            // acc += D * S - E * Xs   (packed fp32 pairs: accumulators (0,1) belong to row g, (2,3) to row g + 8; tokens 2c, 2c + 1)
                            const uint2 xsv = v2_lds64(xs_base + (uint32_t)sb * 32);
                            const unsigned long long xs2 = (unsigned long long)xsv.x | ((unsigned long long)xsv.y << 32);
                            unsigned long long a01 = v2_pack(acc[0], acc[1]), a23 = v2_pack(acc[2], acc[3]);
                            a01 = v2_fma2(v2_pack(D0, D0), v2_pack(d[0], d[1]), a01);
                            a01 = v2_fma2(v2_pack(E0, E0), xs2, a01);
                            a23 = v2_fma2(v2_pack(D8, D8), v2_pack(d[2], d[3]), a23);
                            a23 = v2_fma2(v2_pack(E8, E8), xs2, a23);
                            acc[0] = __uint_as_float((uint32_t)a01); acc[1] = __uint_as_float((uint32_t)(a01 >> 32));
                            acc[2] = __uint_as_float((uint32_t)a23); acc[3] = __uint_as_float((uint32_t)(a23 >> 32));
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);              // a warp without a unit in this stage releases it at once
            if (++s == NS) { s = 0; ph ^= 1u; }
        }

        // ---- row tile complete: reduce the 8 warps' 16 x 8 partials, add the bias, store
        float(*pt)[16][9] = reinterpret_cast<float(*)[16][9]>(part + (t & 1) * (kV2Warps * 16 * 9));
        pt[warp][g][2 * c] = acc[0];
        pt[warp][g][2 * c + 1] = acc[1];
        pt[warp][g + 8][2 * c] = acc[2];
        pt[warp][g + 8][2 * c + 1] = acc[3];
        acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
        v2_bar_consumers();          // the buffer of tile t - 2 was read before its readers arrived at the barrier of tile t - 1
        if (tid < 128) {
            const int f = tid >> 3, m = tid & 7;
            float a = 0.f;
#pragma unroll
            for (int w = 0; w < kV2Warps; ++w) a += pt[w][f][m];
            const long long n = ((long long)blockIdx.x + (long long)t * gridDim.x) * 16 + f;
            if (n < N && m < M) {
                if (bias) {
                    float b;
                    if (bias_dtype == kF32) b = reinterpret_cast<const float *>(bias)[n];
                    else if (bias_dtype == kF16) b = __half2float(reinterpret_cast<const __half *>(bias)[n]);
                    else b = __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(bias)[n]);
                    if constexpr (ACT == kBF16) a += __bfloat162float(__float2bfloat16_rn(b));      // ops.py:205-207: bias is cast to x.dtype first
                    else a += __half2float(__float2half_rn(b));
                }
                if constexpr (ACT == kBF16) reinterpret_cast<__nv_bfloat16 *>(Y)[(long long)m * ldy + n] = __float2bfloat16_rn(a);
                else reinterpret_cast<__half *>(Y)[(long long)m * ldy + n] = __float2half_rn(a);
            }
        }
    }
}

// [N][K / 256][TS] bytes as a 3-D tensor: one box = 16 rows x 6 super-blocks, dense in shared memory
template <int TS> static bool v2_make_map(CUtensorMap *tm, const void *W, long long N, long long K)
{
    G2EncodeFn fn = g2_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[3] = {(cuuint64_t)TS, (cuuint64_t)(K / 256), (cuuint64_t)N};
    cuuint64_t strides[2] = {(cuuint64_t)TS, (cuuint64_t)(K / 256 * TS)};
    cuuint32_t box[3] = {(cuuint32_t)TS, (cuuint32_t)kV2ChunkBlocks, 16u};
    cuuint32_t estr[3] = {1, 1, 1};
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(W), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int QK, int ACT, bool XSM>
static int gemv2_launch2(const void *W, long long N, long long K, const void *X, long long M, long long ldx, const void *bias, int bias_dtype, void *Y,
                         long long ldy, int ns, int ctas, int smem, int w_stable, cudaStream_t st)
{
    constexpr int TS = QK == 4 ? 144 : 176;
    auto kern = gemv2_kernel<QK, ACT, XSM>;
    static unsigned char attr[64] = {};
    if (!ensure_dynamic_smem(kern, 227 * 1024, attr)) return GGUFB200_E_CUDA;      // the size depends on K and M: raise the cap once, to the maximum
    CUtensorMap tmW;
    if (!v2_make_map<TS>(&tmW, W, N, K)) return GGUFB200_E_CUDA;
    const long long tiles = (N + 15) / 16;
    const long long cap = (long long)sm_count() * ctas;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(tiles < cap ? tiles : cap));
    cfg.blockDim = dim3(kV2Threads);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;     // the kernel executes griddepcontrol.wait before its first global access
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, tmW, N, K, reinterpret_cast<const uint8_t *>(X), ldx, (int)M, bias, bias_dtype, reinterpret_cast<uint8_t *>(Y), ldy,
                              ns, w_stable) == cudaSuccess
               ? GGUFB200_OK
               : GGUFB200_E_CUDA;
}

// shared-memory plan: stages of the weight ring, activations staged or not, CTAs per SM
struct V2Plan {
    bool ok, xsm;
    int ns, ctas, smem;
};
template <int TS> static V2Plan v2_plan(long long N, long long K, long long M)
{
    const long long fixed = kV2BarBytes + kV2PartBytes + K / 32 * 32;
    const long long xbytes = M * (2 * K + 64);
    const long long tiles = (N + 15) / 16;
    V2Plan best{false, false, 0, 0, 0};
    double best_score = 0.0;
    for (int ctas = 2; ctas >= 1; --ctas) {          // the activations of 8 tokens + a 3-stage ring leave room for two CTAs per SM at most; three did not pay at M = 1 either (profiles/r02_bench_gemv_v3_ctas_ab.log)
        if (g_gemv2_ctas > 0 && ctas != g_gemv2_ctas) continue;
        const long long budget = 227 * 1024 / ctas - 1024;          // 1 KB per CTA is reserved by the system
        for (int x = 1; x >= 0; --x) {
            const long long room = budget - fixed - (x ? xbytes : 0);
            long long ns = room / V2Cfg<TS>::STAGE;
            if (ns > kV2MaxStages) ns = kV2MaxStages;
            if (ns < 3) continue;
            // makespan of the persistent grid x how well the SM hides latency with that many warps x the cost of re-reading X from L1
            const long long grid = tiles < 148ll * ctas ? tiles : 148ll * ctas;
            const double rounds = (double)((tiles + grid - 1) / grid);
            const double eff = (double)tiles / (rounds * (double)grid);
            const double score = eff * (ctas == 1 ? 0.75 : 1.0) * (x ? 1.0 : (M > 2 ? 0.75 : 0.95));
            if (score > best_score) {
                best_score = score;
                best = V2Plan{true, x != 0, (int)ns, ctas, (int)(fixed + (x ? xbytes : 0) + ns * V2Cfg<TS>::STAGE)};
            }
        }
    }
    return best;
}

template <int QK, int ACT>
static int gemv2_launch(const void *W, long long N, long long K, const void *X, long long M, long long ldx, const void *bias, int bias_dtype, void *Y,
                        long long ldy, int w_stable, cudaStream_t st)
{
    constexpr int TS = QK == 4 ? 144 : 176;
    const V2Plan p = v2_plan<TS>(N, K, M);
    if (!p.ok) return GGUFB200_E_UNSUPPORTED;
    if (p.xsm) return gemv2_launch2<QK, ACT, true>(W, N, K, X, M, ldx, bias, bias_dtype, Y, ldy, p.ns, p.ctas, p.smem, w_stable, st);
    return gemv2_launch2<QK, ACT, false>(W, N, K, X, M, ldx, bias, bias_dtype, Y, ldy, p.ns, p.ctas, p.smem, w_stable, st);
}

bool gemv2_supported(int type, const void *W, long long N, long long K, long long M)
{
    if (type != T_Q4_K && type != T_Q5_K) return false;
    if (M < 1 || M > 8 || K % 256 != 0 || N < 1 || N > 0x7fffffffll / 16 || K > (1ll << 20)) return false;
    if ((reinterpret_cast<uintptr_t>(W) & 15) != 0) return false;          // tensor-map base; rows of whole 144 / 176-byte super-blocks are then 16-byte aligned
    return type == T_Q4_K ? v2_plan<Block<T_Q4_K>::TS>(N, K, M).ok : v2_plan<Block<T_Q5_K>::TS>(N, K, M).ok;
}

int gemv2_dispatch(int type, const void *W, long long N, long long K, const void *X, long long M, long long ldx, int act_dtype, const void *bias,
                   int bias_dtype, void *Y, long long ldy, cudaStream_t st, bool w_stable)
{
    const int ws = w_stable ? 1 : 0;
    if (!gemv2_supported(type, W, N, K, M)) return GGUFB200_E_UNSUPPORTED;
    return with_act(act_dtype, [&](auto act) {
        return type == T_Q4_K ? gemv2_launch<4, act.value>(W, N, K, X, M, ldx, bias, bias_dtype, Y, ldy, ws, st)
                              : gemv2_launch<5, act.value>(W, N, K, X, M, ldx, bias, bias_dtype, Y, ldy, ws, st);
    });
}

}  // namespace ggufb200
