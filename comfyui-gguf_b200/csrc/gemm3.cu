// gemm3.cu -- K2, persistent CTA-pair GEMM for an already dense weight (DENSE mode of the Linear path).
//
//   Y[M,N] = X[M,K] * W[N,K]^T (+ bias)      fp16 / bf16, fp32 accumulation in TMEM
//
// Same operand pipeline as gemm2.cu (cluster of 2, tcgen05.mma.cta_group::2, UMMA 256x256x16, TMA-fed 128B-swizzled
// tiles), but the kernel is PERSISTENT and the accumulator is DOUBLE BUFFERED in TMEM (2 x 256 columns), so the
// epilogue of tile i overlaps the main loop of tile i+1 and the per-tile set-up (launch, barrier init, TMEM alloc,
// pipeline fill) is paid once per CTA pair instead of once per tile.  gemm2's time-vs-K fit showed its k-block cost
// already beats cuBLAS (4.2 vs 4.5 us per 64-wide k-block at 4608x12288) but ~6 us per tile wave were lost outside
// the main loop; this kernel removes that.
//
// grid = 2 * min(#pairs, #tiles); pair p walks tiles p, p+P, p+2P, ... (m fastest, so concurrently running pairs share
// W tiles in L2).  Per CTA (512 threads): warp 0 TMA producer, warp 1 MMA issuer (leader), warp 2 TMEM alloc,
// warps 4-11 epilogue (2 warps per TMEM lane quadrant, 128 columns each).
//   smem ring   full[s] (leader collects both CTAs' TMA bytes) / empty[s] (multicast tcgen05.commit)
//   TMEM ring   tmem_full[b] (multicast commit) / tmem_empty[b] (leader's; one remote arrive per epilogue thread)
#include "umma.cuh"

namespace ggufb200 {

constexpr int kG3Threads = 512;
constexpr int kG3EpiWarps = 8;
constexpr int kG3Pitch = 80;                            // staging row pitch (64 B payload + 16 B pad)
constexpr int kG3StageOut = kG3EpiWarps * 32 * kG3Pitch;

// BN = pair-level tile width (UMMA N): 256 by default; 128 when the problem has too few 256-wide tiles to occupy the
// 74 SM pairs (short activations such as the 512-token text stream / T5): twice as many tiles, same pipeline.
template <int BN> struct Gemm3Cfg {
    static constexpr int A_BYTES = 128 * kG2BK * 2;            // 16 KB
    static constexpr int B_BYTES = (BN / 2) * kG2BK * 2;       // this CTA's half of the B tile: 16 or 8 KB
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int STAGES = BN == 256 ? 5 : 7;
    static constexpr int SMEM = STAGES * STAGE_BYTES + kG3StageOut + 256 + 1024;
};

struct Gemm3Params {
    long long M, N, K;
    const void *bias;
    int bias_dtype;
    uint8_t *Y;
    long long ldy;
    int tiles_m, n_tiles;
};

template <int ACT, int BN>
__global__ void __launch_bounds__(kG3Threads, 1)
gemm3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const Gemm3Params p)
{
    using Cfg = Gemm3Cfg<BN>;
    constexpr int kG3Stages = Cfg::STAGES;
    constexpr int kG3StageBytes = Cfg::STAGE_BYTES;
    extern __shared__ uint8_t g3_smem_raw[];
    uint8_t *tiles = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(g3_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *stage_out = tiles + kG3Stages * kG3StageBytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(stage_out + kG3StageOut);
    uint64_t *full = bars;                         // [STAGES]
    uint64_t *empty = bars + kG3Stages;            // [STAGES]
    uint64_t *tmem_full = bars + 2 * kG3Stages;    // [2]
    uint64_t *tmem_empty = bars + 2 * kG3Stages + 2;   // [2]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kG3Stages + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int pair = blockIdx.x >> 1;
    const int n_pairs = gridDim.x >> 1;
    const int num_kb = (int)((p.K + kG2BK - 1) / kG2BK);   // a ragged last k-block is zero-filled by the TMA engine on both operands

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < kG3Stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tmem_full[b], 1);
            mbar_init(&tmem_empty[b], 2 * kG3EpiWarps * 32);
        }
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc_pair(tmem_slot, 512);
    g2_fence_before();
    __syncthreads();
    cluster_sync_all();
    g2_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer
        if (lane == 0) {
            int it = 0;
            for (int tile = pair; tile < p.n_tiles; tile += n_pairs) {
                const int m0 = (tile % p.tiles_m) * 256 + (int)rank * 128;
                const int n0 = (tile / p.tiles_m) * BN + (int)rank * (BN / 2);
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % kG3Stages;
                    mbar_wait(&empty[s], (uint32_t)(((it / kG3Stages) & 1) ^ 1));
                    uint8_t *dst = tiles + s * kG3StageBytes;
                    const uint32_t bar = mapa_u32(smem_u32(&full[s]), 0);
                    if (leader) mbar_arrive_expect_tx(&full[s], 2 * kG3StageBytes);
                    tma_load_2d_pair(dst, &tmA, bar, kb * kG2BK, m0);
                    tma_load_2d_pair(dst + 128 * 128, &tmB, bar, kb * kG2BK, n0);
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA): warp-uniform loop, one elected lane issues (operands stay in uniform
        // registers; issued from inside `if (lane == 0)` every tcgen05.mma operand went through an ELECT / R2UR.BROADCAST loop)
        if (leader) {
            constexpr uint32_t idesc = g2_idesc<ACT, BN>();
            const bool elected = elect_one_sync();
            const uint64_t desc0 = g2_desc_sw128(smem_u32(tiles));
            int it = 0, ti = 0;
            for (int tile = pair; tile < p.n_tiles; tile += n_pairs, ++ti) {
                const int ab = ti & 1;
                mbar_wait(&tmem_empty[ab], (uint32_t)(((ti >> 1) & 1) ^ 1));   // epilogue drained this buffer
                g2_fence_after();
                const uint32_t tacc = tmem_base + (uint32_t)(ab * BN);
                int s = it % kG3Stages;
                uint32_t par = (uint32_t)((it / kG3Stages) & 1);
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    mbar_wait(&full[s], par);
                    g2_fence_after();
                    if (elected) {
                        const uint64_t da = desc0 + (uint64_t)((uint32_t)(s * kG3StageBytes) >> 4);
#pragma unroll
                        for (int j = 0; j < kG2BK / 16; ++j)
                            umma_f16_pair(tacc, da + (uint64_t)((j * 32) >> 4), da + (uint64_t)((128 * 128 + j * 32) >> 4), idesc, (kb > 0 || j > 0) ? 1u : 0u);
                        umma_commit_pair(&empty[s]);
                    }
                    __syncwarp();
                    if (++s == kG3Stages) { s = 0; par ^= 1u; }
                }
                if (elected) umma_commit_pair(&tmem_full[ab]);
                __syncwarp();
            }
        }
    } else if (warp >= 4 && warp < 4 + kG3EpiWarps) {
        // ===================== epilogue: overlaps the next tile's main loop
        const int quad = warp & 3;
        const int col_begin = ((warp - 4) >> 2) * (BN / 2);
        const uint32_t stage = smem_u32(stage_out) + (uint32_t)(warp - 4) * (32 * kG3Pitch);
        const uint32_t empty_remote0 = mapa_u32(smem_u32(&tmem_empty[0]), 0);
        const uint32_t empty_remote1 = mapa_u32(smem_u32(&tmem_empty[1]), 0);
        int ti = 0;
        for (int tile = pair; tile < p.n_tiles; tile += n_pairs, ++ti) {
            const int ab = ti & 1;
            const long long m_base = (long long)(tile % p.tiles_m) * 256 + rank * 128 + quad * 32;
            const long long n0 = (long long)(tile / p.tiles_m) * BN;
            mbar_wait(&tmem_full[ab], (uint32_t)((ti >> 1) & 1));
            g2_fence_after();
            const uint32_t taddr0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ab * BN);
#pragma unroll 1
            for (int c0 = col_begin; c0 < col_begin + BN / 2; c0 += 32) {
                uint32_t r[32];
                g2_tmem_ld32(taddr0 + c0, r);
                g2_tmem_ld_wait();
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    uint32_t o[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float v0 = __uint_as_float(r[g * 8 + 2 * j]), v1 = __uint_as_float(r[g * 8 + 2 * j + 1]);
                        if (p.bias) {
                            const long long n = n0 + c0 + g * 8 + 2 * j;
                            if (n < p.N) {
                                v0 += g2_bias<ACT>(p.bias, p.bias_dtype, n);
                                v1 += g2_bias<ACT>(p.bias, p.bias_dtype, n + 1);
                            }
                        }
                        o[j] = g2_pack<ACT>(v0, v1);
                    }
                    st_shared_v4(stage + lane * kG3Pitch + g * 16, o[0], o[1], o[2], o[3]);
                }
                __syncwarp();
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int chunk = lane + 32 * q;
                    const int row = chunk >> 2, part = chunk & 3;
                    uint32_t a, b, c, d;
                    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(stage + row * kG3Pitch + part * 16));
                    const long long m = m_base + row;
                    const long long n = n0 + c0 + part * 8;
                    if (m < p.M && n < p.N) st_global_v4(p.Y + (m * p.ldy + n) * 2, a, b, c, d);
                }
                __syncwarp();
            }
            // this thread's TMEM reads of buffer `ab` are complete (tcgen05.wait::ld above): hand it back to the MMA issuer
            g2_fence_before();
            mbar_arrive_remote(ab ? empty_remote1 : empty_remote0);
        }
    }

    g2_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        g2_fence_after();
        tmem_dealloc_pair(tmem_base, 512);
    }
}

template <int ACT, int BN>
static int g3_launch(const CUtensorMap &tmA, const CUtensorMap &tmB, Gemm3Params p, cudaStream_t st)
{
    constexpr int kG3Smem = Gemm3Cfg<BN>::SMEM;
    auto kern = gemm3_kernel<ACT, BN>;
    static unsigned char attr[64] = {};
    if (!ensure_dynamic_smem(kern, kG3Smem, attr)) return GGUFB200_E_CUDA;
    const int sms = sm_count();
    p.tiles_m = (int)((p.M + 255) / 256);
    p.n_tiles = p.tiles_m * (int)((p.N + BN - 1) / BN);
    int pairs = sms / 2;
    if (pairs > p.n_tiles) pairs = p.n_tiles;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(2 * pairs));
    cfg.blockDim = dim3(kG3Threads);
    cfg.dynamicSmemBytes = kG3Smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, tmA, tmB, p) == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
}

int gemm3_dense_dispatch(const void *W, long long N, long long K, long long ldw, const void *X, long long M, long long ldx, int act_dtype,
                         const void *bias, int bias_dtype, void *Y, long long ldy, cudaStream_t st)
{
    if (K % 8 != 0 || N % 8 != 0) return GGUFB200_E_UNSUPPORTED;
    const int sms = sm_count();
    const long long tiles256 = ((M + 255) / 256) * ((N + 255) / 256);
    const bool narrow = tiles256 <= sms / 4;       // far fewer 256-wide tiles than SM pairs: halve the tile width
    CUtensorMap tmA, tmB;
    if (!g2_make_map(&tmA, X, M, K, ldx, act_dtype)) return GGUFB200_E_CUDA;
    if (!g2_make_map(&tmB, W, N, K, ldw, act_dtype, narrow ? 64 : 128)) return GGUFB200_E_CUDA;
    Gemm3Params p{};
    p.M = M; p.N = N; p.K = K;
    p.bias = bias; p.bias_dtype = bias_dtype;
    p.Y = reinterpret_cast<uint8_t *>(Y); p.ldy = ldy;
    return with_act(act_dtype, [&](auto act) { return narrow ? g3_launch<act.value, 128>(tmA, tmB, p, st) : g3_launch<act.value, 256>(tmA, tmB, p, st); });
}

}  // namespace ggufb200
