// gemm2.cu -- K2, CTA-pair version: tcgen05.mma.cta_group::2 (UMMA M=256 across two SMs, N=256).
//
//   Y[M,N] = X[M,K] * W[N,K]^T (+ bias)      fp16 / bf16 activations, fp32 accumulation in TMEM
//
// Why pairs: a single-CTA 128xN UMMA has to stream A (128x16) AND the whole B (Nx16) through one SM's shared
// memory port for every instruction, and that port (128 B/clk) -- not the tensor pipe -- is what bounds a
// single-CTA kernel.  With cta_group::2 each SM of the pair holds 128 rows of A and only HALF of the
// B tile (128 of 256 rows); the hardware reads both halves, so shared-memory traffic per flop halves.
//
// Cluster = 2 CTAs.  Pair tile = (256*ACCS) x 256 x 64:  ACCS accumulator sets of 256 TMEM columns each, so one
// B tile (dequantised once) feeds 2*256*ACCS flops per element.
//   CTA rank c holds   A rows  m0 + a*256 + c*128 .. +128   (a < ACCS)          -> 16 KB * ACCS per stage (TMA)
//                      B rows  n0 + c*128 .. +128                                -> 16 KB per stage (dequant producers)
// Warp roles per CTA (512 threads): 0 TMA producer, 1 MMA issuer (leader CTA only), 2 TMEM alloc, 3 relay,
// 4-7 epilogue acc 0, 8-15 dequant producers, 8-11 epilogue acc 1.
// Barriers live at identical offsets in both CTAs:
//   full_a[s]  leader's copy collects the TMA bytes of BOTH CTAs (cp.async.bulk.tensor ... .cta_group::2, mbarrier
//              operand mapped into the leader with mapa)
//   full_b[s]  leader's copy collects one arrive per dequant thread of both CTAs (remote mbarrier.arrive)
//   empty[s], tmem_full   signalled in both CTAs by tcgen05.commit ... .multicast::cluster (mask 0b11)
#include "umma.cuh"

namespace ggufb200 {

constexpr int kG2Threads = 512;
constexpr int kG2DequantThreads = 256;

template <int ACCS, int SEG = 0> struct Gemm2Cfg {
    static constexpr int A_BYTES = ACCS * 128 * kG2BK * 2;   // 16 KB per accumulator set
    static constexpr int B_BYTES = 128 * kG2BK * 2;          // this CTA's half of the B tile
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int PACKED_BYTES = (128 * SEG + 127) & ~127;   // one staging buffer: 128 rows x SEG bytes
    static constexpr int BUDGET = 227 * 1024 - 256 - 1024 - 2 * PACKED_BYTES;   // what is left of the 227 KB for the A/B ring
    static constexpr int WANT = ACCS == 2 ? 4 : 6;
    static constexpr int STAGES = BUDGET / STAGE_BYTES < WANT ? BUDGET / STAGE_BYTES : WANT;
    static constexpr int SMEM = STAGES * STAGE_BYTES + 2 * PACKED_BYTES + 256 + 1024;
    static constexpr int TMEM_COLS = 256 * ACCS;
};

struct Gemm2Params {
    const uint8_t *W;      // packed rows
    long long row_bytes;
    long long M, N, K;
    const void *bias;
    int bias_dtype;
    uint8_t *Y;
    long long ldy;
    int tiles_m;
    int n_tiles;       // tiles_m * tiles_n
    int kb_per_split;  // k-blocks per split (a multiple of 4); == K/64 when the K loop is not split
    float *partial;    // split-K: fp32 [splits, M, N] partial results (one slice per K range), else nullptr
    int splits;        // host side only
};

// STAGED: the packed rows of the CTA's B half are staged through shared memory by a 2-D TMA over the raw bytes
// (make_packed_map: box = SEG bytes x 128 rows) one 256-wide K-span (4 k-blocks) at a time, double buffered, so the
// dequant warps read shared memory instead of paying an L2 round trip per 8 elements.  tmB is then the tensor map of the
// packed weight (unused otherwise).  The producers run the reference's fp16 sequence.
template <class Q, int ACT, int ACCS, bool STAGED>
__global__ void __launch_bounds__(STAGED ? 768 : kG2Threads, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const Gemm2Params p)
{
    constexpr int SEG = STAGED ? SpanOf<Q>::BYTES : 0;
    constexpr int DQ = STAGED ? 512 : kG2DequantThreads;      // dequant producer threads: 16 warps when the packed rows sit in smem
    using Cfg = Gemm2Cfg<ACCS, SEG>;
    constexpr int STAGES = Cfg::STAGES;
    static_assert(SEG % 16 == 0, "staging needs a format whose K-span is a multiple of 16 bytes");

    extern __shared__ uint8_t g2_smem_raw[];
    uint8_t *tiles = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(g2_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *packed = tiles + STAGES * Cfg::STAGE_BYTES;        // 2 x PACKED_BYTES (STAGED)
    uint64_t *bars = reinterpret_cast<uint64_t *>(packed + 2 * Cfg::PACKED_BYTES);
    uint64_t *full_a = bars;
    uint64_t *full_b = bars + STAGES;
    uint64_t *empty = bars + 2 * STAGES;
    uint64_t *tmem_full = bars + 3 * STAGES;
    uint64_t *full_p = bars + 3 * STAGES + 1;                   // [2] packed buffer landed
    uint64_t *empty_p = bars + 3 * STAGES + 3;                  // [2] packed buffer consumed by all dequant threads
    uint64_t *full_b2 = bars + 3 * STAGES + 5;                  // [STAGES] leader's copy: both CTAs' B halves are complete
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 4 * STAGES + 5);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int pair = blockIdx.x >> 1;
    const int tile = pair % p.n_tiles;
    const int split = pair / p.n_tiles;             // split-K: this pair owns k-blocks [kb0, kb0 + num_kb)
    const int tile_m = tile % p.tiles_m;
    const int tile_n = tile / p.tiles_m;
    const long long m0 = (long long)tile_m * (256 * ACCS);
    const long long n0 = (long long)tile_n * kG2BN;
    const int kb0 = split * p.kb_per_split;
    const int num_kb = min(p.kb_per_split, (int)(p.K / kG2BK) - kb0);

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_a[s], 1);                         // the leader's arrive.expect_tx
            mbar_init(&full_b[s], DQ / 32);                   // LOCAL: one arrive per dequant warp of this CTA
            mbar_init(&full_b2[s], 2);                        // leader's copy: one relay arrive per CTA
            mbar_init(&empty[s], 1);                          // multicast tcgen05.commit
        }
        mbar_init(tmem_full, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&full_p[i], 1);
            mbar_init(&empty_p[i], DQ / 32);
        }
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc_pair(tmem_slot, Cfg::TMEM_COLS);
    g2_fence_before();
    __syncthreads();
    cluster_sync_all();     // both CTAs' barriers are initialised before anything is signalled across the pair
    g2_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer (each CTA loads its own rows; bytes are credited to the leader's barrier)
        if (lane == 0) {
            for (int i = 0; i < num_kb; ++i) {
                const int kb = kb0 + i;    // ring slots / parities follow the local index i, K coordinates the global kb
                if constexpr (STAGED) {
                    if ((i & 3) == 0) {   // next 256-wide K-span of this CTA's 128 packed rows
                        const int lspan = i >> 2, pb = lspan & 1, span = kb >> 2;
                        mbar_wait(&empty_p[pb], (uint32_t)(((lspan >> 1) & 1) ^ 1));
                        mbar_arrive_expect_tx(&full_p[pb], 128 * SEG);
                        asm volatile(
                            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                                smem_u32(packed + pb * Cfg::PACKED_BYTES)),
                            "l"(reinterpret_cast<uint64_t>(&tmB)), "r"(smem_u32(&full_p[pb])), "r"(span * (SEG > 256 ? SEG / 2 : SEG)),
                            "r"((int)(n0 + rank * 128))
                            : "memory");
                    }
                }
                const int s = i % STAGES;
                mbar_wait(&empty[s], (uint32_t)(((i / STAGES) & 1) ^ 1));
                uint8_t *a_dst = tiles + s * Cfg::STAGE_BYTES;
                const uint32_t bar = mapa_u32(smem_u32(&full_a[s]), 0);
                if (leader) mbar_arrive_expect_tx(&full_a[s], 2 * Cfg::A_BYTES);
#pragma unroll
                for (int a = 0; a < ACCS; ++a)
                    tma_load_2d_pair(a_dst + a * (128 * 128), &tmA, bar, kb * kG2BK, (int)(m0 + a * 256 + rank * 128));
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: leader CTA, one thread, drives the tensor cores of both SMs
        if (leader && lane == 0) {
            constexpr uint32_t idesc = g2_idesc<ACT>();
            for (int kb = 0; kb < num_kb; ++kb) {   // local index: only ring slot / parity / first-MMA flag depend on it
                const int s = kb % STAGES;
                const uint32_t par = (uint32_t)((kb / STAGES) & 1);
                mbar_wait_cluster(&full_a[s], par);
                mbar_wait_cluster(&full_b2[s], par);
                g2_fence_after();
                const uint32_t a_addr = smem_u32(tiles + s * Cfg::STAGE_BYTES);
                const uint32_t b_addr = a_addr + Cfg::A_BYTES;
#pragma unroll
                for (int j = 0; j < kG2BK / 16; ++j) {
                    const uint64_t db = g2_desc_sw128(b_addr + j * 32);
                    const uint32_t acc = (kb > 0 || j > 0) ? 1u : 0u;
#pragma unroll
                    for (int a = 0; a < ACCS; ++a)
                        umma_f16_pair(tmem_base + a * 256, g2_desc_sw128(a_addr + a * (128 * 128) + j * 32), db, idesc, acc);
                }
                umma_commit_pair(&empty[s]);
            }
            umma_commit_pair(tmem_full);
        }
    } else if (warp == 3) {
        // ===================== relay: when this CTA's half of the B tile is complete, tell the leader's MMA issuer
        if (lane == 0) {
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % STAGES;
                mbar_wait(&full_b[s], (uint32_t)((kb / STAGES) & 1));
                mbar_arrive_cluster(mapa_u32(smem_u32(&full_b2[s]), 0));
            }
        }
    } else if (warp >= 8) {
        // ===================== dequant producers: this CTA's 128 rows of the B tile
        constexpr int TPR = DQ / 128;       // threads per B row: 2 (32 elements each) or 4 (16 elements each)
        constexpr int CPT = 8 / TPR;        // 16-byte chunks per thread and k-block
        const int t = threadIdx.x - 256;
        const int row = t / TPR;            // 0..127
        const int half = t % TPR;           // which part of the 64-wide k-block
        const long long n = n0 + rank * 128 + row;
        const bool valid = n < p.N;
        const uint8_t *wrow = p.W + (valid ? n : 0) * p.row_bytes;
        constexpr int GROUP = GroupOf<Q>::value;
        for (int i = 0; i < num_kb; ++i) {
            const int kb = kb0 + i;
            const int s = i % STAGES;
            if constexpr (STAGED) {
                if ((i & 3) == 0) mbar_wait(&full_p[(i >> 2) & 1], (uint32_t)((i >> 3) & 1));
            }
            mbar_wait(&empty[s], (uint32_t)(((i / STAGES) & 1) ^ 1));
            const uint32_t b_row = smem_u32(tiles + s * Cfg::STAGE_BYTES + Cfg::A_BYTES) + row * 128;
            if (valid || STAGED) {   // STAGED: rows past N were zero-filled by the TMA and dequantise to 0
                const long long k = (long long)kb * kG2BK + half * (CPT * 8);
                const int kin = STAGED ? (int)(k & (kSpanK - 1)) : 0;   // position inside the staged span
                const uint8_t *blk = STAGED ? packed + ((i >> 2) & 1) * Cfg::PACKED_BYTES + row * SEG + (kin / Q::BS) * Q::TS
                                            : wrow + (k / Q::BS) * Q::TS;
                const int e0 = (int)(k % Q::BS);
                if constexpr (STAGED && CPT == 2 && Fast16<Q, ACT>::available) {
                    uint32_t o[8];
                    Fast16<Q, ACT>::run(blk, e0, o);                  // hand-scheduled 16-element producer
                    st_shared_v4(b_row + (((half * 2) ^ (row & 7)) << 4), o[0], o[1], o[2], o[3]);
                    st_shared_v4(b_row + (((half * 2 + 1) ^ (row & 7)) << 4), o[4], o[5], o[6], o[7]);
                } else {
                    const GroupScale<kF16> g0 = group_scale<Q, kF16>(blk, e0);
                    GroupScale<kF16> g1 = g0;
                    if constexpr (GROUP == 16 && CPT == 4) g1 = group_scale<Q, kF16>(blk, e0 + 16);
#pragma unroll
                    for (int c = 0; c < CPT; ++c) {
                        __half2 v[4];
                        dequant_elems<Q, kF16, 8>(blk, e0 + c * 8, (GROUP == 16 && c >= 2) ? g1 : g0, v);
                        const int chunk = half * CPT + c;
                        st_shared_v4(b_row + ((chunk ^ (row & 7)) << 4), pack16<ACT, kF16>(v[0]), pack16<ACT, kF16>(v[1]),
                                     pack16<ACT, kF16>(v[2]), pack16<ACT, kF16>(v[3]));
                    }
                }
            } else {
#pragma unroll
                for (int c = 0; c < CPT; ++c) st_shared_v4(b_row + (((half * CPT + c) ^ (row & 7)) << 4), 0, 0, 0, 0);
            }
            // every lane publishes its own generic-proxy writes to the async proxy, the warp converges, and ONE lane
            // signals the CTA-local barrier (release is cumulative over what __syncwarp ordered before it).  The
            // cluster-scope hand-off to the MMA issuer is done by the relay warp, off the dequant warps' critical path.
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&full_b[s]);
                if constexpr (STAGED) {
                    if ((i & 3) == 3) mbar_arrive(&empty_p[(i >> 2) & 1]);   // done with this packed buffer
                }
            }
        }
    }

    // ===================== epilogue: every CTA drains its own 128 TMEM lanes of each accumulator set
    // TMEM gives each lane one ROW (32 fp32 columns per tcgen05.ld), but a row-per-lane global store would touch 32
    // different lines with 16 bytes each.  So every warp transposes through a private 32 x 80-byte staging tile in the
    // (now idle) pipeline shared memory: phase 1 lane = row writes 64 B; phase 2 four lanes cover one row's 64 B, i.e.
    // each st.global.v4 instruction writes eight fully covered 64-byte segments.
    // All 16 warps take part once their main-loop role is finished: warp w may only touch TMEM lanes 32*(w%4)..+32, so
    // the 16 warps split into 4 lane quadrants x 4 slots; a slot = (accumulator set, column range).
    __syncwarp();
    // Wait for the accumulators WITHOUT spinning: one lane of the (otherwise idle) TMEM-allocator warp polls the mbarrier
    // with a sleep back-off, every other warp parks on a hardware named barrier.  (Sixteen warps polling
    // mbarrier.try_wait.acquire.cluster -- each success/failure followed by an L1 invalidate -- were ~30 % of all issued
    // instructions of the fused kernel and competed with the dequant warps for issue slots.)
    if (warp == 2) {
        if (lane == 0) {
            while (!mbar_try_wait(tmem_full, 0)) __nanosleep(200);
        }
        __syncwarp();
    }
    asm volatile("bar.sync 1, %0;" ::"r"((int)blockDim.x) : "memory");
    if (warp < 16) {
        const int quad = warp & 3;
        const int slot = warp >> 2;                                  // 0..3
        const int acc = ACCS == 2 ? (slot & 1) : 0;
        constexpr int COLS = ACCS == 2 ? kG2BN / 2 : kG2BN / 4;      // columns per slot
        const int col_begin = (ACCS == 2 ? (slot >> 1) : slot) * COLS;
        g2_fence_after();
        const long long m_base = m0 + acc * 256 + rank * 128 + quad * 32;
        const uint32_t taddr0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * 256);
        constexpr int PITCH = 80;                                   // 64 B of payload + 16 B pad: conflict-free 16-byte accesses
        const uint32_t stage = smem_u32(tiles) + (uint32_t)warp * (32 * PITCH);
#pragma unroll 1
        for (int c0 = col_begin; c0 < col_begin + COLS; c0 += 32) {
            uint32_t r[32];
            g2_tmem_ld32(taddr0 + c0, r);
            g2_tmem_ld_wait();
            if (p.partial) {
                // split-K: store this pair's fp32 partial tile into slice `split` of the workspace (bias / cast / the sum over
                // slices in a FIXED order happen in the finalize kernel, so results are run-to-run reproducible -- no atomics).
                // Same transpose trick, 128-byte rows: eight lanes cover one row with st.global.v4.f32.
                constexpr int PITCH32 = 144;
                const uint32_t stage32 = smem_u32(tiles) + (uint32_t)warp * (32 * PITCH32);
#pragma unroll
                for (int g = 0; g < 8; ++g) st_shared_v4(stage32 + lane * PITCH32 + g * 16, r[4 * g], r[4 * g + 1], r[4 * g + 2], r[4 * g + 3]);
                __syncwarp();
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int chunk = lane + 32 * q;          // 256 chunks of 16 B = 32 rows x 8
                    const int row = chunk >> 3, part = chunk & 7;
                    float4 v;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(stage32 + row * PITCH32 + part * 16));
                    const long long m = m_base + row;
                    const long long n = n0 + c0 + part * 4;
                    if (m < p.M && n < p.N)
                        *reinterpret_cast<float4 *>(p.partial + ((long long)split * p.M + m) * p.N + n) = v;
                }
                __syncwarp();
                continue;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                uint32_t o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float v0 = __uint_as_float(r[g * 8 + 2 * j]), v1 = __uint_as_float(r[g * 8 + 2 * j + 1]);
                    if (p.bias) {
                        const long long n = n0 + c0 + g * 8 + 2 * j;
                        if (n < p.N) {   // N % 8 == 0: the pair (n, n+1) is inside or outside together
                            v0 += g2_bias<ACT>(p.bias, p.bias_dtype, n);
                            v1 += g2_bias<ACT>(p.bias, p.bias_dtype, n + 1);
                        }
                    }
                    o[j] = g2_pack<ACT>(v0, v1);
                }
                st_shared_v4(stage + lane * PITCH + g * 16, o[0], o[1], o[2], o[3]);
            }
            __syncwarp();
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int chunk = lane + 32 * q;          // 128 chunks of 16 B = 32 rows x 4
                const int row = chunk >> 2, part = chunk & 3;
                uint32_t a, b, c, d;
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(stage + row * PITCH + part * 16));
                const long long m = m_base + row;
                const long long n = n0 + c0 + part * 8;
                if (m < p.M && n < p.N) st_global_v4(p.Y + (m * p.ldy + n) * 2, a, b, c, d);
            }
            __syncwarp();
        }
    }

    g2_fence_before();
    __syncthreads();
    cluster_sync_all();     // no CTA leaves while its peer can still signal barriers in it / read its shared memory
    if (warp == 2) {
        g2_fence_after();
        tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS);
    }
}

// ------------------------------------------------------------------ host side
// 512-row pair tiles halve the dequant work and the X traffic per flop; fall back to 256-row tiles when the last
// wave of 512-row tiles would leave too many SM pairs idle.  The kernel is bound by the dequant producers, whose work per
// flop halves with 512-row tiles (measured 1.15 vs 0.62 PFLOP/s), so a partly empty last wave is the smaller evil.
static int g2_pick_accs(long long M, long long N)
{
    const int sms = sm_count();
    const long long pairs = sms / 2;
    auto eff = [&](int accs) {
        long long tiles = ((M + 256 * accs - 1) / (256 * accs)) * ((N + kG2BN - 1) / kG2BN);
        long long waves = (tiles + pairs - 1) / pairs;
        return (double)tiles / (double)(waves * pairs);
    };
    if (M <= 256) return 1;
    return eff(2) * 1.15 >= eff(1) * 0.62 ? 2 : 1;
}

// Tiling of the fused kernel: ACCS (256 or 512 activation rows per pair) and the split-K factor.
// Short activations give too few (256*ACCS x 256) tiles for the 74 SM pairs, so the K loop is cut into S ranges of whole
// 256-wide spans, each handled by its own pair, which stores its fp32 partial tile into its own slice of the caller's
// workspace ([S, M, N] fp32; bounded so the slices stay L2-resident until the finalize kernel sums them).  The fused
// kernel is bound by its dequant producers, and every M tile dequantises its W tile again, so when splitting is possible
// the tallest tile (ACCS = 2) wins: each packed byte is then read and dequantised once per 512 activation rows.
struct G2Plan {
    int accs, splits;
};

constexpr size_t kG2SplitWsCap = 64u << 20;   // half of the 126 MB L2

static G2Plan g2_fused_plan(long long M, long long N, long long K, size_t ws_bytes, bool allow_split = true)
{
    G2Plan plan{g2_pick_accs(M, N), 1};
    const size_t slice = (size_t)M * (size_t)N * 4;
    if (ws_bytes > kG2SplitWsCap) ws_bytes = kG2SplitWsCap;
    if (slice == 0 || ws_bytes < 2 * slice || !allow_split || K % kSpanK != 0) return plan;
    const int sms = sm_count();
    const long long pairs = sms / 2;
    const long long tiles_n = (N + kG2BN - 1) / kG2BN;
    auto tiles = [&](int accs) { return ((M + 256 * accs - 1) / (256 * accs)) * tiles_n; };
    if (M > 256 && tiles(2) * 2 <= pairs) plan.accs = 2;
    const long long t = tiles(plan.accs);
    if (t * 2 > pairs) return plan;   // (accs unchanged in this case)
    const long long spans = K / kSpanK;
    long long s = pairs / t;
    if (s > spans) s = spans;
    if (s > 16) s = 16;
    if (s > (long long)(ws_bytes / slice)) s = (long long)(ws_bytes / slice);
    if (s < 2) return G2Plan{g2_pick_accs(M, N), 1};
    const long long per = (spans + s - 1) / s;
    plan.splits = (int)((spans + per - 1) / per);
    return plan;
}

// split-K factor the fused route would use given a workspace (ggufb200_linear_workspace / AUTO routing)
int gemm2_fused_splits(long long M, long long N, long long K) { return g2_fused_plan(M, N, K, kG2SplitWsCap).splits; }

// k-blocks (64 wide) each K range walks: whole 256-wide spans, the last range may be shorter but never empty
static int g2_kb_per_split(long long K, int splits)
{
    if (splits <= 1) return (int)(K / kG2BK);
    const int spans = (int)(K / kSpanK);
    return ((spans + splits - 1) / splits) * 4;
}

// diagnostics (ggufb200_linear_plan): the tiling the fused kernel uses for this problem and workspace size
void gemm2_fused_plan_info(long long M, long long N, long long K, size_t ws_bytes, int flags, int *accs, int *splits, int *kb_per_split, int *ctas)
{
    const G2Plan plan = g2_fused_plan(M, N, K, ws_bytes, !(flags & GGUFB200_FLAG_NOSPLIT));
    const long long tiles = ((M + 256 * plan.accs - 1) / (256 * plan.accs)) * ((N + kG2BN - 1) / kG2BN);
    *accs = plan.accs;
    *splits = plan.splits;
    *kb_per_split = g2_kb_per_split(K, plan.splits);
    *ctas = (int)(2 * tiles * plan.splits);
}

template <class Q, int ACT, int ACCS, bool STAGED = false>
static int g2_launch(const CUtensorMap &tmA, const CUtensorMap &tmB, const Gemm2Params &p, cudaStream_t st)
{
    using Cfg = Gemm2Cfg<ACCS, STAGED ? SpanOf<Q>::BYTES : 0>;
    auto kern = gemm2_kernel<Q, ACT, ACCS, STAGED>;
    static unsigned char attr[64] = {};
    if (!ensure_dynamic_smem(kern, Cfg::SMEM, attr)) return GGUFB200_E_CUDA;
    Gemm2Params q = p;
    q.tiles_m = (int)((p.M + 256 * ACCS - 1) / (256 * ACCS));
    const long long tiles_n = (p.N + kG2BN - 1) / kG2BN;
    q.n_tiles = (int)(q.tiles_m * tiles_n);
    const int splits = p.partial ? p.splits : 1;
    q.kb_per_split = g2_kb_per_split(p.K, splits);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(2 * q.n_tiles * splits));
    cfg.blockDim = dim3(STAGED ? 768 : kG2Threads);
    cfg.dynamicSmemBytes = Cfg::SMEM;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, tmA, tmB, q) == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
}

template <class Q, int ACT>
static int g2_fused_once(const void *W, long long N, long long K, const void *X, long long M, long long ldx, const void *bias, int bias_dtype,
                         void *Y, long long ldy, float *partial, G2Plan plan, int flags, cudaStream_t st)
{
    CUtensorMap tmA;
    if (!g2_make_map(&tmA, X, M, K, ldx, ACT)) return GGUFB200_E_CUDA;
    Gemm2Params p{};
    p.partial = partial;
    p.splits = plan.splits;
    p.W = reinterpret_cast<const uint8_t *>(W);
    p.row_bytes = K / Q::BS * Q::TS;
    p.M = M; p.N = N; p.K = K;
    p.bias = bias; p.bias_dtype = bias_dtype;
    p.Y = reinterpret_cast<uint8_t *>(Y); p.ldy = ldy;
    const int accs = plan.accs;
    if constexpr (SpanOf<Q>::BYTES % 16 == 0) {
        // stage the packed rows through shared memory when a 2-D tensor map over the raw bytes is legal
        if (!(flags & GGUFB200_FLAG_UNSTAGED) && K % kSpanK == 0 && packed_map_ok<Q>(W, K)) {
            CUtensorMap tmW;
            if (!make_packed_map<Q>(&tmW, W, N, K)) return GGUFB200_E_CUDA;
            if (accs == 2) return g2_launch<Q, ACT, 2, true>(tmA, tmW, p, st);
            return g2_launch<Q, ACT, 1, true>(tmA, tmW, p, st);
        }
    }
    if (accs == 2) return g2_launch<Q, ACT, 2>(tmA, tmA, p, st);
    return g2_launch<Q, ACT, 1>(tmA, tmA, p, st);
}

template <class Q, int ACT>
static int g2_fused_act(const void *W, long long N, long long K, const void *X, long long M, long long ldx, const void *bias, int bias_dtype,
                        void *Y, long long ldy, void *ws, size_t ws_bytes, int flags, cudaStream_t st)
{
    // split-K needs room for the fp32 [splits, M, N] partial results in the caller's workspace
    const bool ws_ok = ws && (reinterpret_cast<uintptr_t>(ws) & 15) == 0;
    const G2Plan plan = g2_fused_plan(M, N, K, ws_ok ? ws_bytes : 0, !(flags & GGUFB200_FLAG_NOSPLIT));
    if (plan.splits <= 1) return g2_fused_once<Q, ACT>(W, N, K, X, M, ldx, bias, bias_dtype, Y, ldy, nullptr, plan, flags, st);
    float *P = reinterpret_cast<float *>(ws);
    int rc = g2_fused_once<Q, ACT>(W, N, K, X, M, ldx, nullptr, 0, Y, ldy, P, plan, flags, st);
    if (rc != GGUFB200_OK) return rc;
    return splitk_finalize(P, plan.splits, bias, bias_dtype, Y, M, N, ldy, ACT, st);
}

// flags: the GGUFB200_FLAG_* bits of the call (NOSPLIT, UNSTAGED)
int gemm2_fused_dispatch(int type, const void *W, long long N, long long K, const void *X, long long M, long long ldx, int act_dtype,
                         int math_dtype, const void *bias, int bias_dtype, void *Y, long long ldy, void *ws, size_t ws_bytes, int flags,
                         cudaStream_t st)
{
    if (math_dtype != kF16 || K % kG2BK != 0 || N % 8 != 0) return GGUFB200_E_UNSUPPORTED;
    return with_block(type, (int)GGUFB200_E_UNSUPPORTED, [&](auto q) {
        return with_act(act_dtype, [&](auto act) {
            return g2_fused_act<decltype(q), act.value>(W, N, K, X, M, ldx, bias, bias_dtype, Y, ldy, ws, ws_bytes, flags, st);
        });
    });
}

}  // namespace ggufb200
