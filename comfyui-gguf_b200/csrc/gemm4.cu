// gemm4.cu -- K2/K3 v2: persistent fused dequant -> TENSOR MEMORY -> tcgen05 Linear (the default fused route).
//
//   Y[M,N] = X[M,K] * dequant(W)[N,K]^T (+ bias)      X fp16 / bf16, W packed GGUF blocks, fp32 accumulation in TMEM
//
// The product is computed TRANSPOSED:  D[feature n, token m] = sum_k W[n,k] * X[m,k],  i.e. the dequantised weight is the
// A operand of the UMMA and the activations are the B operand.  tcgen05.mma can read A from tensor memory, so the dequant
// warps write their fp16 results with tcgen05.st straight into TMEM columns and W never touches shared memory: the
// shared-memory port, which bounds both the smem-fed fused kernel (gemm2.cu: A by TMA + B by STS + UMMA reads of both
// = 119 B/clk of 128) and the dense kernel, only carries the activation tiles (TMA write + UMMA read, <= 64 B/clk) and the
// packed bytes (0.56 B/element).  (kind::f16 does NOT take A = f16 with B = bf16 -- measured: illegal-instruction trap -- so
// with bf16 activations the producers append the reference's cast of W to bf16.)
//
// Cluster = 2 CTAs, tcgen05.mma.cta_group::2: UMMA M = 256 features (128 TMEM lanes per CTA), N = TT tokens.
//   TMEM (512 columns per CTA):  [0, 2*TT) two accumulator slots of TT fp32 columns,  [A_BASE, A_BASE + 32*AST) ring of
//   AST A-operand stages, one stage = this CTA's 128 features x 64 k as fp16 pairs (32 columns).
//   ACCS = 1: an item is one TT-token tile, the slots alternate between items (epilogue of item i overlaps the main loop
//             of item i+1).   ACCS = 2: an item is 2*TT tokens, both slots are fed from the same A stage (each dequantised
//             element feeds twice the flops; the epilogue is not overlapped).
// Persistent: grid = min(#SM pairs, #items) clusters, item = (K range, feature tile, token tile), token tile fastest.
// Warp roles per CTA (768 threads):
//   0      TMA producer, activations: X tile [ACCS x TT/2 tokens x 64 k] per k-block, 128B-swizzled, bytes of both CTAs are
//          credited to the leader's full_x barrier (.cta_group::2)
//   1      MMA issuer (leader CTA; warp-uniform loop, one elected lane issues)
//   2      TMEM allocation; relay: forwards "this CTA's A stage is complete" to the leader with one cluster-scope arrive
//   3      TMA producer, packed weight: this CTA's 128 rows of one 256-wide K-span per copy (2-D tensor map over the raw
//          bytes, or one bulk copy from the re-packed span-major layout), ring of NP buffers
//   4-7    epilogue: TMEM -> registers -> (+bias, cast) -> [32 tokens][128 features] smem tile -> one bulk tensor store per tile
//   8-23   dequant producers: group g = (warp-8)/4 owns the k-blocks with kb % 4 == g, warp quadrant = warp % 4, lane = feature
//          row; a thread unpacks 64 consecutive k of its row (produce.cuh) and stores them with two tcgen05.st.32x32b.x16
// K is processed in whole 256-wide spans: a ragged tail (K % 256 != 0) is zero-filled by the TMA engine on both operands.
#include <type_traits>

#include "produce.cuh"
#include "umma.cuh"

namespace ggufb200 {

constexpr int kG4Threads = 768;
constexpr int kG4EpiWarp0 = 4;
constexpr int kG4ProdWarp0 = 8;

template <int TT> struct G4Tmem {
    static constexpr int A_BASE = ((2 * TT + 31) / 32) * 32;
    static constexpr int AST_RAW = (512 - A_BASE) / 32;
    static constexpr int AST = AST_RAW >= 12 ? 12 : (AST_RAW / 4) * 4;      // a multiple of 4: group g owns stages == g (mod 4)
    static_assert(AST >= 4, "token tile too wide for the A ring");
};

template <int SPAN_BYTES, int TT, int ACCS> struct G4Cfg {
    static constexpr int X_BYTES = (TT / 2) * 128;                 // one X sub-tile of this CTA: TT/2 tokens x 64 k x 2 B
    static constexpr int XSTAGE = ACCS * X_BYTES;
    static constexpr int XS = TT >= 128 ? (ACCS == 2 ? 4 : 6) : 8;
    static constexpr int P_BYTES = (128 * SPAN_BYTES + 1023) & ~1023;
    static constexpr int EPI_BYTES = 2 * 32 * 128 * 2;             // two [32 tokens][128 features] 16-bit output tiles (TMA-stored)
    static constexpr int BUDGET = 227 * 1024 - 1024 - 1024 - EPI_BYTES - XS * XSTAGE;
    static constexpr int NP_MAX = TT >= 128 ? 4 : 8;
    static constexpr int NP = BUDGET / P_BYTES < NP_MAX ? BUDGET / P_BYTES : NP_MAX;
    static constexpr int SMEM = XS * XSTAGE + NP * P_BYTES + EPI_BYTES + 1024 + 1024;
    static_assert(NP >= 2, "packed span buffers do not fit");
    static_assert(X_BYTES % 1024 == 0, "swizzled tiles need 1024-byte alignment");
};

struct G4Params {
    long long M, N, K;
    const void *bias;
    int bias_dtype;
    uint8_t *Y;
    long long ldy;
    float *partial;          // split-K: fp32 [splits, M, N]
    const uint8_t *Wspan;    // re-packed span-major layout (nullptr: 2-D tensor map over the canonical rows)
    long long span_stride;   // bytes between consecutive spans of the re-packed layout (= padded rows * span bytes)
    int ttiles, ftiles, splits;
    int spans_total, spans_per_split;
    int n_items;
    const uint16_t *loraU;   // LoRA: fp16 [N, 64] = scale * up, zero padded beyond the rank (nullptr: no LoRA k-block)
};

__device__ __forceinline__ void g4_tmem_st16(uint32_t taddr, const uint32_t (&r)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void g4_tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem desc]   (A from tensor memory: SASS UTCHMMA.2CTA tmem, gdesc, tmem)
__device__ __forceinline__ void g4_umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// kind::f16 instruction descriptor: D = f32, A (the dequantised weight) and B (the activations) in the activation dtype,
// both K-major, UMMA M = 256 (pair), N = TT
template <int ACT, int TT, bool WCAST> __device__ __forceinline__ constexpr uint32_t g4_idesc()
{
    const uint32_t bfmt = ACT == kBF16 ? 1u : 0u;
    const uint32_t afmt = (WCAST && ACT == kBF16) ? 1u : 0u;
    return (1u << 4) | (afmt << 7) | (bfmt << 10) | ((uint32_t)(TT >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}

// fp16 pair -> bf16 pair (round to nearest even), the cast the reference applies to W before F.linear (dequant.py:23)
__device__ __forceinline__ uint32_t g4_h2_to_bf2(uint32_t h)
{
    const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&h));
    const __nv_bfloat162 b = __floats2bfloat162_rn(f.x, f.y);
    return *reinterpret_cast<const uint32_t *>(&b);
}

struct G4Item {
    int split, ftile, ttile, span0, nspans;
    int lora;      // this item ends with the LoRA k-block: A = U rows (scale * up), B = T = x * down^T  (K range 0 only)
};
__device__ __forceinline__ G4Item g4_item(const G4Params &p, int item)
{
    G4Item it;
    const int per = p.ftiles * p.ttiles;
    it.split = item / per;
    const int rem = item - it.split * per;
    it.ftile = rem / p.ttiles;
    it.ttile = rem - it.ftile * p.ttiles;
    it.span0 = it.split * p.spans_per_split;
    it.nspans = min(p.spans_per_split, p.spans_total - it.span0);
    it.lora = (p.loraU != nullptr && it.split == 0) ? 1 : 0;
    return it;
}

template <class Q, int ACT, int TT, int ACCS, int PROD>
__global__ void __launch_bounds__(kG4Threads, 1)
gemm4_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmT,
             const __grid_constant__ CUtensorMap tmY, const G4Params p)
{
    // kind::f16 rejects A = f16 with B = bf16 (illegal-instruction trap on B200: profiles/r02_probe_mixed_operand_types.txt),
    // so with bf16 activations the producers cast W to bf16 -- the cast the reference applies before F.linear (dequant.py:23)
    constexpr bool WCAST = ACT == kBF16;
    constexpr int SPAN = SpanOf<Q>::BYTES;        // packed bytes of one row's K-span (coordinate step of the 2-D tensor map)
    constexpr int PITCH = SpanOf<Q>::PITCH;       // row pitch of a staged span (== SPAN whenever the 2-D tensor map is legal)
    using Cfg = G4Cfg<PITCH, TT, ACCS>;
    using TM = G4Tmem<TT>;
    // PROD: 0 = generic producers (reference sequence, every format), 1 = hand-written, fused multiply-add step,
    //       2 = hand-written, reference sequence (bit-identical weight)
    using Prod = typename std::conditional<PROD == 0, Producer<Q>, FastProducer<Q, PROD == 1>>::type;
    constexpr int XS = Cfg::XS, NP = Cfg::NP, AST = TM::AST;

    extern __shared__ uint8_t g4_smem_raw[];
    uint8_t *xt = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(g4_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *packed = xt + XS * Cfg::XSTAGE;
    uint8_t *ytile = packed + NP * Cfg::P_BYTES;            // 2 x [32][128] 16-bit, epilogue staging for the TMA store
    uint64_t *bars = reinterpret_cast<uint64_t *>(ytile + Cfg::EPI_BYTES);
    uint64_t *full_x = bars;                     // [XS]  leader's copy collects both CTAs' TMA bytes
    uint64_t *empty_x = full_x + XS;             // [XS]  multicast tcgen05.commit
    uint64_t *full_p = empty_x + XS;             // [NP]  packed span landed (local)
    uint64_t *empty_p = full_p + NP;             // [NP]  16 producer warps are done with the span (local)
    uint64_t *full_a = empty_p + NP;             // [AST] local: the 4 warps of the owning group stored their quadrants
    uint64_t *full_a2 = full_a + AST;            // [AST] leader's copy: one relay arrive per CTA
    uint64_t *empty_a = full_a2 + AST;           // [AST] multicast tcgen05.commit
    uint64_t *tmem_full = empty_a + AST;         // [2]   multicast tcgen05.commit
    uint64_t *tmem_empty = tmem_full + 2;        // [2]   leader's copy: one arrive per epilogue thread of both CTAs
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tmem_empty + 2);
    static_assert((2 * XS + 2 * NP + 3 * AST + 4) * 8 + 8 <= 1024, "barrier block");

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int pair = blockIdx.x >> 1;
    const int n_pairs = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < XS; ++s) {
            mbar_init(&full_x[s], 1);
            mbar_init(&empty_x[s], 1);
        }
        for (int s = 0; s < NP; ++s) {
            mbar_init(&full_p[s], 1);
            mbar_init(&empty_p[s], 16);
        }
        for (int s = 0; s < AST; ++s) {
            mbar_init(&full_a[s], 4);
            mbar_init(&full_a2[s], 2);
            mbar_init(&empty_a[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tmem_full[b], 1);
            mbar_init(&tmem_empty[b], 2 * 128);
        }
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc_pair(tmem_slot, 512);
    g2_fence_before();
    __syncthreads();
    cluster_sync_all();
    g2_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation, cluster hand-shake) overlaps the tail of
    // the previous kernel in the stream; nothing below may touch global memory before that kernel's writes are visible.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 0) {
        // ===================== TMA producer: activation tiles
        if (lane == 0) {
            int it = 0;
            for (int item = pair; item < p.n_items; item += n_pairs) {
                const G4Item w = g4_item(p, item);
                const int m0 = w.ttile * (TT * ACCS) + (int)rank * (TT / 2);
                const int kb0 = w.span0 * 4, nkb = w.nspans * 4 + w.lora;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % XS;
                    mbar_wait(&empty_x[s], (uint32_t)(((it / XS) & 1) ^ 1));
                    uint8_t *dst = xt + s * Cfg::XSTAGE;
                    const uint32_t bar = mapa_u32(smem_u32(&full_x[s]), 0);
                    if (leader) mbar_arrive_expect_tx(&full_x[s], 2 * Cfg::XSTAGE);
                    const bool lora_kb = kb == w.nspans * 4;      // the extra k-block reads T = x * down^T instead of X
#pragma unroll
                    for (int a = 0; a < ACCS; ++a)
                        tma_load_2d_pair(dst + a * Cfg::X_BYTES, lora_kb ? &tmT : &tmX, bar, lora_kb ? 0 : (kb0 + kb) * kG2BK, m0 + a * TT);
                }
            }
        }
    } else if (warp == 3) {
        // ===================== TMA producer: packed weight spans of this CTA's 128 feature rows
        if (lane == 0) {
            int sp = 0;
            for (int item = pair; item < p.n_items; item += n_pairs) {
                const G4Item w = g4_item(p, item);
                const int n0 = w.ftile * 256 + (int)rank * 128;
                for (int i = 0; i < w.nspans; ++i, ++sp) {
                    const int b = sp % NP;
                    mbar_wait(&empty_p[b], (uint32_t)(((sp / NP) & 1) ^ 1));
                    mbar_arrive_expect_tx(&full_p[b], 128 * PITCH);
                    if (p.Wspan) {
                        bulk_g2s(packed + b * Cfg::P_BYTES, p.Wspan + (long long)(w.span0 + i) * p.span_stride + (long long)n0 * PITCH, 128 * PITCH,
                                 &full_p[b]);
                    } else {
                        asm volatile(
                            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                                smem_u32(packed + b * Cfg::P_BYTES)),
                            "l"(reinterpret_cast<uint64_t>(&tmW)), "r"(smem_u32(&full_p[b])), "r"((w.span0 + i) * (SPAN > 256 ? SPAN / 2 : SPAN)),
                            "r"(n0)
                            : "memory");
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA).  The WHOLE warp runs the loop with warp-uniform control flow and one
        // elected lane issues: the addresses / descriptors are then provably uniform and stay in uniform registers.  (Issued
        // from inside `if (lane == 0)` every operand of every tcgen05.mma went through an ELECT / R2UR.BROADCAST loop: ~15
        // instructions per MMA on one thread -- ncu showed the issuing thread, not the tensor pipe, pacing the kernel:
        // 58 % tensor-pipe-active with the producers idle 55 % of the time, profiles/r02_gemm4_v2_tile384_ncu.txt.)
        if (leader) {
            constexpr uint32_t idesc = g4_idesc<ACT, TT, WCAST>();
            const bool elected = elect_one_sync();
            const uint64_t desc0 = g2_desc_sw128(smem_u32(xt));          // descriptor of stage 0; later stages / k steps add (bytes >> 4)
            int it = 0, ti = 0;
            for (int item = pair; item < p.n_items; item += n_pairs, ++ti) {
                const G4Item w = g4_item(p, item);
                const int nkb = w.nspans * 4 + w.lora;
                // accumulator slot(s) of this item must have been drained by the epilogue
                if constexpr (ACCS == 1) {
                    mbar_wait(&tmem_empty[ti & 1], (uint32_t)(((ti >> 1) & 1) ^ 1));
                } else {
                    mbar_wait(&tmem_empty[0], (uint32_t)((ti & 1) ^ 1));
                    mbar_wait(&tmem_empty[1], (uint32_t)((ti & 1) ^ 1));
                }
                g2_fence_after();
                const uint32_t d_col = tmem_base + (uint32_t)((ACCS == 1 ? (ti & 1) : 0) * TT);
                int sx = it % XS, sa = it % AST;
                uint32_t px = (uint32_t)((it / XS) & 1), pa = (uint32_t)((it / AST) & 1);
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    mbar_wait(&full_x[sx], px);
                    mbar_wait(&full_a2[sa], pa);
                    g2_fence_after();
                    if (elected) {
                        const uint64_t dx = desc0 + (uint64_t)((uint32_t)(sx * Cfg::XSTAGE) >> 4);
                        const uint32_t a_col = tmem_base + (uint32_t)(TM::A_BASE + sa * 32);
#pragma unroll
                        for (int j = 0; j < kG2BK / 16; ++j) {
#pragma unroll
                            for (int a = 0; a < ACCS; ++a)
                                g4_umma_ts(d_col + (uint32_t)(a * TT), a_col + (uint32_t)(j * 8), dx + (uint64_t)((a * Cfg::X_BYTES + j * 32) >> 4), idesc,
                                           (kb > 0 || j > 0) ? 1u : 0u);
                        }
                        umma_commit_pair(&empty_x[sx]);
                        umma_commit_pair(&empty_a[sa]);
                    }
                    __syncwarp();
                    if (++sx == XS) { sx = 0; px ^= 1u; }
                    if (++sa == AST) { sa = 0; pa ^= 1u; }
                }
                if (elected) {
                    if constexpr (ACCS == 1) {
                        umma_commit_pair(&tmem_full[ti & 1]);
                    } else {
                        umma_commit_pair(&tmem_full[0]);
                        umma_commit_pair(&tmem_full[1]);
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp == 2) {
        // ===================== relay: this CTA's A stage is complete -> one cluster-scope arrive on the leader's barrier
        if (lane == 0) {
            int it = 0;
            for (int item = pair; item < p.n_items; item += n_pairs) {
                const G4Item w = g4_item(p, item);
                const int nkb = w.nspans * 4 + w.lora;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int sa = it % AST;
                    mbar_wait(&full_a[sa], (uint32_t)((it / AST) & 1));
                    g2_fence_after();
                    g2_fence_before();
                    mbar_arrive_remote(mapa_u32(smem_u32(&full_a2[sa]), 0));
                }
            }
        }
    } else if (warp >= kG4ProdWarp0) {
        // ===================== dequant producers: packed span (smem) -> fp16 pairs -> tensor memory
        const int g = (warp - kG4ProdWarp0) >> 2;            // k-block owner group 0..3
        const int quad = warp & 3;                           // TMEM lane quadrant of this warp
        const int row = quad * 32 + lane;                    // feature row inside this CTA's 128
        const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)TM::A_BASE;
        int sp = 0, it0 = 0;                                 // spans seen; global k-block index at the start of the item
        auto store_half = [&](uint32_t taddr, int half, const uint32_t (&o)[16]) {
            if constexpr (WCAST && ACT == kBF16) {
                uint32_t c[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) c[j] = g4_h2_to_bf2(o[j]);
                g4_tmem_st16(taddr + (uint32_t)(half * 16), c);
            } else {
                g4_tmem_st16(taddr + (uint32_t)(half * 16), o);
            }
        };
        for (int item = pair; item < p.n_items; item += n_pairs) {
            const G4Item w = g4_item(p, item);
            // Group g produces the k-blocks whose GLOBAL index is == g (mod 4), so it is the only writer of the A stages == g
            // (mod 4) for the whole kernel: the parity wait on empty_a below can then never be satisfied by a phase two uses old.
            // A LoRA k-block shifts the next item's first index off a multiple of 4; with the quarter taken from the ITEM-local
            // index (round 2's first version: quarter g) another group became the next writer of a stage and, whenever the MMA
            // warp lagged by more than one use, passed the wait on a stale phase -- the intermittent hang of the in-kernel LoRA
            // route (profiles/r02_lora_in_kernel_intermittent_hang.log).
            const int qr = g4_group_quarter(g, it0);         // this group's quarter of every span of the item (produce.cuh)
            for (int i = 0; i < w.nspans; ++i, ++sp) {
                const int b = sp % NP;
                const int it = it0 + 4 * i + qr;             // global k-block index of this group's quarter of the span: == g (mod 4)
                const int sa = it % AST;
                mbar_wait(&full_p[b], (uint32_t)((sp / NP) & 1));
                mbar_wait(&empty_a[sa], (uint32_t)(((it / AST) & 1) ^ 1));
                g2_fence_after();
                const uint8_t *src = packed + b * Cfg::P_BYTES + row * PITCH;
                const uint32_t taddr = lane_base + (uint32_t)(sa * 32);
                Prod::run64(src, qr, [&](int half, const uint32_t (&o)[16]) { store_half(taddr, half, o); });
                g4_tmem_st_wait();
                g2_fence_before();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&full_a[sa]);
                    mbar_arrive(&empty_p[b]);
                }
            }
            if (w.lora && g == g4_lora_group(it0, w.nspans)) {       // the group that owns the stage of the LoRA k-block's global index
                // LoRA k-block: this row of U = scale * up (64 fp16, zero padded beyond the rank) straight from global memory
                const int it = it0 + 4 * w.nspans;
                const int sa = it % AST;
                mbar_wait(&empty_a[sa], (uint32_t)(((it / AST) & 1) ^ 1));
                g2_fence_after();
                const long long n = (long long)w.ftile * 256 + rank * 128 + row;
                const uint32_t taddr = lane_base + (uint32_t)(sa * 32);
                const uint4 *urow = reinterpret_cast<const uint4 *>(p.loraU + (n < p.N ? n : 0) * 64);
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t o[16];
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        uint4 v = make_uint4(0, 0, 0, 0);
                        if (n < p.N) v = urow[half * 4 + q4];
                        o[4 * q4] = v.x; o[4 * q4 + 1] = v.y; o[4 * q4 + 2] = v.z; o[4 * q4 + 3] = v.w;
                    }
                    store_half(taddr, half, o);
                }
                g4_tmem_st_wait();
                g2_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&full_a[sa]);
            }
            it0 += 4 * w.nspans + w.lora;
        }
    } else if (warp >= kG4EpiWarp0) {
        // ===================== epilogue: D[feature (lane), token (column)] -> Y[token, feature]
        // A TMEM lane is a feature, so a thread holds 32 consecutive TOKENS of one feature.  The four epilogue warps (lane
        // quadrants = 128 consecutive features) transpose through a [32 tokens][128 features] shared-memory tile (2-byte
        // stores, lanes contiguous: conflict free) and ONE bulk tensor store per tile writes 32 token rows x 256 contiguous
        // bytes (the TMA engine clips the M / N edges); two tiles alternate so the store of block b overlaps block b+1.
        const int quad = warp & 3;
        const int et = threadIdx.x - kG4EpiWarp0 * 32;          // 0..127
        const uint32_t lane_sel = (uint32_t)(quad * 32) << 16;
        const uint32_t empty_remote0 = mapa_u32(smem_u32(&tmem_empty[0]), 0);
        const uint32_t empty_remote1 = mapa_u32(smem_u32(&tmem_empty[1]), 0);
        int ti = 0, blk = 0;
        for (int item = pair; item < p.n_items; item += n_pairs, ++ti) {
            const G4Item w = g4_item(p, item);
            const long long n = (long long)w.ftile * 256 + rank * 128 + quad * 32 + lane;      // this thread's feature
            const bool n_ok = n < p.N;
            float bv = 0.f;
            if (p.bias && n_ok && !p.partial) bv = g2_bias<ACT>(p.bias, p.bias_dtype, n);
#pragma unroll 1
            for (int a = 0; a < ACCS; ++a) {
                const int slot = ACCS == 1 ? (ti & 1) : a;
                const uint32_t par = ACCS == 1 ? (uint32_t)((ti >> 1) & 1) : (uint32_t)(ti & 1);
                mbar_wait(&tmem_full[slot], par);
                g2_fence_after();
                const long long m_base = (long long)w.ttile * (TT * ACCS) + a * TT;
#pragma unroll 1
                for (int c0 = 0; c0 < TT; c0 += 32) {
                    uint32_t r[32];
                    g2_tmem_ld32(tmem_base + lane_sel + (uint32_t)(slot * TT + c0), r);
                    g2_tmem_ld_wait();
                    if (p.partial) {
                        float *dst = p.partial + ((long long)w.split * p.M + m_base + c0) * p.N + n;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (n_ok && m_base + c0 + j < p.M) dst[(long long)j * p.N] = __uint_as_float(r[j]);
                        continue;
                    }
                    if (m_base + c0 >= p.M) continue;        // block-uniform: whole 32-token block past the end
                    uint8_t *tile = ytile + (blk & 1) * (32 * 128 * 2);
                    // the bulk store issued from this tile two blocks ago must have finished READING it
                    if (et == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                    asm volatile("bar.sync 2, 128;" ::: "memory");
                    const uint32_t trow = smem_u32(tile) + (uint32_t)(et * 2);
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float v = __uint_as_float(r[j]) + bv;
                        uint16_t hb;
                        if constexpr (ACT == kBF16) hb = __bfloat16_as_ushort(__float2bfloat16_rn(v));
                        else hb = __half_as_ushort(__float2half_rn(v));
                        asm volatile("st.shared.u16 [%0], %1;" ::"r"(trow + (uint32_t)(j * 256)), "h"(hb) : "memory");
                    }
                    fence_proxy_async_smem();
                    asm volatile("bar.sync 2, 128;" ::: "memory");
                    if (et == 0) {
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                                         reinterpret_cast<uint64_t>(&tmY)),
                                     "r"(smem_u32(tile)), "r"((int)(w.ftile * 256 + rank * 128)), "r"((int)(m_base + c0))
                                     : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    ++blk;
                }
                g2_fence_before();
                mbar_arrive_remote(slot ? empty_remote1 : empty_remote0);
            }
        }
        if (et == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");     // all output tiles have left shared memory and landed
    }

    g2_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        g2_fence_after();
        tmem_dealloc_pair(tmem_base, 512);
    }
}

// ------------------------------------------------------------------ host side
struct G4Plan {
    int tt, accs, splits, spans_per_split, ttiles, ftiles, n_items;
};

// Tiling: token tile TT in {32, 128, 192}; ACCS = 2 (384-token items) when asked for; K split into ranges of whole spans
// when the output has fewer items than SM pairs (short activations; every packed byte is still read exactly once).
// Tiling by a small cost model (cycles per SM pair): an item of `tile` tokens x `kb` k-blocks costs
//   kb * max(2 * tile, 400)   (UMMA 256 x tile x 64 = 2 * tile cycles; ~400 cycles is what the dequant producers need per k-block)
//   + 3000 (pipeline fill + drain) + 1500 if the epilogue is exposed (384-token items)
// and the kernel runs ceil(items / pairs) rounds of the most expensive item.  Candidates: token tile 32 (M <= 32) / 128 / 192 /
// 384, K cut into 1..32 ranges of whole spans when a workspace for the fp32 partials is available (finalize pass charged at
// 16 bytes / cycle / SM: the slices stay L2 resident).  want_accs: 0 = let the model decide, 1 = force 192-token items, 2 = force 384-token items.
static G4Plan g4_plan(long long M, long long N, long long K, size_t ws_bytes, int want_accs, bool allow_split = true)
{
    const int pairs = sm_count() / 2;
    const int ftiles = (int)((N + 255) / 256);
    const int spans = (int)((K + 255) / 256);
    const size_t slice = (size_t)M * (size_t)N * 4;
    int max_s = 1;
    if (allow_split && slice > 0 && ws_bytes >= 2 * slice) {
        long long cap = (long long)(ws_bytes / slice);
        max_s = (int)(cap < 32 ? cap : 32);
        if (max_s > spans) max_s = spans;
    }
    struct Cand { int tt, accs; };
    Cand cands[4];
    int nc = 0;
    if (M <= 32) cands[nc++] = {32, 1};
    else {
        if (want_accs == 0 || M <= 192) cands[nc++] = {128, 1};
        if (want_accs != 2 || M <= 192) cands[nc++] = {192, 1};
        if (want_accs != 1 && M > 192) cands[nc++] = {192, 2};
    }
    G4Plan best{};
    double best_cost = 0;
    for (int c = 0; c < nc; ++c) {
        const int tile = cands[c].tt * cands[c].accs;
        const int ttiles = (int)((M + tile - 1) / tile);
        const long long tiles = (long long)ftiles * ttiles;
        for (int s = 1; s <= max_s; ++s) {
            const int per = (spans + s - 1) / s;
            const int splits = (spans + per - 1) / per;
            if (splits != s) continue;                                  // same split count as a smaller s: already evaluated
            const long long items = tiles * splits;
            const long long rounds = (items + pairs - 1) / pairs;
            const double t_kb = 2.0 * tile > 400.0 ? 2.0 * tile : 400.0;
            double cost = (double)rounds * (4.0 * per * t_kb + 3000.0 + (cands[c].accs == 2 ? 1500.0 : 0.0));
            if (splits > 1) cost += (double)(splits + 1) * (double)slice / (16.0 * 2 * pairs) + 6000.0;   // partial stores + finalize pass (L2 resident) + its launch
            if (best.n_items == 0 || cost < best_cost * 0.98) {         // prefer the earlier (simpler) candidate on near ties
                best_cost = cost;
                best.tt = cands[c].tt; best.accs = cands[c].accs; best.splits = splits; best.spans_per_split = per;
                best.ttiles = ttiles; best.ftiles = ftiles; best.n_items = (int)items;
            }
        }
    }
    return best;
}

constexpr size_t kG4SplitWsCap = 64u << 20;

// item height from the ABI flags: 2 = force 384-token items (TILE384 wins over TILE192), 1 = force 192-token items, 0 = cost model
static int g4_want_accs(int flags)
{
    return (flags & GGUFB200_FLAG_TILE384) ? 2 : ((flags & GGUFB200_FLAG_TILE192) ? 1 : 0);
}

size_t gemm4_workspace(long long M, long long N, long long K, int flags)
{
    const G4Plan pl = g4_plan(M, N, K, kG4SplitWsCap, g4_want_accs(flags), !(flags & GGUFB200_FLAG_NOSPLIT));
    return pl.splits > 1 ? (size_t)pl.splits * (size_t)M * (size_t)N * 4 : 0;
}

void gemm4_plan_info(long long M, long long N, long long K, size_t ws_bytes, int flags, int *tile_tokens, int *splits, int *spans_per_split, int *items)
{
    const G4Plan pl = g4_plan(M, N, K, ws_bytes > kG4SplitWsCap ? kG4SplitWsCap : ws_bytes, g4_want_accs(flags), !(flags & GGUFB200_FLAG_NOSPLIT));
    *tile_tokens = pl.tt * pl.accs;
    *splits = pl.splits;
    *spans_per_split = pl.spans_per_split;
    *items = pl.n_items;
}

// Split-K finalize of both fused kernels (gemm2.cu, gemm4.cu): Y = act(sum_s P[s] + bias), slices added in ascending order
// (bit-reproducible)
template <int ACT>
__global__ void __launch_bounds__(256) splitk_finalize_kernel(const float *__restrict__ P, int splits, const void *__restrict__ bias, int bias_dtype,
                                                              uint8_t *__restrict__ Y, long long M, long long N, long long ldy)
{
    const long long n8 = N / 8;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < M * n8; i += (long long)gridDim.x * 256) {
        const long long m = i / n8, n = (i % n8) * 8;
        float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int sp = 0; sp < splits; ++sp) {
            const float *src = P + ((long long)sp * M + m) * N + n;
            const float4 a = *reinterpret_cast<const float4 *>(src), b = *reinterpret_cast<const float4 *>(src + 4);
            v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w;
            v[4] += b.x; v[5] += b.y; v[6] += b.z; v[7] += b.w;
        }
        if (bias) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] += g2_bias<ACT>(bias, bias_dtype, n + j);
        }
        st_global_v4(Y + (m * ldy + n) * 2, g2_pack<ACT>(v[0], v[1]), g2_pack<ACT>(v[2], v[3]), g2_pack<ACT>(v[4], v[5]), g2_pack<ACT>(v[6], v[7]));
    }
}

int splitk_finalize(const float *P, int splits, const void *bias, int bias_dtype, void *Y, long long M, long long N, long long ldy, int act_dtype,
                    cudaStream_t st)
{
    const long long work = M * (N / 8);
    const unsigned grid = (unsigned)((work + 255) / 256 < 148 * 8 ? (work + 255) / 256 : 148 * 8);
    return with_act(act_dtype, [&](auto act) {
        splitk_finalize_kernel<act.value><<<grid, 256, 0, st>>>(P, splits, bias, bias_dtype, reinterpret_cast<uint8_t *>(Y), M, N, ldy);
        return cudaGetLastError() == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
    });
}

struct G4Args {
    const void *W;             // canonical packed rows
    const void *Wspan;         // re-packed span-major layout or nullptr
    long long span_stride;
    long long N, K;
    const void *X;
    long long M, ldx;
    const void *bias;
    int bias_dtype;
    void *Y;
    long long ldy;
    void *ws;
    size_t ws_bytes;
    int flags;                 // GGUFB200_FLAG_* bits of the call
    const void *loraT;         // LoRA: T = x * down^T, [M, 64] activation dtype, row stride ldt (nullptr: none)
    long long ldt;
    const void *loraU;         // LoRA: U = scale * up, fp16 [N, 64] contiguous
    cudaStream_t st;
};

template <class Q, int ACT, int TT, int ACCS, int PROD>
static int g4_launch(const G4Args &a, const G4Plan &pl, float *partial)
{
    using Cfg = G4Cfg<SpanOf<Q>::PITCH, TT, ACCS>;
    auto kern = gemm4_kernel<Q, ACT, TT, ACCS, PROD>;
    static unsigned char attr[64] = {};
    if (!ensure_dynamic_smem(kern, Cfg::SMEM, attr)) return GGUFB200_E_CUDA;
    G2EncodeFn fn = g2_encode_fn();
    if (!fn) return GGUFB200_E_CUDA;
    CUtensorMap tmX, tmW, tmT;
    if (!g2_make_map(&tmX, a.X, a.M, a.K, a.ldx, ACT, TT / 2)) return GGUFB200_E_CUDA;
    tmT = tmX;
    if (a.loraT && !g2_make_map(&tmT, a.loraT, a.M, 64, a.ldt, ACT, TT / 2)) return GGUFB200_E_CUDA;
    CUtensorMap tmY;
    {   // output: [M tokens, N features] 16-bit, stored in boxes of 32 tokens x 128 features, no swizzle
        cuuint64_t dims[2] = {(cuuint64_t)a.N, (cuuint64_t)a.M};
        cuuint64_t strides[1] = {(cuuint64_t)a.ldy * 2};
        cuuint32_t box[2] = {128u, 32u};
        cuuint32_t estr[2] = {1, 1};
        if (fn(&tmY, ACT == kBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, a.Y, dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return GGUFB200_E_CUDA;
    }
    if (a.Wspan) tmW = tmX;   // unused by the kernel in this mode
    else if (!make_packed_map<Q>(&tmW, a.W, a.N, a.K)) return GGUFB200_E_CUDA;
    G4Params p{};
    p.M = a.M; p.N = a.N; p.K = a.K;
    p.bias = partial ? nullptr : a.bias;
    p.bias_dtype = a.bias_dtype;
    p.Y = reinterpret_cast<uint8_t *>(a.Y);
    p.ldy = a.ldy;
    p.partial = partial;
    p.Wspan = reinterpret_cast<const uint8_t *>(a.Wspan);
    p.span_stride = a.span_stride;
    p.ttiles = pl.ttiles; p.ftiles = pl.ftiles; p.splits = pl.splits;
    p.spans_total = (int)((a.K + 255) / 256);
    p.spans_per_split = pl.spans_per_split;
    p.n_items = pl.n_items;
    p.loraU = a.loraT ? reinterpret_cast<const uint16_t *>(a.loraU) : nullptr;
    int pairs = sm_count() / 2;
    if (pairs > p.n_items) pairs = p.n_items;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(2 * pairs));
    cfg.blockDim = dim3(kG4Threads);
    cfg.dynamicSmemBytes = Cfg::SMEM;
    cfg.stream = a.st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;     // the kernel executes griddepcontrol.wait before its first global access
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 2;
    return cudaLaunchKernelEx(&cfg, kern, tmX, tmW, tmT, tmY, p) == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
}

template <class Q, int ACT, int PROD> static int g4_tiles(const G4Args &a, const G4Plan &pl, float *partial)
{
    if (pl.tt == 32) return g4_launch<Q, ACT, 32, 1, PROD>(a, pl, partial);
    if (pl.tt == 128) return g4_launch<Q, ACT, 128, 1, PROD>(a, pl, partial);
    if (pl.accs == 2) return g4_launch<Q, ACT, 192, 2, PROD>(a, pl, partial);
    return g4_launch<Q, ACT, 192, 1, PROD>(a, pl, partial);
}

// does the fused-multiply-add flag change the hand-written producer of this format?  (only Q4_K / Q5_K have a two-rounding step)
template <class Q> struct FmaMatters {
    static constexpr bool value = Q::TS == 144 || Q::TS == 176;
};

template <class Q, int ACT> static int g4_run(const G4Args &a)
{
    const bool ws_ok = a.ws && (reinterpret_cast<uintptr_t>(a.ws) & 15) == 0;
    size_t wsb = ws_ok ? a.ws_bytes : 0;
    if (wsb > kG4SplitWsCap) wsb = kG4SplitWsCap;
    const G4Plan pl = g4_plan(a.M, a.N, a.K, wsb, g4_want_accs(a.flags), !(a.flags & GGUFB200_FLAG_NOSPLIT));
    float *partial = pl.splits > 1 ? reinterpret_cast<float *>(a.ws) : nullptr;
    // producers: GENERIC wins over EXACT_W; otherwise hand-written, with the reference sequence under EXACT_W, else fused multiply-add
    int rc;
    if ((a.flags & GGUFB200_FLAG_GENERIC) || !FastProducer<Q>::fast) {
        rc = g4_tiles<Q, ACT, 0>(a, pl, partial);
    } else if (a.flags & GGUFB200_FLAG_EXACT_W) {
        if constexpr (FmaMatters<Q>::value) rc = g4_tiles<Q, ACT, 2>(a, pl, partial);
        else rc = g4_tiles<Q, ACT, 1>(a, pl, partial);
    } else {
        rc = g4_tiles<Q, ACT, 1>(a, pl, partial);
    }
    if (rc != GGUFB200_OK || !partial) return rc;
    return splitk_finalize(partial, pl.splits, a.bias, a.bias_dtype, a.Y, a.M, a.N, a.ldy, ACT, a.st);
}

// flags: the GGUFB200_FLAG_* bits of the call (EXACT_W, GENERIC, TILE384, TILE192, NOSPLIT)
int gemm4_fused_dispatch(int type, const void *W, const void *Wspan, long long span_stride, long long N, long long K, const void *X, long long M,
                         long long ldx, int act_dtype, const void *bias, int bias_dtype, void *Y, long long ldy, void *ws, size_t ws_bytes,
                         int flags, const void *loraT, long long ldt, const void *loraU, cudaStream_t st)
{
    if (N % 8 != 0 || K % 8 != 0) return GGUFB200_E_UNSUPPORTED;
    const G4Args a{W, Wspan, span_stride, N, K, X, M, ldx, bias, bias_dtype, Y, ldy, ws, ws_bytes, flags, loraT, ldt, loraU, st};
    return with_block(type, (int)GGUFB200_E_UNSUPPORTED, [&](auto q) {
        using Q = decltype(q);
        if (!Wspan && !packed_map_ok<Q>(W, K)) return (int)GGUFB200_E_UNSUPPORTED;
        return with_act(act_dtype, [&](auto act) { return g4_run<Q, act.value>(a); });
    });
}

// the canonical rows can be staged (every other weight needs the re-packed span-major layout of repack.cu)
bool gemm4_supported(int type, const void *W, long long N, long long K)
{
    if (N % 8 != 0 || K % 8 != 0) return false;
    return with_block(type, false, [&](auto q) { return packed_map_ok<decltype(q)>(W, K); });
}

}  // namespace ggufb200
