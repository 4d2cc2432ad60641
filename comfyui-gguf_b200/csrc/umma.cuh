// umma.cuh -- PTX wrappers of the CTA-pair tensor-core kernels (gemm2.cu, gemm3.cu, gemm4.cu): cluster addressing,
// cta_group::2 TMA / TMEM / tcgen05.mma / tcgen05.commit, TMEM loads, operand descriptors, epilogue helpers; and the host
// side's tensor-map encoders, which dequant.cu and gemv2.cu use as well.
#pragma once
#include <cuda.h>

#include "blocks.cuh"

namespace ggufb200 {

constexpr int kG2BK = 64;
constexpr int kG2BN = 256;          // pair-level N (UMMA N); each CTA stages 128 rows of B

// ------------------------------------------------------------------ PTX helpers (cluster / cta_group::2 flavours)
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_smem_addr, uint32_t cta_rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta_rank));
    return r;
}
// one lane of a CONVERGED warp (the same lane every time)
__device__ __forceinline__ bool elect_one_sync()
{
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t *bar, uint32_t parity)
{
    uint32_t ok = 0;
    while (!ok) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
}
// arrive on the barrier at `cluster_addr` (a shared::cluster address obtained with mapa), release at cluster scope
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr)
{
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// Same arrive with the default semantics (release at CTA scope), the form CUTLASS uses for remote barrier arrives.  When the
// payload handed over lives in tensor memory (ordered by tcgen05.fence + the barrier itself), no cluster-scope memory release is
// needed -- and the cluster-scope form above costs a full cluster fence (~0.7 us measured on the relay thread of gemm4: it capped
// the kernel at one k-block per 0.75-0.85 us whatever the MMA size was).
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr)
{
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// TMA 2-D tile load whose completion bytes are credited to an mbarrier that may live in the PEER CTA of the pair
__device__ __forceinline__ void tma_load_2d_pair(void *smem_dst, const CUtensorMap *tm, uint32_t bar_cluster_addr, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t *dst_smem, uint32_t cols)
{
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t *bar)   // arrives on `bar` in BOTH CTAs of the pair
{
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void g2_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void g2_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void g2_tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void g2_tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint64_t g2_desc_sw128(uint32_t smem_addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// kind::f16 instruction descriptor, D = f32, A/B K-major, UMMA M = 256 (pair), N = 256
template <int ACT, int UN = kG2BN> __device__ __forceinline__ constexpr uint32_t g2_idesc()
{
    uint32_t fmt = ACT == kBF16 ? 1u : 0u;
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(UN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}
template <int ACT> __device__ __forceinline__ float g2_bias(const void *bias, int bias_dtype, long long n)
{
    float b;
    if (bias_dtype == kF32) b = reinterpret_cast<const float *>(bias)[n];
    else if (bias_dtype == kF16) b = __half2float(reinterpret_cast<const __half *>(bias)[n]);
    else b = __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(bias)[n]);
    if constexpr (ACT == kBF16) return __bfloat162float(__float2bfloat16_rn(b));   // ops.py:205-207: bias is cast to x.dtype first
    else return __half2float(__float2half_rn(b));
}
template <int ACT> __device__ __forceinline__ uint32_t g2_pack(float a, float b)
{
    if constexpr (ACT == kBF16) {
        __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t *>(&v);
    } else {
        __half2 v = __floats2half2_rn(a, b);
        return *reinterpret_cast<uint32_t *>(&v);
    }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*G2EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                               const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                               CUtensorMapFloatOOBfill);

static inline G2EncodeFn g2_encode_fn()
{
    static G2EncodeFn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<G2EncodeFn>(ptr);
    }
    return fn;
}

static inline bool g2_make_map(CUtensorMap *tm, const void *base, long long rows, long long K, long long ld, int act, int box_rows = 128)
{
    G2EncodeFn fn = g2_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)kG2BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUtensorMapDataType dt = act == kBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    return fn(tm, dt, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Can make_packed_map stage the canonical rows of W: one row's span and the row stride multiples of 16 bytes, W 16-byte aligned
template <class Q> static inline bool packed_map_ok(const void *W, long long K)
{
    const long long row_bytes = K / Q::BS * Q::TS;
    return SpanOf<Q>::BYTES % 16 == 0 && row_bytes % 16 == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0;
}

// 2-D tensor map over the raw packed rows of W [N rows, K / BS blocks]: one box = one row's span x 128 rows, no swizzle.  The inner
// box extent is limited to 256 elements, so spans wider than 256 bytes use 2-byte elements (the kernels step the span coordinate
// by SpanOf<Q>::BYTES / 2 then).
template <class Q> static inline bool make_packed_map(CUtensorMap *tm, const void *W, long long N, long long K)
{
    constexpr int SPAN = SpanOf<Q>::BYTES;
    G2EncodeFn fn = g2_encode_fn();
    if (!fn) return false;
    const long long row_bytes = K / Q::BS * Q::TS;
    const bool wide = SPAN > 256;
    cuuint64_t dims[2] = {(cuuint64_t)(wide ? row_bytes / 2 : row_bytes), (cuuint64_t)N};
    cuuint64_t strides[1] = {(cuuint64_t)row_bytes};
    cuuint32_t box[2] = {(cuuint32_t)(wide ? SPAN / 2 : SPAN), 128u};
    cuuint32_t estr[2] = {1, 1};
    return fn(tm, wide ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(W), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Split-K finalize of the fused kernels (gemm4.cu): Y[M, N] = act(sum of the fp32 slices P[splits][M][N] + bias), N % 8 == 0
int splitk_finalize(const float *P, int splits, const void *bias, int bias_dtype, void *Y, long long M, long long N, long long ldy, int act_dtype,
                    cudaStream_t st);

}  // namespace ggufb200
