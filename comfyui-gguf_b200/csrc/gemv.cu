// gemv.cu -- K3 (reference-exact W): small-M fused dequant + dot product  Y[m,n] = sum_k X[m,k] * W[n,k] (+bias).
//
// For M <= 8 (modulation / adaLN / time-embedding Linears at batch 1..8) the Linear is bound by
// reading the PACKED weight once from HBM; the weight is never materialised.  One warp owns an
// output feature n, lanes stride the row in runs of 8 consecutive k (one 16-byte X vector per m),
// the packed bytes are read straight from global memory through the shared blocks.cuh unpackers,
// W is rounded to the activation dtype exactly as the reference does before F.linear
// (dequant.py:23, ops.py:210) and accumulated in fp32; warp-shuffle reduction at the end.
#include "blocks.cuh"

namespace ggufb200 {

constexpr int kGemvThreads = 256;
constexpr int kGemvMaxM = 8;

int gemv_max_m() { return kGemvMaxM; }

template <int ACT> __device__ __forceinline__ float2 act_bits_to_f32x2(uint32_t b)
{
    if constexpr (ACT == kBF16) return make_float2(__uint_as_float(b << 16), __uint_as_float(b & 0xFFFF0000u));
    else return __half22float2(*reinterpret_cast<__half2 *>(&b));
}

// bias value rounded to the activation dtype first: the reference casts the bias to x.dtype
// (ops.py:205-207, bias_dtype = dtype) before F.linear adds it
template <int ACT> __device__ __forceinline__ float load_bias(const void *bias, int bias_dtype, long long n)
{
    float b;
    if (bias_dtype == kF32) b = reinterpret_cast<const float *>(bias)[n];
    else if (bias_dtype == kF16) b = __half2float(reinterpret_cast<const __half *>(bias)[n]);
    else b = __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(bias)[n]);
    if constexpr (ACT == kBF16) return __bfloat162float(__float2bfloat16_rn(b));
    else return __half2float(__float2half_rn(b));
}

// ------------------------------------------------------------------ tensor-core variant (default)
// The dot products of 16 output features x up to 8 activation rows are one mma.sync.m16n8k16 tile (legacy HMMA path: the
// kernel is bound by the weight stream, not by flops; tcgen05 needs M = 128 lanes and would idle 94 % of them here).
// A = dequantised W (16 features x 16 k), B = X^T (16 k x 8 rows), D = fp32 16 x 8.  The k index of a dot product may be
// permuted freely as long as A and B use the same permutation, so thread (g = lane/4, c = lane%4) simply owns the run of 32
// consecutive k  [128*span + 32c, +32)  of rows g and g+8 (header decoded once per run) and of activation row g: every
// 8-element chunk feeds two MMAs, no shuffles, no per-element FMA / unpack.  The 8 warps of a CTA split K and reduce
// their 16x8 partial tiles through shared memory.
template <int ACT> __device__ __forceinline__ void mma_16x8x16(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1)
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

template <class Q, int MATH, int ACT>
__global__ void __launch_bounds__(kGemvThreads) gemv_mma_kernel(const uint8_t *__restrict__ W, long long N, long long K, const uint8_t *__restrict__ X,
                                                                long long ldx, int M, const void *__restrict__ bias, int bias_dtype,
                                                                uint8_t *__restrict__ Y, long long ldy)
{
    __shared__ float part[kGemvThreads / 32][16][8 + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, c = lane & 3;
    const long long row_bytes = K / Q::BS * Q::TS;
    const long long n_tiles = (N + 15) / 16;
    const long long n_spans = (K + 127) / 128;
    constexpr int GROUP = GroupOf<Q>::value;
    const bool xrow_ok = g < M;
    const uint8_t *xrow = X + (long long)(xrow_ok ? g : 0) * ldx * 2;

    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long n0 = tile * 16;
        const bool ok0 = n0 + g < N, ok1 = n0 + g + 8 < N;
        const uint8_t *w0 = W + (ok0 ? n0 + g : 0) * row_bytes;
        const uint8_t *w1 = W + (ok1 ? n0 + g + 8 : 0) * row_bytes;
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        for (long long span = warp; span < n_spans; span += kGemvThreads / 32) {
            // K % 32 == 0, so a run is entirely inside or outside; lanes whose run is past K must still execute the
            // warp-wide mma.sync, so they contribute zero fragments instead of skipping
            const long long kreal = span * 128 + c * 32;
            const bool kin = kreal < K;
            const long long k = kin ? kreal : 0;
            const uint8_t *b0p = w0 + (k / Q::BS) * Q::TS, *b1p = w1 + (k / Q::BS) * Q::TS;
            const int e0 = (int)(k % Q::BS);
            if constexpr (MATH == kF16 && Fast16<Q, ACT>::available) {
                // hand-scheduled producers (one 16-byte header load + one 16-byte quant load per 16 elements)
                // interior tiles / spans (warp-uniform test) skip the per-register edge masking
                const bool interior = n0 + 16 <= N && span * 128 + 128 <= K;
#pragma unroll
                for (int hseg = 0; hseg < 2; ++hseg) {
                    uint32_t a[8], b[8];
                    Fast16<Q, ACT>::run(b0p, e0 + hseg * 16, a);
                    Fast16<Q, ACT>::run(b1p, e0 + hseg * 16, b);
                    if (interior) {
#pragma unroll
                        for (int t = 0; t < 2; ++t) {
                            uint4 xv = make_uint4(0, 0, 0, 0);
                            if (xrow_ok) xv = *reinterpret_cast<const uint4 *>(xrow + (k + hseg * 16 + t * 8) * 2);
                            mma_16x8x16<ACT>(d, a[4 * t], b[4 * t], a[4 * t + 1], b[4 * t + 1], xv.x, xv.y);
                            mma_16x8x16<ACT>(d, a[4 * t + 2], b[4 * t + 2], a[4 * t + 3], b[4 * t + 3], xv.z, xv.w);
                        }
                    } else {
#pragma unroll
                        for (int t = 0; t < 2; ++t) {
                            uint4 xv = make_uint4(0, 0, 0, 0);
                            if (xrow_ok && kin) xv = *reinterpret_cast<const uint4 *>(xrow + (k + hseg * 16 + t * 8) * 2);
                            const uint32_t a0 = (ok0 && kin) ? a[4 * t] : 0u, a1 = (ok0 && kin) ? a[4 * t + 1] : 0u;
                            const uint32_t a2 = (ok0 && kin) ? a[4 * t + 2] : 0u, a3 = (ok0 && kin) ? a[4 * t + 3] : 0u;
                            const uint32_t c0 = (ok1 && kin) ? b[4 * t] : 0u, c1 = (ok1 && kin) ? b[4 * t + 1] : 0u;
                            const uint32_t c2 = (ok1 && kin) ? b[4 * t + 2] : 0u, c3 = (ok1 && kin) ? b[4 * t + 3] : 0u;
                            mma_16x8x16<ACT>(d, a0, c0, a1, c1, xv.x, xv.y);
                            mma_16x8x16<ACT>(d, a2, c2, a3, c3, xv.z, xv.w);
                        }
                    }
                }
            } else {
            const GroupScale<MATH> ga0 = group_scale<Q, MATH>(b0p, e0), gb0 = group_scale<Q, MATH>(b1p, e0);
            GroupScale<MATH> ga1 = ga0, gb1 = gb0;
            if constexpr (GROUP == 16) {
                ga1 = group_scale<Q, MATH>(b0p, e0 + 16);
                gb1 = group_scale<Q, MATH>(b1p, e0 + 16);
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                typename Math<MATH>::T2 va[4], vb[4];
                dequant_elems<Q, MATH, 8>(b0p, e0 + t * 8, (GROUP == 16 && t >= 2) ? ga1 : ga0, va);
                dequant_elems<Q, MATH, 8>(b1p, e0 + t * 8, (GROUP == 16 && t >= 2) ? gb1 : gb0, vb);
                uint32_t a[4], b[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    a[j] = (ok0 && kin) ? pack16<ACT, MATH>(va[j]) : 0u;
                    b[j] = (ok1 && kin) ? pack16<ACT, MATH>(vb[j]) : 0u;
                }
                uint4 xv = make_uint4(0, 0, 0, 0);
                if (xrow_ok && kin) xv = *reinterpret_cast<const uint4 *>(xrow + (k + t * 8) * 2);
                mma_16x8x16<ACT>(d, a[0], b[0], a[1], b[1], xv.x, xv.y);
                mma_16x8x16<ACT>(d, a[2], b[2], a[3], b[3], xv.z, xv.w);
            }
            }
        }
        // d[0]: (feature g, row 2c)  d[1]: (g, 2c+1)  d[2]: (g+8, 2c)  d[3]: (g+8, 2c+1)
        part[warp][g][2 * c] = d[0];
        part[warp][g][2 * c + 1] = d[1];
        part[warp][g + 8][2 * c] = d[2];
        part[warp][g + 8][2 * c + 1] = d[3];
        __syncthreads();
        if (threadIdx.x < 128) {
            const int f = threadIdx.x >> 3, m = threadIdx.x & 7;
            float a = 0.f;
#pragma unroll
            for (int w = 0; w < kGemvThreads / 32; ++w) a += part[w][f][m];
            const long long n = n0 + f;
            if (n < N && m < M) {
                if (bias) a += load_bias<ACT>(bias, bias_dtype, n);
                if constexpr (ACT == kBF16) reinterpret_cast<__nv_bfloat16 *>(Y)[(long long)m * ldy + n] = __float2bfloat16_rn(a);
                else reinterpret_cast<__half *>(Y)[(long long)m * ldy + n] = __float2half_rn(a);
            }
        }
        __syncthreads();
    }
}

// BF16-typed weight (is_quantized() is true for BF16, dequant.py:7): W -> fp32 -> act dtype
template <int ACT, int MM>
__global__ void __launch_bounds__(kGemvThreads) gemv_bf16w_kernel(const uint16_t *__restrict__ W, long long N, long long K, const uint8_t *__restrict__ X,
                                                                  long long ldx, int M, const void *__restrict__ bias, int bias_dtype,
                                                                  uint8_t *__restrict__ Y, long long ldy)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * kGemvThreads + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * kGemvThreads) >> 5;
    for (long long n = warp; n < N; n += n_warps) {
        float acc[MM];
#pragma unroll
        for (int m = 0; m < MM; ++m) acc[m] = 0.0f;
        for (long long k = lane; k < K; k += 32) {
            float w = __uint_as_float((uint32_t)W[n * K + k] << 16);
            if constexpr (ACT == kF16) w = __half2float(__float2half_rn(w));
#pragma unroll
            for (int m = 0; m < MM; ++m) {
                if (m < M) {
                    uint16_t xb = reinterpret_cast<const uint16_t *>(X)[(long long)m * ldx + k];
                    float xf = ACT == kBF16 ? __uint_as_float((uint32_t)xb << 16) : __half2float(__ushort_as_half(xb));
                    acc[m] = fmaf(w, xf, acc[m]);
                }
            }
        }
#pragma unroll
        for (int m = 0; m < MM; ++m) {
            float a = acc[m];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0 && m < M) {
                if (bias) a += load_bias<ACT>(bias, bias_dtype, n);
                if constexpr (ACT == kBF16) reinterpret_cast<__nv_bfloat16 *>(Y)[(long long)m * ldy + n] = __float2bfloat16_rn(a);
                else reinterpret_cast<__half *>(Y)[(long long)m * ldy + n] = __float2half_rn(a);
            }
        }
    }
}

static unsigned gemv_grid(long long N)
{
    const int sms = sm_count();
    long long blocks = (N + 7) / 8;
    long long cap = (long long)sms * 8;
    return (unsigned)(blocks < cap ? blocks : cap);
}

template <class Q, int MATH, int ACT>
static int gemv_launch(const void *W, long long N, long long K, const void *X, long long M, long long ldx, const void *bias, int bias_dtype,
                       void *Y, long long ldy, cudaStream_t st)
{
    const uint8_t *w = reinterpret_cast<const uint8_t *>(W);
    const uint8_t *x = reinterpret_cast<const uint8_t *>(X);
    uint8_t *y = reinterpret_cast<uint8_t *>(Y);
    if ((reinterpret_cast<uintptr_t>(W) & 15) != 0) return GGUFB200_E_ALIGN;   // the 16-byte header / quant loads need an aligned base
    long long tiles = (N + 15) / 16;
    const int sms = sm_count();
    long long cap = (long long)sms * 8;
    unsigned g = (unsigned)(tiles < cap ? tiles : cap);
    gemv_mma_kernel<Q, MATH, ACT><<<g, kGemvThreads, 0, st>>>(w, N, K, x, ldx, (int)M, bias, bias_dtype, y, ldy);
    return cudaGetLastError() == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
}

int gemv_dispatch(int type, const void *W, long long N, long long K, const void *X, long long M, long long ldx, int act_dtype, int math_dtype,
                  const void *bias, int bias_dtype, void *Y, long long ldy, cudaStream_t st)
{
    if (M > kGemvMaxM) return GGUFB200_E_SHAPE;
    if (type == T_BF16) {
        const uint16_t *w = reinterpret_cast<const uint16_t *>(W);
        const uint8_t *x = reinterpret_cast<const uint8_t *>(X);
        uint8_t *y = reinterpret_cast<uint8_t *>(Y);
        unsigned grid = gemv_grid(N);
        if (act_dtype == kBF16) gemv_bf16w_kernel<kBF16, 8><<<grid, kGemvThreads, 0, st>>>(w, N, K, x, ldx, (int)M, bias, bias_dtype, y, ldy);
        else gemv_bf16w_kernel<kF16, 8><<<grid, kGemvThreads, 0, st>>>(w, N, K, x, ldx, (int)M, bias, bias_dtype, y, ldy);
        return cudaGetLastError() == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
    }
    return with_block(type, (int)GGUFB200_E_TYPE, [&](auto q) {
        return with_dtype(math_dtype, [&](auto math) {
            return with_act(act_dtype, [&](auto act) {
                return gemv_launch<decltype(q), math.value, act.value>(W, N, K, X, M, ldx, bias, bias_dtype, Y, ldy, st);
            });
        });
    });
}

}  // namespace ggufb200
