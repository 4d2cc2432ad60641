// repack.cu -- one-time re-layout of a packed GGUF weight into the SPAN-MAJOR shadow layout the TMEM-fed fused kernel
// (gemm4.cu) can stage with ONE bulk async copy per tile, whatever the block size is (SURVEY 8f rank 3).
//
// Canonical layout (loader.py:96-120, gguf-py): N rows of K/bs blocks, row stride = K/bs*ts bytes.  Block sizes of
// 84 / 110 / 136 / 210 bytes (Q2_K / Q3_K / IQ4_XS / Q6_K) and row strides that are not multiples of 16 bytes (Q8_0 at
// K = 2432: 2584 B) make 2-D tensor maps over the raw bytes illegal, so those weights could only use the direct-load
// producers.  Shadow layout:
//
//     out[s][n][PITCH]      s = 256-wide K-span index (ceil(K/256)), n = row index padded to a multiple of 256,
//                           PITCH = SpanOf<Q>::PITCH >= the span's packed bytes, a multiple of 16 (odd multiple of 16
//                           for the formats that need padding: conflict-free 16-byte shared-memory reads at lane = row)
//
// The 128 rows of one CTA for one span are then 128*PITCH contiguous, 16-byte aligned bytes.  Pad bytes, rows >= N and the
// tail of a ragged last span are zero (a zero block dequantises to 0 in every format).  The canonical bytes stay where
// they are: GGMLTensor / state_dict semantics are untouched, the shadow is a cache the host layer may drop at any time.
#include "blocks.cuh"

namespace ggufb200 {

template <int SPAN, int PITCH>
__global__ void __launch_bounds__(256) repack_kernel(const uint8_t *__restrict__ W, long long N, long long n_pad, long long row_bytes, int spans,
                                                     uint8_t *__restrict__ out)
{
    // one thread = one 2-byte unit (every block size and row stride is even): unit u of shadow row (s, n)
    constexpr int UNITS = PITCH / 2;
    const long long total = (long long)spans * n_pad * UNITS;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const int u = (int)(i % UNITS);
        const long long sn = i / UNITS;
        const long long n = sn % n_pad;
        const long long s = sn / n_pad;
        const long long src = s * SPAN + 2 * u;                 // byte offset inside the canonical row
        uint16_t v = 0;
        if (n < N && 2 * u < SPAN && src + 1 < row_bytes) v = *reinterpret_cast<const uint16_t *>(W + n * row_bytes + src);
        reinterpret_cast<uint16_t *>(out)[i] = v;
    }
}

template <class Q> static int repack_run(const void *W, long long N, long long K, void *out, cudaStream_t st)
{
    constexpr int SPAN = SpanOf<Q>::BYTES, PITCH = SpanOf<Q>::PITCH;
    const long long n_pad = (N + 255) / 256 * 256;
    const int spans = (int)((K + 255) / 256);
    const long long total = (long long)spans * n_pad * (PITCH / 2);
    long long blocks = (total + 255) / 256;
    const long long cap = (long long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    repack_kernel<SPAN, PITCH><<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const uint8_t *>(W), N, n_pad, K / Q::BS * Q::TS, spans,
                                                                   reinterpret_cast<uint8_t *>(out));
    return cudaGetLastError() == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
}

// bytes of the shadow buffer and its geometry; 0 for types without a block layout
size_t repack_bytes(int type, long long N, long long K, int *pitch, long long *span_stride)
{
    const int pt = with_block(type, 0, [](auto q) { return SpanOf<decltype(q)>::PITCH; });
    if (pt == 0) return 0;
    const long long n_pad = (N + 255) / 256 * 256;
    if (pitch) *pitch = pt;
    if (span_stride) *span_stride = n_pad * pt;
    return (size_t)((K + 255) / 256) * (size_t)n_pad * (size_t)pt;
}

int repack_dispatch(int type, const void *W, long long N, long long K, void *out, cudaStream_t st)
{
    return with_block(type, (int)GGUFB200_E_TYPE, [&](auto q) { return repack_run<decltype(q)>(W, N, K, out, st); });
}

}  // namespace ggufb200
