// rows.cu -- gather + dequant of selected rows of a quantised [n_table_rows, K] tensor.
//
// Replaces the Embedding path of the reference (ops.py:251-259), which dequantises the WHOLE
// table on every call and then runs F.embedding: here only the requested rows are read
// (K/BS*TS bytes each) and written (K elements each).  One CTA per (row, 2048-element chunk).
#include "blocks.cuh"

namespace ggufb200 {

constexpr int kRowThreads = 256;
constexpr int kChunkElems = 2048;

template <class Q, int MATH, int OUT>
__global__ void __launch_bounds__(kRowThreads) rows_kernel(const uint8_t *__restrict__ table, long long n_table_rows, long long K,
                                                           const long long *__restrict__ rows, void *__restrict__ dst)
{
    constexpr int EPT = 16 / OutT<OUT>::bytes;
    constexpr int CHUNK_BLOCKS = kChunkElems / Q::BS;
    constexpr int CHUNK_BYTES = CHUNK_BLOCKS * Q::TS;
    __shared__ __align__(16) uint8_t tile[CHUNK_BYTES];

    const long long i = blockIdx.y;
    const long long r = rows[i];
    const long long row_blocks = K / Q::BS;
    const long long b0 = (long long)blockIdx.x * CHUNK_BLOCKS;
    long long nb = row_blocks - b0;
    if (nb > CHUNK_BLOCKS) nb = CHUNK_BLOCKS;
    const int elems = (int)nb * Q::BS;
    uint8_t *o_row = reinterpret_cast<uint8_t *>(dst) + (i * K + b0 * Q::BS) * (long long)OutT<OUT>::bytes;
    const bool valid = (r >= 0 && r < n_table_rows);

    if (valid) {
        const uint8_t *src = table + (r * row_blocks + b0) * (long long)Q::TS;
        const int len = (int)nb * Q::TS;
        if ((reinterpret_cast<uintptr_t>(src) & 3) == 0 && (len & 3) == 0) {
            const uint32_t *s4 = reinterpret_cast<const uint32_t *>(src);
            uint32_t *d4 = reinterpret_cast<uint32_t *>(tile);
            for (int k = threadIdx.x; k < len / 4; k += kRowThreads) d4[k] = s4[k];
        } else {
            for (int k = threadIdx.x; k < len; k += kRowThreads) tile[k] = src[k];
        }
    }
    __syncthreads();

    for (int idx = threadIdx.x * EPT; idx < elems; idx += kRowThreads * EPT) {
        uint8_t *o = o_row + (long long)idx * OutT<OUT>::bytes;
        if (!valid) {  // out-of-range index: defined result (zeros) instead of a device assert
            st_global_v4(o, 0, 0, 0, 0);
            continue;
        }
        typename Math<MATH>::T2 v[EPT / 2];
        dequant_run<Q, MATH, EPT>(tile + (idx / Q::BS) * Q::TS, idx % Q::BS, v);
        if constexpr (OUT == kF32) {
            float2 f0 = Math<MATH>::to_f32x2(v[0]), f1 = Math<MATH>::to_f32x2(v[1]);
            st_global_v4(o, __float_as_uint(f0.x), __float_as_uint(f0.y), __float_as_uint(f1.x), __float_as_uint(f1.y));
        } else {
            st_global_v4(o, pack16<OUT, MATH>(v[0]), pack16<OUT, MATH>(v[1]), pack16<OUT, MATH>(v[2]), pack16<OUT, MATH>(v[3]));
        }
    }
}

template <int OUT>
__global__ void __launch_bounds__(kRowThreads) rows_bf16_kernel(const uint16_t *__restrict__ table, long long n_table_rows, long long K,
                                                                const long long *__restrict__ rows, void *__restrict__ dst)
{
    using O = typename OutT<OUT>::type;
    const long long i = blockIdx.y;
    const long long r = rows[i];
    const bool valid = (r >= 0 && r < n_table_rows);
    O *o = reinterpret_cast<O *>(dst) + i * K;
    for (long long k = (long long)blockIdx.x * kRowThreads + threadIdx.x; k < K; k += (long long)gridDim.x * kRowThreads) {
        float f = valid ? __uint_as_float((uint32_t)table[r * K + k] << 16) : 0.0f;
        if constexpr (OUT == kF16) o[k] = __float2half_rn(f);
        else if constexpr (OUT == kBF16) o[k] = __float2bfloat16_rn(f);
        else o[k] = f;
    }
}

template <class Q, int MATH, int OUT>
static int launch_rows(const void *packed, long long n_table_rows, long long K, const long long *rows, long long n_rows, void *out, cudaStream_t st)
{
    long long chunks = (K + kChunkElems - 1) / kChunkElems;
    for (long long y0 = 0; y0 < n_rows; y0 += 65535) {  // gridDim.y limit
        long long ny = n_rows - y0 < 65535 ? n_rows - y0 : 65535;
        dim3 grid((unsigned)chunks, (unsigned)ny);
        rows_kernel<Q, MATH, OUT><<<grid, kRowThreads, 0, st>>>(reinterpret_cast<const uint8_t *>(packed), n_table_rows, K, rows + y0,
                                                               reinterpret_cast<uint8_t *>(out) + y0 * K * (long long)OutT<OUT>::bytes);
    }
    return cudaGetLastError() == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
}

int rows_dispatch(int type, const void *packed, long long n_table_rows, long long K, const long long *rows, long long n_rows, void *out,
                  int out_dtype, int math_dtype, cudaStream_t st)
{
    if (type == T_BF16) {
        for (long long y0 = 0; y0 < n_rows; y0 += 65535) {
            long long ny = n_rows - y0 < 65535 ? n_rows - y0 : 65535;
            dim3 grid((unsigned)((K + kRowThreads * 4 - 1) / (kRowThreads * 4)), (unsigned)ny);
            const uint16_t *t = reinterpret_cast<const uint16_t *>(packed);
            if (out_dtype == kF16) rows_bf16_kernel<kF16><<<grid, kRowThreads, 0, st>>>(t, n_table_rows, K, rows + y0, (uint8_t *)out + y0 * K * 2);
            else if (out_dtype == kBF16) rows_bf16_kernel<kBF16><<<grid, kRowThreads, 0, st>>>(t, n_table_rows, K, rows + y0, (uint8_t *)out + y0 * K * 2);
            else rows_bf16_kernel<kF32><<<grid, kRowThreads, 0, st>>>(t, n_table_rows, K, rows + y0, (uint8_t *)out + y0 * K * 4);
        }
        return cudaGetLastError() == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
    }
    return with_block(type, (int)GGUFB200_E_TYPE, [&](auto q) {
        return with_dtype(math_dtype, [&](auto math) {
            return with_dtype(out_dtype, [&](auto o) {
                return launch_rows<decltype(q), math.value, o.value>(packed, n_table_rows, K, rows, n_rows, out, st);
            });
        });
    });
}

}  // namespace ggufb200
