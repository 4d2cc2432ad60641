// dequant.cu -- K1: standalone GGUF block dequant (HBM-bound streaming kernel).
//
// Replaces dequant.py:30-44 + every dequantize_blocks_* (dequant.py:61-285) + the final
// `.to(dtype)` (dequant.py:23) with ONE kernel launch per tensor.
//
// Data movement (algorithmic bytes per element = TS/BS read + sizeof(out) written):
//   * the packed block stream is treated as a flat byte stream (block sizes 18/22/34/84/110/
//     210 B are not 16 B multiples, so 2-D tensor maps are illegal for most shapes); it is cut
//     into tiles of 4096 elements whose byte span is always a multiple of 16 B
//   * ONE TILE PER CTA (128 threads), CTAs handed out by the hardware in address order: the write front stays
//     compact, an SM that happens to be slower simply takes fewer tiles, and 16 CTAs per SM cover each other's load
//     latency.  (Round 1's persistent CTAs with a 3-stage prefetch ring and strided tiles: 0.885 of the measured copy peak
//     on the Flux-shape sweep, 5.8 TB/s on a 1 GB output; this form: 0.949 and 6.75 TB/s --
//     profiles/r02_k1_variants_ab.log, same effect as in tools/probe_write.cu's plain-store probes.)
//   * the tile is staged into shared memory by thread 0 with the TMA engine (cp.async.bulk, SASS UBLKCP), completion on
//     an mbarrier that only thread 0 polls; the other threads sleep in the CTA barrier
//   * every thread unpacks one run of 32 consecutive elements from shared memory (blocks.cuh) into its row of the output
//     tile in shared memory, which leaves through ONE swizzled tensor-map store (cp.async.bulk.tensor.2d, SASS UTMASTG): no
//     thread computes a global address, every HBM write is a full line, and the unpack runs with immediate offsets
#include "blocks.cuh"
#include "umma.cuh"

namespace ggufb200 {

constexpr int kThreads = 128;       // threads per CTA of the dequant kernel = 4096-element tiles (256: 0.929, 64: 0.80 of the copy peak on the Flux-shape sweep)

int g_dequant_pdl = 1;          // programmatic dependent launch of the dequant kernel; ggufb200_set_tuning(1, 0/1)
int g_dequant_prefetch = 1;     // L2 prefetch distance of the dequant kernel in waves (0 = off); ggufb200_set_tuning(3, n)

// Store into the OUTPUT tile.  No "memory" clobber: the output tile never aliases the packed tile the unpack reads, so the
// compiler may keep the bytes it has already loaded (the high nibbles of a 4-bit block sit in the same bytes as the low ones)
// across these stores; `volatile` keeps them in order before the fence + barrier that publish the tile.
__device__ __forceinline__ void st_otile_v4(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d));
}

// One thread = one run of 32 consecutive elements of the packed tile at `tile` (shared memory).  The output tile is laid out for
// a swizzled 2-D tensor-map store, one row per thread (fp16 / bf16: 64-byte rows, CU_TENSOR_MAP_SWIZZLE_64B; fp32: 128-byte rows,
// SWIZZLE_128B): 16-byte chunk p of a row sits at chunk p ^ (address bits 7.. of the row), so the chunks are processed in their
// natural order -- every byte offset and shift of the unpack is an immediate -- and the STS.128 of a quarter-warp still hit eight
// different bank groups.  (A linear tile needs the chunk ORDER rotated per lane instead: dynamic offsets and shifts, 7-17 % more
// instructions, 0.951 instead of 0.997 of the copy peak on the Flux-shape sweep -- profiles/r02_k1_variants_ab.log.)
template <class Q, int MATH, int OUT>
__device__ __forceinline__ void dequant_tile(const uint8_t *tile, uint8_t *otile, int tile_elems, int tid)
{
    constexpr int OB = OutT<OUT>::bytes;
    constexpr int EPC = 16 / OB;                           // elements per 16-byte chunk: 8 or 4
    constexpr int CH = 32 / EPC;                           // chunks per thread: 4 or 8
    constexpr int GROUP = GroupOf<Q>::value;
    const int blk_in_tile = (tid * 32) / Q::BS;
    const int e0 = (tid * 32) % Q::BS;
    if (tid * 32 < tile_elems) {
        const uint8_t *blk = tile + blk_in_tile * Q::TS;
        const GroupScale<MATH> g0 = group_scale<Q, MATH>(blk, e0);
        GroupScale<MATH> g1 = g0;
        if constexpr (GROUP == 16) g1 = group_scale<Q, MATH>(blk, e0 + 16);
        const uint32_t obase = smem_u32(otile) + tid * (32 * OB);
        const uint32_t sw = (obase >> 7) & (CH - 1);       // the engine's swizzle key: shared-memory address bits 7-8 (64B mode) / 7-9 (128B mode)
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int e = e0 + c * EPC;
            const bool second = (GROUP == 16) && (c * EPC >= 16);
            typename Math<MATH>::T2 v[EPC / 2];
            dequant_elems<Q, MATH, EPC>(blk, e, second ? g1 : g0, v);
            const uint32_t oaddr = obase + ((uint32_t)c ^ sw) * 16;
            if constexpr (OUT == kF32) {
                float2 f0 = Math<MATH>::to_f32x2(v[0]), f1 = Math<MATH>::to_f32x2(v[1]);
                st_otile_v4(oaddr, __float_as_uint(f0.x), __float_as_uint(f0.y), __float_as_uint(f1.x), __float_as_uint(f1.y));
            } else {
                st_otile_v4(oaddr, pack16<OUT, MATH>(v[0]), pack16<OUT, MATH>(v[1]), pack16<OUT, MATH>(v[2]), pack16<OUT, MATH>(v[3]));
            }
        }
    }
}

// One tile per CTA (see the file header).  flags: bit 0 = the packed pointer is 16-byte aligned (bulk copy legal),
// bit 1 = GGUFB200_DEQUANT_SRC_STABLE.  pf_tiles > 0: once its own tile is requested, the CTA asks L2 for the packed tile
// pf_tiles further on (one wave of resident CTAs ahead), so the CTA that later takes that slot finds its bytes in L2.
template <class Q, int MATH, int OUT, int THREADS>
__global__ void __launch_bounds__(THREADS) dequant_kernel(const __grid_constant__ CUtensorMap tmOut, const uint8_t *__restrict__ src,
                                                          void *__restrict__ dst, long long n_blocks, int flags, int pf_tiles)
{
    constexpr int OB = OutT<OUT>::bytes;
    constexpr int TILE_ELEMS = THREADS * 32;
    constexpr int TILE_BLOCKS = TILE_ELEMS / Q::BS;
    constexpr int TILE_BYTES = TILE_BLOCKS * Q::TS;
    static_assert(TILE_BYTES % 16 == 0, "tile byte span must be a multiple of 16");
    static_assert(TILE_ELEMS % Q::BS == 0, "tile shape");
    const int bulk_ok = flags & 1;
    const bool early = bulk_ok && (flags & 2);

    // output tile first (the swizzle pattern of the tensor-map store is a function of the shared-memory ADDRESS bits; the
    // threads derive their key from the address too, so the two agree wherever the window starts)
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *otile = smem;
    uint8_t *tile = smem + TILE_ELEMS * OB;
    uint64_t *full = reinterpret_cast<uint64_t *>(tile + ((TILE_BYTES + 16 + 15) & ~15));

    const int tid = threadIdx.x;
    const long long t = blockIdx.x;
    const long long total_bytes = n_blocks * (long long)Q::TS;
    const long long n_elems = n_blocks * (long long)Q::BS;
    long long off = t * (long long)TILE_BYTES;
    long long len = total_bytes - off;
    if (len > TILE_BYTES) len = TILE_BYTES;

    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (bulk_ok) {
        // Only thread 0 touches the mbarrier (init, copy, wait); the other 255 threads sleep in the CTA barrier instead of
        // polling, so the warps of the SM's other CTAs that are unpacking get the issue slots.
        if (tid == 0) {
            mbar_init(full, 1);
            fence_mbar_init();
            if (!early) asm volatile("griddepcontrol.wait;" ::: "memory");
            uint32_t bytes = (uint32_t)((len + 15) & ~15LL);
            mbar_arrive_expect_tx(full, bytes);
            bulk_g2s(tile, src + off, bytes, full);
            if (pf_tiles > 0) {
                // whole 16-byte units inside the tensor only: the prefetch never reaches past its last byte
                const long long poff = off + (long long)pf_tiles * TILE_BYTES;
                long long plen = total_bytes - poff;
                if (plen > TILE_BYTES) plen = TILE_BYTES;
                plen &= ~15LL;
                if (plen > 0)
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src + poff), "r"((uint32_t)plen) : "memory");
            }
            mbar_wait(full, 0);
        }
    } else {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        for (int i = tid; i < (int)len; i += THREADS) tile[i] = src[off + i];
    }
    __syncthreads();
    const long long elem_base = t * (long long)TILE_ELEMS;
    const long long left = n_elems - elem_base;
    const int tile_elems = left < TILE_ELEMS ? (int)left : TILE_ELEMS;
    dequant_tile<Q, MATH, OUT>(tile, otile, tile_elems, tid);
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
        if (early) asm volatile("griddepcontrol.wait;" ::: "memory");
        // one box = this tile's THREADS rows; rows past the end of the tensor (short last tile) are clipped by the TMA engine
        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(&tmOut)),
                     "r"(smem_u32(otile)), "r"(0), "r"((int)(t * THREADS))
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");      // the shared-memory tile must outlive the engine's read of it
    }
}

// BF16 "quantised" type (dequant.py:61-62): widen to fp32, then cast to the output dtype
template <int OUT> __global__ void __launch_bounds__(kThreads) bf16_kernel(const uint16_t *__restrict__ src, void *__restrict__ dst, long long n)
{
    using O = typename OutT<OUT>::type;
    O *out = reinterpret_cast<O *>(dst);
    const long long stride = (long long)gridDim.x * kThreads;
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
    const long long n8 = vec_ok ? n / 8 : 0;
    for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n8; i += stride) {
        uint4 w = *reinterpret_cast<const uint4 *>(src + i * 8);
        uint32_t ws[4] = {w.x, w.y, w.z, w.w};
        if constexpr (OUT == kBF16) {
            st_global_v4(out + i * 8, ws[0], ws[1], ws[2], ws[3]);
        } else if constexpr (OUT == kF32) {
            st_global_v4(out + i * 8, ws[0] << 16, ws[0] & 0xFFFF0000u, ws[1] << 16, ws[1] & 0xFFFF0000u);
            st_global_v4(out + i * 8 + 4, ws[2] << 16, ws[2] & 0xFFFF0000u, ws[3] << 16, ws[3] & 0xFFFF0000u);
        } else {
            uint32_t r[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                __half2 h = __floats2half2_rn(__uint_as_float(ws[j] << 16), __uint_as_float(ws[j] & 0xFFFF0000u));
                r[j] = *reinterpret_cast<uint32_t *>(&h);
            }
            st_global_v4(out + i * 8, r[0], r[1], r[2], r[3]);
        }
    }
    for (long long i = n8 * 8 + (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
        float f = __uint_as_float((uint32_t)src[i] << 16);
        if constexpr (OUT == kF16) out[i] = __float2half_rn(f);
        else if constexpr (OUT == kBF16) out[i] = __float2bfloat16_rn(f);
        else out[i] = f;
    }
}

// integer-unpack debug kernel: exercises exactly the q4()/scales() the product kernels use
template <class Q>
__global__ void unpack_int_kernel(const uint8_t *__restrict__ src, long long n_blocks, int16_t *q, int16_t *sc, int16_t *mn)
{
    const long long n4 = n_blocks * (Q::BS / 4);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / (Q::BS / 4);
        const int e0 = (int)(i % (Q::BS / 4)) * 4;
        // global pointers carry no alignment guarantee here -> byte-assemble through a local copy
        uint8_t local[Q::TS + 2] __attribute__((aligned(16)));
        for (int k = 0; k < Q::TS; ++k) local[k] = src[b * Q::TS + k];
        uint32_t u = Q::q4(local, e0);
        int s, m;
        Q::scales(local, e0, s, m);
        for (int j = 0; j < 4; ++j) {
            long long o = b * Q::BS + e0 + j;
            if (q) q[o] = (int16_t)((int)((u >> (8 * j)) & 0xFF) - Q::BIAS);
            if (sc) sc[o] = (int16_t)s;
            if (mn) mn[o] = (int16_t)m;
        }
    }
}

// ------------------------------------------------------------------ host-side dispatch
template <class Q, int MATH, int OUT> static int launch_dequant(const void *packed, long long n_blocks, void *out, bool src_stable, cudaStream_t st)
{
    constexpr int THREADS = kThreads;
    constexpr int TILE_BLOCKS = THREADS * 32 / Q::BS;
    constexpr int OB = OutT<OUT>::bytes;
    constexpr int TB = ((TILE_BLOCKS * Q::TS + 16 + 15) & ~15);
    constexpr int SMEM = THREADS * 32 * OB + TB + 16;
    auto kern = dequant_kernel<Q, MATH, OUT, THREADS>;
    static unsigned char smem_set[64] = {};
    if (!ensure_dynamic_smem(kern, SMEM, smem_set)) return GGUFB200_E_CUDA;
    const long long n_tiles = (n_blocks + TILE_BLOCKS - 1) / TILE_BLOCKS;
    if (n_tiles > 0x7fffffffll) return GGUFB200_E_SHAPE;
    CUtensorMap tmOut{};
    {
        // the output as [runs of 32 elements][64 | 128 bytes]: one row per thread, one box of THREADS rows per tile
        G2EncodeFn fn = g2_encode_fn();
        const long long n_rows = n_blocks * (long long)Q::BS / 32;
        if (!fn || n_rows > 0x7fffffffll) return GGUFB200_E_CUDA;
        cuuint64_t dims[2] = {(cuuint64_t)(32 * OB), (cuuint64_t)n_rows};
        cuuint64_t strides[1] = {(cuuint64_t)(32 * OB)};
        cuuint32_t box[2] = {(cuuint32_t)(32 * OB), (cuuint32_t)THREADS};
        cuuint32_t estr[2] = {1, 1};
        if (fn(&tmOut, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, out, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               OB == 2 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return GGUFB200_E_CUDA;
    }
    int flags = ((reinterpret_cast<uintptr_t>(packed) & 15) == 0) ? 1 : 0;
    if (src_stable) flags |= 2;
    // one wave = the CTAs resident on the whole GPU at once (occupancy query, once per device)
    static int wave[64] = {};
    const int dev = device_slot();
    if (dev < 0) return GGUFB200_E_CUDA;
    if (wave[dev] == 0) {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, SMEM) != cudaSuccess || per_sm <= 0) return GGUFB200_E_CUDA;
        wave[dev] = per_sm * sm_count();
    }
    const long long pf = (long long)g_dequant_prefetch * wave[dev];
    const int pf_tiles = pf < n_tiles ? (int)pf : 0;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)n_tiles);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = SMEM;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_dequant_pdl ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmOut, reinterpret_cast<const uint8_t *>(packed), out, (long long)n_blocks, flags, pf_tiles);
    return e == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
}

int dequant_dispatch(int type, const void *packed, long long n_blocks, void *out, int out_dtype, int math_dtype, cudaStream_t st, bool stable)
{
    if (n_blocks == 0) return GGUFB200_OK;
    if (type == T_BF16) {
        // one 8-element vector per thread, CTAs in address order (the grid-stride loop of the kernel only runs past the first
        // iteration for tensors beyond 2^31 CTAs): same reasoning as for the block formats above
        long long blocks = (n_blocks + (long long)kThreads * 8 - 1) / ((long long)kThreads * 8);
        long long cap = 0x7fffffffll;
        unsigned grid = (unsigned)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
        const uint16_t *s = reinterpret_cast<const uint16_t *>(packed);
        if (out_dtype == kF16) bf16_kernel<kF16><<<grid, kThreads, 0, st>>>(s, out, n_blocks);
        else if (out_dtype == kBF16) bf16_kernel<kBF16><<<grid, kThreads, 0, st>>>(s, out, n_blocks);
        else if (out_dtype == kF32) bf16_kernel<kF32><<<grid, kThreads, 0, st>>>(s, out, n_blocks);
        else return GGUFB200_E_DTYPE;
        return cudaGetLastError() == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
    }
    return with_block(type, (int)GGUFB200_E_TYPE, [&](auto q) {
        return with_dtype(math_dtype, [&](auto math) {
            return with_dtype(out_dtype, [&](auto o) {
                return launch_dequant<decltype(q), math.value, o.value>(packed, n_blocks, out, stable, st);
            });
        });
    });
}

template <class Q> static int launch_unpack(const void *packed, long long n_blocks, int16_t *q, int16_t *sc, int16_t *mn, cudaStream_t st)
{
    long long n4 = n_blocks * (Q::BS / 4);
    long long blocks = (n4 + 127) / 128;
    if (blocks > 65535) blocks = 65535;
    unpack_int_kernel<Q><<<(unsigned)blocks, 128, 0, st>>>(reinterpret_cast<const uint8_t *>(packed), n_blocks, q, sc, mn);
    return cudaGetLastError() == cudaSuccess ? GGUFB200_OK : GGUFB200_E_CUDA;
}

int unpack_dispatch(int type, const void *packed, long long n_blocks, int16_t *q, int16_t *sc, int16_t *mn, cudaStream_t st)
{
    if (n_blocks == 0) return GGUFB200_OK;
    return with_block(type, (int)GGUFB200_E_TYPE, [&](auto b) { return launch_unpack<decltype(b)>(packed, n_blocks, q, sc, mn, st); });
}

}  // namespace ggufb200
