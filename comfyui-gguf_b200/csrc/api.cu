// api.cu -- the extern "C" boundary declared in include/ggufb200.h.
// Argument validation and route selection live here; kernels live in dequant.cu / rows.cu / gemv.cu / gemm2.cu /
// gemm3.cu / gemm4.cu / repack.cu.  Routing is a pure function of the call's arguments (algo | flags): no process-wide
// routing state.
#include <stdlib.h>

#include "blocks.cuh"

namespace ggufb200 {
extern int g_dequant_pdl;
extern int g_dequant_prefetch;
extern int g_gemv2_ctas;
int dequant_dispatch(int type, const void *packed, long long n_blocks, void *out, int out_dtype, int math_dtype, cudaStream_t st, bool stable = false);
int unpack_dispatch(int type, const void *packed, long long n_blocks, int16_t *q, int16_t *sc, int16_t *mn, cudaStream_t st);
int rows_dispatch(int type, const void *packed, long long n_table_rows, long long K, const long long *rows, long long n_rows,
                  void *out, int out_dtype, int math_dtype, cudaStream_t st);
int gemv_dispatch(int type, const void *W, long long N, long long K, const void *X, long long M, long long ldx, int act_dtype,
                  int math_dtype, const void *bias, int bias_dtype, void *Y, long long ldy, cudaStream_t st);
int gemm2_fused_dispatch(int type, const void *W, long long N, long long K, const void *X, long long M, long long ldx, int act_dtype,
                         int math_dtype, const void *bias, int bias_dtype, void *Y, long long ldy, void *ws, size_t ws_bytes, int flags,
                         cudaStream_t st);
int gemm2_fused_splits(long long M, long long N, long long K);
void gemm2_fused_plan_info(long long M, long long N, long long K, size_t ws_bytes, int flags, int *accs, int *splits, int *kb_per_split, int *ctas);
int gemm3_dense_dispatch(const void *W, long long N, long long K, long long ldw, const void *X, long long M, long long ldx,
                         int act_dtype, const void *bias, int bias_dtype, void *Y, long long ldy, cudaStream_t st);
int gemm4_fused_dispatch(int type, const void *W, const void *Wspan, long long span_stride, long long N, long long K, const void *X, long long M,
                         long long ldx, int act_dtype, const void *bias, int bias_dtype, void *Y, long long ldy, void *ws, size_t ws_bytes,
                         int flags, const void *loraT, long long ldt, const void *loraU, cudaStream_t st);
bool gemm4_supported(int type, const void *W, long long N, long long K);
size_t gemm4_workspace(long long M, long long N, long long K, int flags);
void gemm4_plan_info(long long M, long long N, long long K, size_t ws_bytes, int flags, int *tile_tokens, int *splits, int *spans_per_split, int *items);
int gemv_max_m();
bool gemv2_supported(int type, const void *W, long long N, long long K, long long M);
int gemv2_dispatch(int type, const void *W, long long N, long long K, const void *X, long long M, long long ldx, int act_dtype, const void *bias,
                   int bias_dtype, void *Y, long long ldy, cudaStream_t st, bool w_stable = false);
size_t repack_bytes(int type, long long N, long long K, int *pitch, long long *span_stride);
int repack_dispatch(int type, const void *W, long long N, long long K, void *out, cudaStream_t st);
}  // namespace ggufb200

using namespace ggufb200;

// block size (elements) and type size (bytes) of a ggml type; BF16 counts as blocks of one 2-byte element
static bool type_geom(int t, int *bs, int *ts)
{
    int b = 1, s = 2;
    const bool ok = t == T_BF16 || with_block(t, false, [&](auto q) {
        b = decltype(q)::BS;
        s = decltype(q)::TS;
        return true;
    });
    if (ok && bs) *bs = b;
    if (ok && ts) *ts = s;
    return ok;
}

static bool dtype_ok(int d) { return d >= 0 && d <= 2; }
static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static bool fused_type(int t) { return with_block(t, false, [](auto) { return true; }); }     // every block format has a fused producer

// ------------------------------------------------------------------ device gate
// The library contains sm_100a code only.  Checked once per device, right before the first launch on it (argument
// errors are still reported without a GPU).
static int device_check()
{
    static signed char ok[64] = {};     // 0 = unknown, 1 = sm_100, -1 = something else
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        return GGUFB200_E_CUDA;
    }
    if (dev < 0 || dev >= 64) return GGUFB200_OK;
    if (ok[dev] == 0) {
        int major = 0, minor = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev) != cudaSuccess) {
            cudaGetLastError();
            return GGUFB200_E_CUDA;
        }
        ok[dev] = (major == 10 && minor == 0) ? 1 : -1;
    }
    return ok[dev] == 1 ? GGUFB200_OK : GGUFB200_E_DEVICE;
}

// ------------------------------------------------------------------ route selection
// Fallback thresholds (round 1) for weights the TMEM-fed kernel cannot stage: short activations split-K fused through shared
// memory, long activations dequant once into the workspace + dense tcgen05 GEMM.
static bool exact_prefers_fused(long long M, long long N, long long K)
{
    if ((K % 64) != 0) return false;
    if (M > 1024) return false;
    const int splits = gemm2_fused_splits(M, N, K);
    if (splits >= 4 || (splits >= 2 && K >= 2 * N)) return true;
    if (splits >= 2) return false;
    return M > 256 && N >= 12288;
}

struct Route {
    int algo;          // GGUFB200_ALGO_* without flags
    size_t ws;         // workspace bytes the route wants (0 = none)
};

static size_t fused_mma_ws(long long M, long long N, long long K, int flags)
{
    if (flags & GGUFB200_FLAG_NOSPLIT) return 0;
    const int s = gemm2_fused_splits(M, N, K);
    return s > 1 ? (size_t)s * (size_t)M * (size_t)N * 4 : 0;
}

// `W` may be NULL (workspace query: assume a 16-byte aligned weight); ws_avail = workspace the caller supplied (SIZE_MAX in a query);
// have_spans: the caller also holds the re-packed span-major copy of the weight (ggufb200_repack), which the TMEM-fed
// kernel can stage for every block format and every K
static Route pick_route(int type, const void *W, long long M, long long N, long long K, int math, int algo_flags, size_t ws_avail,
                        bool have_spans = false)
{
    const int algo = algo_flags & GGUFB200_ALGO_MASK;
    const int flags = algo_flags & ~GGUFB200_ALGO_MASK;
    const size_t dense = (size_t)N * (size_t)K * 2;
    const bool w_ok = !W || aligned16(W);
    const bool fusable = fused_type(type) && math == kF16 && (K % 64) == 0 && (N % 8) == 0;
    Route r{algo, 0};
    if (algo == GGUFB200_ALGO_AUTO) {
        // Measured on B200 (profiles/r02_bench_linear_*.log, r02_bench_gemv*.log).  The TMEM-fed fused kernel is the route for
        // every M > 8 (with EXACT_W it runs the reference-sequence producers at the same speed: it is tensor-pipe bound) and for
        // M <= 8 on large weights; the mma.sync GEMV keeps small weights at M <= 8 (its fixed cost is lower).  A math dtype other
        // than fp16 means the reference's own sequence in that dtype: standalone dequant + dense GEMM (or the GEMV).
        const bool tmem_ok = w_ok && fused_type(type) && math == kF16 && (N % 8) == 0 && (have_spans || gemm4_supported(type, W, N, K));
        const bool exact = (flags & GGUFB200_FLAG_EXACT_W) != 0 || math != kF16;
        if (!w_ok) r.algo = GGUFB200_ALGO_DEQUANT_MMA;
        else if (M <= gemv_max_m() && !exact && gemv2_supported(type, W ? W : (const void *)16, N, K, M)) r.algo = GGUFB200_ALGO_GEMV_FAST;
        else if (M <= gemv_max_m()) r.algo = (tmem_ok && (long long)N * K >= (40ll << 20)) ? GGUFB200_ALGO_FUSED_TMEM : GGUFB200_ALGO_GEMV;
        else if (tmem_ok) r.algo = GGUFB200_ALGO_FUSED_TMEM;
        else if (fusable && (exact_prefers_fused(M, N, K) || ws_avail < dense)) r.algo = GGUFB200_ALGO_FUSED_MMA;
        else r.algo = GGUFB200_ALGO_DEQUANT_MMA;
    }
    switch (r.algo) {
    case GGUFB200_ALGO_DEQUANT_MMA: r.ws = dense; break;
    case GGUFB200_ALGO_FUSED_MMA: r.ws = fusable ? fused_mma_ws(M, N, K, flags) : 0; break;
    case GGUFB200_ALGO_FUSED_TMEM: r.ws = gemm4_workspace(M, N, K, flags); break;
    default: r.ws = 0;
    }
    return r;
}

extern "C" {

int ggufb200_version(void) { return GGUFB200_VERSION; }

const char *ggufb200_strerror(int rc)
{
    switch (rc) {
    case GGUFB200_OK: return "ok";
    case GGUFB200_E_TYPE: return "unsupported ggml quantization type (no CPU fallback is provided)";
    case GGUFB200_E_DTYPE: return "dtype code must be 0 (float16), 1 (bfloat16) or 2 (float32)";
    case GGUFB200_E_ALIGN: return "output / activation pointers must be 16-byte aligned";
    case GGUFB200_E_SHAPE: return "bad shape: sizes must be non-negative, K a multiple of the block size, ld >= row length";
    case GGUFB200_E_NULL: return "required pointer is NULL";
    case GGUFB200_E_CUDA: return "CUDA launch failed";
    case GGUFB200_E_WORKSPACE: return "workspace too small (see ggufb200_linear_workspace)";
    case GGUFB200_E_UNSUPPORTED: return "operation not implemented for this type / dtype / shape combination";
    case GGUFB200_E_DEVICE: return "current CUDA device is not sm_100 (B200)";
    }
    return "unknown error";
}

int ggufb200_type_info(int ggml_type, int *block_size, int *type_size)
{
    return type_geom(ggml_type, block_size, type_size) ? GGUFB200_OK : GGUFB200_E_TYPE;
}

int ggufb200_supported(int ggml_type, int op)
{
    if (!type_geom(ggml_type, nullptr, nullptr)) return 0;
    switch (op) {
    case GGUFB200_OP_DEQUANT: return 1;
    case GGUFB200_OP_ROWS: return 1;
    case GGUFB200_OP_LINEAR: return 1;
    case GGUFB200_OP_LINEAR_MMA: return 1;   // a fused kernel, or dequant + tensor-core GEMM for types / shapes it does not cover
    }
    return 0;
}

int ggufb200_set_tuning(int key, int value)
{
    static const bool allowed = [] {
        const char *e = getenv("GGUFB200_ALLOW_TUNING");
        return e && e[0] == '1';
    }();
    if (!allowed) return GGUFB200_E_UNSUPPORTED;
    if (key == 1) {
        g_dequant_pdl = value ? 1 : 0;
        return GGUFB200_OK;
    }
    if (key == 2) {
        g_gemv2_ctas = value;
        return GGUFB200_OK;
    }
    if (key == 3 && value >= 0 && value <= 8) {
        g_dequant_prefetch = value;
        return GGUFB200_OK;
    }
    return GGUFB200_E_UNSUPPORTED;
}

int ggufb200_dequant(int ggml_type, const void *packed, int64_t n_blocks, void *out, int out_dtype, int math_dtype, void *stream)
{
    if (!type_geom(ggml_type, nullptr, nullptr)) return GGUFB200_E_TYPE;
    const bool stable = (math_dtype & GGUFB200_DEQUANT_SRC_STABLE) != 0;
    math_dtype &= ~GGUFB200_DEQUANT_SRC_STABLE;
    if (!dtype_ok(out_dtype) || !dtype_ok(math_dtype)) return GGUFB200_E_DTYPE;
    if (n_blocks < 0) return GGUFB200_E_SHAPE;
    if (n_blocks == 0) return GGUFB200_OK;
    if (!packed || !out) return GGUFB200_E_NULL;
    if (!aligned16(out)) return GGUFB200_E_ALIGN;
    if (int rc = device_check()) return rc;
    return dequant_dispatch(ggml_type, packed, n_blocks, out, out_dtype, math_dtype, (cudaStream_t)stream, stable);
}

int ggufb200_unpack_int(int ggml_type, const void *packed, int64_t n_blocks, int16_t *q, int16_t *sc, int16_t *mn, void *stream)
{
    if (!type_geom(ggml_type, nullptr, nullptr) || ggml_type == T_BF16) return GGUFB200_E_TYPE;
    if (n_blocks < 0) return GGUFB200_E_SHAPE;
    if (n_blocks == 0) return GGUFB200_OK;
    if (!packed) return GGUFB200_E_NULL;
    if (int rc = device_check()) return rc;
    return unpack_dispatch(ggml_type, packed, n_blocks, q, sc, mn, (cudaStream_t)stream);
}

int ggufb200_dequant_rows(int ggml_type, const void *packed, int64_t n_table_rows, int64_t K, const int64_t *rows, int64_t n_rows,
                          void *out, int out_dtype, int math_dtype, void *stream)
{
    int bs, ts;
    if (!type_geom(ggml_type, &bs, &ts)) return GGUFB200_E_TYPE;
    if (!dtype_ok(out_dtype) || !dtype_ok(math_dtype)) return GGUFB200_E_DTYPE;
    if (n_rows < 0 || n_table_rows < 0 || K <= 0 || K % bs != 0 || K % 8 != 0) return GGUFB200_E_SHAPE;
    if (n_rows == 0) return GGUFB200_OK;
    if (!packed || !rows || !out) return GGUFB200_E_NULL;
    if (!aligned16(out)) return GGUFB200_E_ALIGN;
    if (int rc = device_check()) return rc;
    return rows_dispatch(ggml_type, packed, n_table_rows, K, (const long long *)rows, n_rows, out, out_dtype, math_dtype,
                         (cudaStream_t)stream);
}

size_t ggufb200_linear_workspace_ex(int ggml_type, int64_t M, int64_t N, int64_t K, int act_dtype, int math_dtype, int algo)
{
    if (!type_geom(ggml_type, nullptr, nullptr) || N <= 0 || K <= 0 || M <= 0) return 0;
    return pick_route(ggml_type, nullptr, M, N, K, math_dtype, algo, (size_t)-1).ws;
}

size_t ggufb200_linear_workspace(int ggml_type, int64_t M, int64_t N, int64_t K, int act_dtype, int algo)
{
    return ggufb200_linear_workspace_ex(ggml_type, M, N, K, act_dtype, kF16, algo);
}

struct LoraSide {
    const void *T;      // [M, 64] activation dtype: x * down^T, zero padded beyond the rank
    int64_t ldt;
    const void *U;      // [N, 64] fp16: scale * up, zero padded
};

static int linear_impl(int ggml_type, const void *W_packed, const void *W_spans, int64_t N, int64_t K, const void *X, int64_t M, int64_t ldx,
                       int act_dtype, int math_dtype, const void *bias, int bias_dtype, void *Y, int64_t ldy, void *workspace,
                       size_t workspace_bytes, int algo, void *stream, const LoraSide *lora = nullptr)
{
    int bs, ts;
    if (!type_geom(ggml_type, &bs, &ts)) return GGUFB200_E_TYPE;
    if (act_dtype != kF16 && act_dtype != kBF16) return GGUFB200_E_DTYPE;
    if (!dtype_ok(math_dtype) || (bias && !dtype_ok(bias_dtype))) return GGUFB200_E_DTYPE;
    if (M < 0 || N <= 0 || K <= 0 || K % bs != 0 || K % 8 != 0 || ldx < K || ldy < N) return GGUFB200_E_SHAPE;
    if (M == 0) return GGUFB200_OK;
    if (!W_packed || !X || !Y) return GGUFB200_E_NULL;
    const int flags = algo & ~GGUFB200_ALGO_MASK;
    const bool w_ok = aligned16(W_packed);
    const size_t dense = (size_t)N * (size_t)K * 2;
    const size_t ws_avail = (workspace && aligned16(workspace)) ? workspace_bytes : 0;
    // The fused producers read the packed rows with the per-format natural alignment (up to 16 bytes).  A packed tensor
    // that does not start on a 16-byte boundary (never produced by torch allocations, only by byte-offset views) is
    // always routed through the standalone dequant kernel, which stages any alignment, plus the dense GEMM.
    if (!w_ok) {
        if (ws_avail < dense) return GGUFB200_E_ALIGN;
        algo = GGUFB200_ALGO_DEQUANT_MMA | flags;
    }
    if (W_spans && !aligned16(W_spans)) return GGUFB200_E_ALIGN;
    const Route r = pick_route(ggml_type, W_packed, M, N, K, math_dtype, algo, ws_avail, W_spans != nullptr);
    // the small-M kernel stores per element: it only needs 2-byte aligned Y rows; every other route moves 16-byte vectors
    const bool vec_y = r.algo != GGUFB200_ALGO_GEMV && r.algo != GGUFB200_ALGO_GEMV_FAST;
    if (!aligned16(X) || (ldx % 8) != 0) return GGUFB200_E_ALIGN;
    if (vec_y && (!aligned16(Y) || (ldy % 8) != 0)) return GGUFB200_E_ALIGN;
    if (workspace && !aligned16(workspace) && r.ws) return GGUFB200_E_ALIGN;
    if (lora) {     // the rank-r update rides as one extra k-block of the TMEM-fed kernel: no other route can carry it
        if (r.algo != GGUFB200_ALGO_FUSED_TMEM) return GGUFB200_E_UNSUPPORTED;
        if (!lora->T || !lora->U) return GGUFB200_E_NULL;
        if (!aligned16(lora->T) || !aligned16(lora->U) || lora->ldt < 64 || (lora->ldt % 8) != 0) return GGUFB200_E_ALIGN;
    }
    if (int rc = device_check()) return rc;
    cudaStream_t st = (cudaStream_t)stream;

    switch (r.algo) {
    case GGUFB200_ALGO_GEMV:
        return gemv_dispatch(ggml_type, W_packed, N, K, X, M, ldx, act_dtype, math_dtype, bias, bias_dtype, Y, ldy, st);
    case GGUFB200_ALGO_GEMV_FAST:
        if (math_dtype != kF16 || (flags & GGUFB200_FLAG_EXACT_W)) return GGUFB200_E_UNSUPPORTED;
        return gemv2_dispatch(ggml_type, W_packed, N, K, X, M, ldx, act_dtype, bias, bias_dtype, Y, ldy, st, (flags & GGUFB200_FLAG_W_STABLE) != 0);
    case GGUFB200_ALGO_FUSED_MMA:
        if (!fused_type(ggml_type)) return GGUFB200_E_UNSUPPORTED;
        return gemm2_fused_dispatch(ggml_type, W_packed, N, K, X, M, ldx, act_dtype, math_dtype, bias, bias_dtype, Y, ldy, workspace,
                                    ws_avail, flags, st);
    case GGUFB200_ALGO_FUSED_TMEM: {
        if (!fused_type(ggml_type) || math_dtype != kF16) return GGUFB200_E_UNSUPPORTED;
        long long span_stride = 0;
        if (W_spans) repack_bytes(ggml_type, N, K, nullptr, &span_stride);
        return gemm4_fused_dispatch(ggml_type, W_packed, W_spans, span_stride, N, K, X, M, ldx, act_dtype, bias, bias_dtype, Y, ldy, workspace,
                                    ws_avail, flags, lora ? lora->T : nullptr, lora ? lora->ldt : 0, lora ? lora->U : nullptr, st);
    }
    case GGUFB200_ALGO_DEQUANT_MMA: {
        if (ws_avail < dense) return GGUFB200_E_WORKSPACE;
        int rc = dequant_dispatch(ggml_type, W_packed, N * (K / bs), workspace, act_dtype, math_dtype, st, (flags & GGUFB200_FLAG_W_STABLE) != 0);
        if (rc != GGUFB200_OK) return rc;
        return gemm3_dense_dispatch(workspace, N, K, K, X, M, ldx, act_dtype, bias, bias_dtype, Y, ldy, st);
    }
    }
    return GGUFB200_E_UNSUPPORTED;
}

int ggufb200_linear(int ggml_type, const void *W_packed, int64_t N, int64_t K, const void *X, int64_t M, int64_t ldx, int act_dtype,
                    int math_dtype, const void *bias, int bias_dtype, void *Y, int64_t ldy, void *workspace, size_t workspace_bytes,
                    int algo, void *stream)
{
    return linear_impl(ggml_type, W_packed, nullptr, N, K, X, M, ldx, act_dtype, math_dtype, bias, bias_dtype, Y, ldy, workspace, workspace_bytes,
                       algo, stream);
}

int ggufb200_linear_spans(int ggml_type, const void *W_packed, const void *W_spans, int64_t N, int64_t K, const void *X, int64_t M, int64_t ldx,
                          int act_dtype, int math_dtype, const void *bias, int bias_dtype, void *Y, int64_t ldy, void *workspace,
                          size_t workspace_bytes, int algo, void *stream)
{
    return linear_impl(ggml_type, W_packed, W_spans, N, K, X, M, ldx, act_dtype, math_dtype, bias, bias_dtype, Y, ldy, workspace, workspace_bytes,
                       algo, stream);
}

int ggufb200_linear_lora(int ggml_type, const void *W_packed, const void *W_spans, int64_t N, int64_t K, const void *X, int64_t M, int64_t ldx,
                         int act_dtype, const void *bias, int bias_dtype, const void *T, int64_t ldt, const void *U, void *Y, int64_t ldy,
                         void *workspace, size_t workspace_bytes, int algo, void *stream)
{
    const LoraSide side{T, ldt, U};
    return linear_impl(ggml_type, W_packed, W_spans, N, K, X, M, ldx, act_dtype, kF16, bias, bias_dtype, Y, ldy, workspace, workspace_bytes, algo,
                       stream, &side);
}

size_t ggufb200_repack_bytes(int ggml_type, int64_t N, int64_t K)
{
    int bs;
    if (!type_geom(ggml_type, &bs, nullptr) || N <= 0 || K <= 0 || K % bs != 0) return 0;
    return repack_bytes(ggml_type, N, K, nullptr, nullptr);
}

int ggufb200_repack(int ggml_type, const void *W_packed, int64_t N, int64_t K, void *out, void *stream)
{
    int bs;
    if (!type_geom(ggml_type, &bs, nullptr) || ggml_type == T_BF16) return GGUFB200_E_TYPE;
    if (N <= 0 || K <= 0 || K % bs != 0) return GGUFB200_E_SHAPE;
    if (!W_packed || !out) return GGUFB200_E_NULL;
    if (!aligned16(out) || (reinterpret_cast<uintptr_t>(W_packed) & 1)) return GGUFB200_E_ALIGN;
    if (int rc = device_check()) return rc;
    return repack_dispatch(ggml_type, W_packed, N, K, out, (cudaStream_t)stream);
}

int ggufb200_linear_plan(int ggml_type, int64_t M, int64_t N, int64_t K, size_t workspace_bytes, int algo, int *tile_rows, int *k_ranges,
                         int *kblocks_per_range, int *ctas)
{
    if (!type_geom(ggml_type, nullptr, nullptr)) return GGUFB200_E_TYPE;
    if (!tile_rows || !k_ranges || !kblocks_per_range || !ctas) return GGUFB200_E_NULL;
    if (M <= 0 || N <= 0 || K <= 0 || K % 64 != 0 || N % 8 != 0) return GGUFB200_E_SHAPE;
    if (!fused_type(ggml_type)) return GGUFB200_E_UNSUPPORTED;
    const int flags = algo & ~GGUFB200_ALGO_MASK;
    if ((algo & GGUFB200_ALGO_MASK) == GGUFB200_ALGO_FUSED_TMEM) {
        int spans = 1;
        gemm4_plan_info(M, N, K, workspace_bytes, flags, tile_rows, k_ranges, &spans, ctas);
        *kblocks_per_range = 4 * spans;
        return GGUFB200_OK;
    }
    if ((algo & GGUFB200_ALGO_MASK) != GGUFB200_ALGO_FUSED_MMA) return GGUFB200_E_UNSUPPORTED;
    int accs = 1;
    gemm2_fused_plan_info(M, N, K, workspace_bytes, flags, &accs, k_ranges, kblocks_per_range, ctas);
    *tile_rows = 256 * accs;
    return GGUFB200_OK;
}

int ggufb200_gemm(const void *W, int64_t N, int64_t K, int64_t ldw, const void *X, int64_t M, int64_t ldx, int act_dtype,
                  const void *bias, int bias_dtype, void *Y, int64_t ldy, void *stream)
{
    if (act_dtype != kF16 && act_dtype != kBF16) return GGUFB200_E_DTYPE;
    if (bias && !dtype_ok(bias_dtype)) return GGUFB200_E_DTYPE;
    if (M < 0 || N <= 0 || K <= 0 || K % 8 != 0 || ldw < K || ldx < K || ldy < N) return GGUFB200_E_SHAPE;
    if (M == 0) return GGUFB200_OK;
    if (!W || !X || !Y) return GGUFB200_E_NULL;
    if (!aligned16(W) || !aligned16(X) || !aligned16(Y) || (ldw % 8) || (ldx % 8) || (ldy % 8)) return GGUFB200_E_ALIGN;
    if (int rc = device_check()) return rc;
    return gemm3_dense_dispatch(W, N, K, ldw, X, M, ldx, act_dtype, bias, bias_dtype, Y, ldy, (cudaStream_t)stream);
}

}  // extern "C"
