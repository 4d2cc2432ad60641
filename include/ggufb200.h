/*
 * ggufb200.h -- C ABI of libggufb200.so: B200 (sm_100a) GGUF block dequant and the
 * Linear that consumes the dequantised weight.
 *
 * This is the drop-in boundary for the hot path of city96/ComfyUI-GGUF.  The
 * reference has no native code, so each entry point names the PYTHON function it
 * replaces (reference file:line); INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer owned by the
 *     caller (PyTorch); the library never allocates, frees or retains device memory
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream)
 *   - all calls are asynchronous on `stream` and re-entrant; routing depends only on the arguments of the call
 *     (the library keeps no mutable routing state; ggufb200_set_tuning() is a benchmark-only switch that is refused
 *     unless the process opted in with GGUFB200_ALLOW_TUNING=1)
 *   - the device code is sm_100a only: calls that would launch a kernel return GGUFB200_E_DEVICE on any other GPU
 *   - return value: 0 = GGUFB200_OK, negative = error (ggufb200_strerror()); no C++
 *     exception crosses the boundary
 *   - ggml_type uses gguf-py's GGMLQuantizationType integer values
 *     (Q4_0=2 Q4_1=3 Q5_0=6 Q5_1=7 Q8_0=8 Q2_K=10 Q3_K=11 Q4_K=12 Q5_K=13 Q6_K=14
 *      IQ4_NL=20 IQ4_XS=23 BF16=30), i.e. the keys of dequant.py:287-301
 *   - dtype codes: 0 = float16, 1 = bfloat16, 2 = float32
 */
#ifndef GGUFB200_H
#define GGUFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GGUFB200_VERSION 200 /* major*10000 + minor*100 + patch */

/* error codes */
#define GGUFB200_OK 0
#define GGUFB200_E_TYPE (-1)      /* ggml_type not in dequant.py:287-301 */
#define GGUFB200_E_DTYPE (-2)     /* dtype code out of range */
#define GGUFB200_E_ALIGN (-3)     /* output / activation pointer not 16-byte aligned */
#define GGUFB200_E_SHAPE (-4)     /* K not a multiple of the block size, negative size, ld too small ... */
#define GGUFB200_E_NULL (-5)      /* required pointer is NULL */
#define GGUFB200_E_CUDA (-6)      /* a CUDA call failed (cudaGetLastError preserved for the caller) */
#define GGUFB200_E_WORKSPACE (-7) /* workspace smaller than ggufb200_linear_workspace() */
#define GGUFB200_E_UNSUPPORTED (-8) /* op / dtype combination not implemented for this type */
#define GGUFB200_E_DEVICE (-9)    /* current device is not sm_100 */

/* dtype codes */
#define GGUFB200_F16 0
#define GGUFB200_BF16 1
#define GGUFB200_F32 2

/* op codes for ggufb200_supported() */
#define GGUFB200_OP_DEQUANT 0
#define GGUFB200_OP_LINEAR 1
#define GGUFB200_OP_ROWS 2
#define GGUFB200_OP_LINEAR_MMA 3 /* large-M tcgen05 path (fused or dequant+GEMM) available for this type */

/* algorithm selector for ggufb200_linear(): one GGUFB200_ALGO_* value, optionally OR-ed with GGUFB200_FLAG_* bits */
#define GGUFB200_ALGO_AUTO 0
#define GGUFB200_ALGO_GEMV 1        /* M <= 8: fused dequant + mma.sync dot products, W bit-identical to the reference */
#define GGUFB200_ALGO_FUSED_MMA 2   /* fused dequant -> shared memory -> tcgen05.mma (W bit-identical to the reference) */
#define GGUFB200_ALGO_DEQUANT_MMA 3 /* dequant into the caller's workspace, then the tcgen05 GEMM on it (W bit-identical) */
#define GGUFB200_ALGO_FUSED_TMEM 4  /* fused dequant -> TENSOR MEMORY -> tcgen05.mma, any M (persistent; what AUTO picks for M > 8) */
#define GGUFB200_ALGO_GEMV_FAST 5   /* M <= 8, Q4_K / Q5_K: integer patterns on mma.sync, sub-block scales applied to the partial sums
                                       (W is never formed or rounded: the `fast` contract; AUTO picks it only without EXACT_W) */
#define GGUFB200_ALGO_MASK 0xFF

/* Per-call switches (no process-wide state):
 *   EXACT_W    the weight operand must be bit-identical to what the reference hands to F.linear (dequant.py float sequence with
 *              per-op rounding, then the cast to the activation dtype): FUSED_TMEM then runs its reference-sequence
 *              producers (same speed at large M: the kernel is tensor-pipe bound), every other route is exact anyway.
 *              Without it FUSED_TMEM uses the `fast` producers, whose contract is: integer unpack bit-exact; sub-block scale
 *              products as the reference; for Q4_K / Q5_K the per-element float step is ONE fused multiply-add in fp16 (the
 *              correctly rounded value of the step) instead of multiply + subtract; then the reference's cast to the
 *              activation dtype.  Result as close to the exact product as the reference's, within 1e-3 (fp16) / 8e-3
 *              (bf16, = the same bound in bf16 ulps) of the reference's.
 *   GENERIC    FUSED_TMEM: functor producers that follow the reference's rounding sequence op for op (every format; also exact)
 *   TILE384    FUSED_TMEM: force 384-token items (both accumulator slots per dequantised tile, epilogue not overlapped)
 *   TILE192    FUSED_TMEM: force 192-token items (accumulator slots alternate between items); default: a cost model picks
 *   NOSPLIT    FUSED_MMA / FUSED_TMEM: never cut K into ranges
 *   UNSTAGED   FUSED_MMA: producers read packed rows from global memory instead of TMA-staged shared memory */
#define GGUFB200_FLAG_EXACT_W 0x100
#define GGUFB200_FLAG_GENERIC 0x200
#define GGUFB200_FLAG_TILE384 0x400
#define GGUFB200_FLAG_NOSPLIT 0x800
#define GGUFB200_FLAG_UNSTAGED 0x1000
#define GGUFB200_FLAG_TILE192 0x2000 /* FUSED_TMEM: force 192-token items (double-buffered accumulators); default: cost model */
/*   W_STABLE   the caller promises that no kernel still in flight on `stream` writes W_packed (model weights: written once at
 *              load time).  The kernels are launched with programmatic stream serialization; with the promise GEMV_FAST starts
 *              streaming the packed weight into its shared-memory ring while the preceding kernel drains (the activations, the
 *              bias and Y are only touched after that kernel has completed), and DEQUANT_MMA passes
 *              GGUFB200_DEQUANT_SRC_STABLE to its dequant launch.  A kernel that does not signal programmatic completion early
 *              (every torch / cuBLAS kernel) is complete before its successor starts, so the promise only excludes producers
 *              of the packed bytes that execute griddepcontrol.launch_dependents before their last write. */
#define GGUFB200_FLAG_W_STABLE 0x4000

int ggufb200_version(void);
const char *ggufb200_strerror(int rc);

/* Block geometry: replaces gguf.GGML_QUANT_SIZES[qtype] as used at dequant.py:34. */
int ggufb200_type_info(int ggml_type, int *block_size, int *type_size);

/* 1 if (ggml_type, op) is implemented, else 0.  Mirrors `qtype in dequantize_functions`
 * (dequant.py:21, 287-301).  There is no CPU/numpy fallback (dequant.py:24-28 is NOT reproduced). */
int ggufb200_supported(int ggml_type, int op);

/*
 * Standalone dequant.  Replaces dequant.py:30-44 `dequantize()` + the per-type
 * `dequantize_blocks_*` (dequant.py:61-285) + the final `.to(dtype)` (dequant.py:23).
 *   packed     n_blocks * type_size bytes, block b covers out[b*block_size .. +block_size)
 *   out        n_blocks * block_size elements of out_dtype, 16-byte aligned
 *   math_dtype dtype the float ops run in and round to after every op: 0 (fp16) is the
 *              reference default (`dequant_dtype=None`), the activation dtype reproduces
 *              `dequant_dtype="target"`, 2 an explicit float32.  Results are bit-identical
 *              to the reference for every (math_dtype, out_dtype) pair.
 *              Optionally OR-ed with GGUFB200_DEQUANT_SRC_STABLE: the caller promises that no kernel still in flight on
 *              `stream` writes the packed bytes (model weights: written once at load time).  The kernel is launched with
 *              programmatic stream serialization; with the promise it fetches packed tiles and unpacks the first of them
 *              into shared memory while the preceding kernel drains, and only its stores wait for that kernel (whatever
 *              the preceding kernels read or wrote in `out` is complete before the first byte lands).  Same results.
 */
#define GGUFB200_DEQUANT_SRC_STABLE 0x100
int ggufb200_dequant(int ggml_type, const void *packed, int64_t n_blocks, void *out, int out_dtype,
                     int math_dtype, void *stream);

/*
 * Integer unpack only (test/debug surface for the "bit-exact integer unpack" contract):
 * per element the integer quant value q as it enters the float multiply, the integer
 * sub-block scale sc (1 if the type has none) and min mn (0 if none).  Any of the three
 * int16 output arrays (n_blocks*block_size each) may be NULL.
 */
int ggufb200_unpack_int(int ggml_type, const void *packed, int64_t n_blocks, int16_t *q, int16_t *sc,
                        int16_t *mn, void *stream);

/*
 * Row gather + dequant: out[i, :] = dequant(W[rows[i], :]).  Replaces the
 * "dequantise the whole table, then F.embedding" of ops.py:251-259 for quantised
 * Embedding weights.  rows: n_rows int64 indices on the device; K = logical row length.
 */
int ggufb200_dequant_rows(int ggml_type, const void *packed, int64_t n_table_rows, int64_t K,
                          const int64_t *rows, int64_t n_rows, void *out, int out_dtype, int math_dtype,
                          void *stream);

/*
 * Fused Linear: Y[M,N] = X[M,K] * dequant(W)[N,K]^T (+ bias[N]).  Replaces
 * ops.py:242-244 `forward_ggml_cast_weights` = cast_bias_weight (ops.py:193-211)
 * -> get_weight/dequantize_tensor (ops.py:166-191) -> F.linear.
 *   W_packed    N rows of K/block_size*type_size bytes (loader.py:118-120 layout)
 *   X, Y        act_dtype (0 fp16 / 1 bf16), row strides ldx / ldy in ELEMENTS, 16-byte aligned
 *   math_dtype  as in ggufb200_dequant().  Routes 1-3: W is first produced in math_dtype with the reference's rounding
 *               sequence and then cast to act_dtype, exactly the weight the reference hands to F.linear.  Route 4
 *               (GGUFB200_ALGO_FUSED_TMEM, fp16 math only) follows the contract under GGUFB200_FLAG_EXACT_W above.
 *               Accumulation is fp32 on every route.
 *   bias        NULL or N values of bias_dtype (0/1/2)
 *   workspace   scratch of at least ggufb200_linear_workspace() bytes (may be NULL if that is 0).  A W_packed that is
 *               not 16-byte aligned is always served by GGUFB200_ALGO_DEQUANT_MMA and needs that algo's workspace.
 *               GGUFB200_ALGO_FUSED_MMA with few output tiles (short M) cuts K into S ranges across SM pairs and keeps
 *               the fp32 partial results in the workspace (S*M*N*4 bytes, summed in a fixed order: reproducible);
 *               with less room it uses fewer ranges, with none it runs unsplit; GGUFB200_ALGO_FUSED_TMEM likewise.
 *               ggufb200_linear_workspace() assumes math_dtype == fp16 (the reference default);
 *               ggufb200_linear_workspace_ex() takes the math dtype of the call.
 *   algo        GGUFB200_ALGO_* | GGUFB200_FLAG_*
 */
size_t ggufb200_linear_workspace(int ggml_type, int64_t M, int64_t N, int64_t K, int act_dtype, int algo);

/* Same query with the math dtype of the call: GGUFB200_ALGO_AUTO routes a non-fp16 math dtype to
 * GGUFB200_ALGO_DEQUANT_MMA, and this variant reports that route's size (query and call always agree). */
size_t ggufb200_linear_workspace_ex(int ggml_type, int64_t M, int64_t N, int64_t K, int act_dtype, int math_dtype, int algo);

int ggufb200_linear(int ggml_type, const void *W_packed, int64_t N, int64_t K, const void *X, int64_t M,
                    int64_t ldx, int act_dtype, int math_dtype, const void *bias, int bias_dtype, void *Y,
                    int64_t ldy, void *workspace, size_t workspace_bytes, int algo, void *stream);

/*
 * Span-major shadow layout (SURVEY 8f rank 3, "one-time GPU repack").  The canonical GGUF rows (loader.py:96-120) can be
 * staged by the TMA engine only when a row's 256-wide K-span and the row stride are multiples of 16 bytes; Q2_K / Q3_K /
 * Q6_K / IQ4_XS blocks (84 / 110 / 210 / 136 bytes) and e.g. Q8_0 rows of 2432 elements (2584 bytes) are not.
 * ggufb200_repack() writes a copy out[span][row padded to 256][pitch] (pitch = span bytes padded to a multiple of 16, zero
 * filled) that GGUFB200_ALGO_FUSED_TMEM stages with one bulk copy per tile for EVERY block format and every K.  The
 * canonical bytes are not modified (GGMLTensor / state_dict semantics are the reference's); the copy is a cache owned by
 * the caller: ggufb200_repack_bytes() bytes, 16-byte aligned, valid as long as the caller keeps it.
 * ggufb200_linear_spans() = ggufb200_linear() with that copy at hand: AUTO then takes the TMEM-fed kernel for every format
 * (W_packed is still required: the reference-exact routes and EXACT_W read the canonical bytes).
 */
size_t ggufb200_repack_bytes(int ggml_type, int64_t N, int64_t K);
int ggufb200_repack(int ggml_type, const void *W_packed, int64_t N, int64_t K, void *out, void *stream);
int ggufb200_linear_spans(int ggml_type, const void *W_packed, const void *W_spans, int64_t N, int64_t K, const void *X,
                          int64_t M, int64_t ldx, int act_dtype, int math_dtype, const void *bias, int bias_dtype, void *Y,
                          int64_t ldy, void *workspace, size_t workspace_bytes, int algo, void *stream);

/*
 * Packed-weight Linear with a low-rank (LoRA) update folded into the SAME kernel (SURVEY 8f rank 1; replaces the
 * per-forward dequant + comfy.lora.calculate_weight + F.linear of ops.py:171-190 / nodes.py:43-47 for plain LoRA patches):
 *     Y = X * dequant(W)^T + T * U^T (+ bias),   T = X * down^T  [M, 64] act_dtype (row stride ldt, zero padded beyond the
 *     total rank R <= 64),   U = scale * up  [N, 64] fp16, contiguous, zero padded.
 * The update is one extra 64-wide k-block of GGUFB200_ALGO_FUSED_TMEM (U rows go to tensor memory like a dequantised
 * span, the T tile is TMA-fed like an activation tile): no second pass over Y, no extra GEMM launch for the up-projection.
 * algo must resolve to GGUFB200_ALGO_FUSED_TMEM (AUTO without EXACT_W on a weight that route supports, or explicit),
 * otherwise GGUFB200_E_UNSUPPORTED.  W_spans may be NULL.  fp16 dequant math.
 * (Round 2 fixed an intermittent hang of this entry point under many unsynchronised back-to-back calls: two producer groups
 * could become writers of one A stage after the LoRA k-block; profiles/r02_lora_in_kernel_hang_and_fix.log.)
 */
int ggufb200_linear_lora(int ggml_type, const void *W_packed, const void *W_spans, int64_t N, int64_t K, const void *X, int64_t M,
                         int64_t ldx, int act_dtype, const void *bias, int bias_dtype, const void *T, int64_t ldt, const void *U,
                         void *Y, int64_t ldy, void *workspace, size_t workspace_bytes, int algo, void *stream);

/*
 * Plain tensor-core GEMM on an already-dense weight: Y = X * W^T (+bias), W[N,K] in
 * act_dtype.  Used for the F16/BF16 (torch-compatible) Linears of a model and as the
 * second half of GGUFB200_ALGO_DEQUANT_MMA.
 */
int ggufb200_gemm(const void *W, int64_t N, int64_t K, int64_t ldw, const void *X, int64_t M, int64_t ldx,
                  int act_dtype, const void *bias, int bias_dtype, void *Y, int64_t ldy, void *stream);

/* Diagnostics: the tiling a fused kernel uses for this problem when given `workspace_bytes` of scratch.
 * algo = GGUFB200_ALGO_FUSED_MMA (| flags): activation rows per SM-pair tile (256 or 512), number of K ranges (1 = unsplit),
 *   64-wide k-blocks per range (the last range may be shorter, never empty), CTAs launched.
 * algo = GGUFB200_ALGO_FUSED_TMEM (| flags): tokens per item (32 / 128 / 192 / 384), number of K ranges, k-blocks per range,
 *   number of work items (persistent grid = min(items, SM pairs) clusters).
 * Pure host arithmetic, no GPU needed. */
int ggufb200_linear_plan(int ggml_type, int64_t M, int64_t N, int64_t K, size_t workspace_bytes, int algo, int *tile_rows, int *k_ranges,
                         int *kblocks_per_range, int *ctas);

/* Benchmark-only launch knobs (they never change routing or results):
 * key 1 = programmatic dependent launch of the standalone dequant kernel (default 1),
 * key 2 = CTAs per SM of the small-M integer-pattern kernel (0 = planner picks),
 * key 3 = L2 prefetch distance of the standalone dequant kernel in waves of resident CTAs, 0..8 (default 1, 0 = off).
 * Refused with GGUFB200_E_UNSUPPORTED unless the environment variable GGUFB200_ALLOW_TUNING=1 is set when the
 * library is first used; every other key is refused always (route selection is per call: GGUFB200_ALGO_* | GGUFB200_FLAG_*). */
int ggufb200_set_tuning(int key, int value);

#ifdef __cplusplus
}
#endif
#endif /* GGUFB200_H */
