/*
 * gguf_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * A plain-C CPU restatement of the GGUF block-dequantisation algorithm of
 * city96/ComfyUI-GGUF (reference `dequant.py`).  Only tests/, bench.py's
 * cpu_baseline / --impl reference leg and __graft_entry__.smoke() may load this
 * library, and only as the checker.  The product path (comfyui-gguf_b200/) never
 * links, imports or falls back to it.
 *
 * Parity pinning: the reference ships no golden vectors of its own (SURVEY.md
 * section 8c), so this restatement is pinned against outputs of the reference
 * itself: tests/golden/make_golden.py imports the reference's dequant.py
 * unmodified, runs it on seeded blocks and commits the results under
 * tests/golden/; tests/test_oracle.py requires bit-equality with those files and
 * with gguf-py's numpy `gguf.quants.dequantize` (the reference's fallback path,
 * dequant.py:24-28).
 *
 * What is restated (reference file:line):
 *   dequant.py:30-44    block addressing (n_blocks x type_size -> n_blocks x block_size)
 *   dequant.py:46-53    little-endian assembly of u16/u32 fields
 *   dequant.py:61-62    BF16
 *   dequant.py:65-123   Q8_0, Q5_1, Q5_0, Q4_1, Q4_0
 *   dequant.py:129-139  6-bit scale/min unpack shared by Q4_K/Q5_K
 *   dequant.py:141-238  Q6_K, Q5_K, Q4_K, Q3_K, Q2_K
 *   dequant.py:241-285  IQ4_NL / IQ4_XS and their 16-entry value table
 *   dequant.py:15-28    final `.to(dtype)` cast
 *
 * Numerics contract.  The reference runs every float op as a separate torch op
 * in a "math dtype" (fp16 by default, or the activation dtype / an explicit
 * dtype, dequant.py:22) so every intermediate is rounded to that dtype.  This
 * file reproduces exactly that: each product / sum is computed in binary32
 * (exact or correctly rounded) and then rounded to the math dtype; binary32 has
 * >= 2p+2 significand bits for p = 11 (fp16) and p = 8 (bf16), so the double
 * rounding is innocuous and equals what torch produces.  Build with
 * -ffp-contract=off so no FMA is ever formed.
 */
#include <stdint.h>
#include <string.h>
#include <stddef.h>

#ifdef _OPENMP
#include <omp.h>
#endif

enum {
    GG_Q4_0 = 2, GG_Q4_1 = 3, GG_Q5_0 = 6, GG_Q5_1 = 7, GG_Q8_0 = 8,
    GG_Q2_K = 10, GG_Q3_K = 11, GG_Q4_K = 12, GG_Q5_K = 13, GG_Q6_K = 14,
    GG_IQ4_NL = 20, GG_IQ4_XS = 23, GG_BF16 = 30
};
enum { DT_F16 = 0, DT_BF16 = 1, DT_F32 = 2 };

/* ---------------------------------------------------------------- soft floats */
static inline float bits2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t f2bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

static inline float h2f(uint16_t h)
{
    uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
    uint32_t exp = (h >> 10) & 0x1Fu;
    uint32_t man = h & 0x3FFu;
    if (exp == 0) {
        if (man == 0) return bits2f(sign);
        /* subnormal: value = man * 2^-24 */
        float v = (float)man * bits2f(0x33800000u); /* 2^-24 */
        return sign ? -v : v;
    }
    if (exp == 31) return bits2f(sign | 0x7F800000u | (man << 13));
    return bits2f(sign | ((exp + 112u) << 23) | (man << 13));
}

/* binary32 -> binary16, round to nearest even (what torch's .to(float16) does) */
static inline uint16_t f2h(float f)
{
    uint32_t x = f2bits(f);
    uint32_t sign = (x >> 16) & 0x8000u;
    uint32_t ax = x & 0x7FFFFFFFu;
    if (ax >= 0x7F800000u) {                       /* inf / nan */
        if (ax > 0x7F800000u) return (uint16_t)(sign | 0x7E00u | ((ax >> 13) & 0x3FFu));
        return (uint16_t)(sign | 0x7C00u);
    }
    if (ax >= 0x477FF000u) return (uint16_t)(sign | 0x7C00u);   /* >= 65520 -> inf */
    if (ax < 0x33000001u) return (uint16_t)sign;                /* <= 2^-25 -> 0 (tie to even) */
    int32_t e = (int32_t)(ax >> 23) - 127;
    uint32_t m = (ax & 0x7FFFFFu) | 0x800000u;
    uint32_t shift, half_bits;
    if (e < -14) {                                  /* subnormal result */
        shift = (uint32_t)(13 + (-14 - e));
        half_bits = 0;
    } else {
        shift = 13;
        half_bits = (uint32_t)(e + 15) << 10;
    }
    uint32_t q = m >> shift;
    uint32_t rem = m & ((1u << shift) - 1u);
    uint32_t halfway = 1u << (shift - 1);
    if (e >= -14) q &= 0x3FFu;                      /* drop the implicit bit for normals */
    uint32_t r = half_bits + q;
    if (rem > halfway || (rem == halfway && (r & 1u))) r += 1u;   /* carries into exponent correctly */
    return (uint16_t)(sign | r);
}

static inline float b2f(uint16_t b) { return bits2f((uint32_t)b << 16); }

/* binary32 -> bfloat16, round to nearest even */
static inline uint16_t f2b(float f)
{
    uint32_t x = f2bits(f);
    if ((x & 0x7FFFFFFFu) > 0x7F800000u) return (uint16_t)((x >> 16) | 0x40u);
    uint32_t lsb = (x >> 16) & 1u;
    x += 0x7FFFu + lsb;
    return (uint16_t)(x >> 16);
}

/* round a binary32 value to the math dtype and come back to binary32 */
static inline float rnd(int math, float v)
{
    if (math == DT_F16) return h2f(f2h(v));
    if (math == DT_BF16) return b2f(f2b(v));
    return v;
}

static inline void store_out(void *out, int64_t i, int out_dtype, float v)
{
    if (out_dtype == DT_F16) ((uint16_t *)out)[i] = f2h(v);
    else if (out_dtype == DT_BF16) ((uint16_t *)out)[i] = f2b(v);
    else ((float *)out)[i] = v;
}

/* ---------------------------------------------------------------- type table */
int ggor_type_info(int type, int *block_size, int *type_size)
{
    int bs, ts;
    switch (type) {
    case GG_Q4_0: bs = 32; ts = 18; break;
    case GG_Q4_1: bs = 32; ts = 20; break;
    case GG_Q5_0: bs = 32; ts = 22; break;
    case GG_Q5_1: bs = 32; ts = 24; break;
    case GG_Q8_0: bs = 32; ts = 34; break;
    case GG_Q2_K: bs = 256; ts = 84; break;
    case GG_Q3_K: bs = 256; ts = 110; break;
    case GG_Q4_K: bs = 256; ts = 144; break;
    case GG_Q5_K: bs = 256; ts = 176; break;
    case GG_Q6_K: bs = 256; ts = 210; break;
    case GG_IQ4_NL: bs = 32; ts = 18; break;
    case GG_IQ4_XS: bs = 256; ts = 136; break;
    case GG_BF16: bs = 1; ts = 2; break;
    default: return -1;
    }
    if (block_size) *block_size = bs;
    if (type_size) *type_size = ts;
    return 0;
}

static inline uint16_t rd16(const uint8_t *p) { return (uint16_t)(p[0] | (p[1] << 8)); }
static inline uint32_t rd32(const uint8_t *p)
{
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

/* dequant.py:241 */
static const int8_t IQ4_VALUES[16] = {-127, -104, -83, -65, -49, -35, -22, -10, 1, 13, 25, 38, 53, 69, 89, 113};

/* dequant.py:129-139: the 12 scale bytes hold eight 6-bit scales and eight 6-bit mins */
static inline void k_scale_min(const uint8_t *s, int j, int *sc, int *mn)
{
    if (j < 4) {
        *sc = s[j] & 63;
        *mn = s[j + 4] & 63;
    } else {
        *sc = (s[j + 4] & 0x0F) | ((s[j - 4] >> 6) << 4);
        *mn = (s[j + 4] >> 4) | ((s[j] >> 6) << 4);
    }
}

/*
 * Integer unpack of element e of one block: the integer quant value q exactly
 * as it enters the float multiply in the reference, the integer sub-block
 * scale sc (1 when the type has none) and integer sub-block min mn (0 when
 * none).  This is the "bit-exact integer unpack" contract.
 */
static inline void unpack_elem(int type, const uint8_t *B, int e, int *q, int *sc, int *mn)
{
    *sc = 1;
    *mn = 0;
    switch (type) {
    case GG_Q4_0: /* dequant.py:115-123 */
        *q = (int)((B[2 + (e & 15)] >> (4 * (e >> 4))) & 0x0F) - 8;
        break;
    case GG_Q4_1: /* dequant.py:103-113 */
        *q = (B[4 + (e & 15)] >> (4 * (e >> 4))) & 0x0F;
        break;
    case GG_Q5_0: { /* dequant.py:87-101 */
        uint32_t qh = rd32(B + 2);
        int lo = (B[6 + (e & 15)] >> (4 * (e >> 4))) & 0x0F;
        *q = (lo | (int)(((qh >> e) & 1u) << 4)) - 16;
        break;
    }
    case GG_Q5_1: { /* dequant.py:71-85 */
        uint32_t qh = rd32(B + 4);
        int lo = (B[8 + (e & 15)] >> (4 * (e >> 4))) & 0x0F;
        *q = lo | (int)(((qh >> e) & 1u) << 4);
        break;
    }
    case GG_Q8_0: /* dequant.py:65-69 */
        *q = (int8_t)B[2 + e];
        break;
    case GG_Q2_K: { /* dequant.py:221-238 */
        int sb = e >> 4;
        *q = (B[16 + 32 * (e >> 7) + (e & 31)] >> (2 * ((e >> 5) & 3))) & 3;
        *sc = B[sb] & 0x0F;
        *mn = B[sb] >> 4;
        break;
    }
    case GG_Q3_K: { /* dequant.py:197-219 */
        int i = e >> 4;
        int lo = (B[32 + 32 * (e >> 7) + (e & 31)] >> (2 * ((e >> 5) & 3))) & 3;
        int hb = (B[e & 31] >> (e >> 5)) & 1;
        int ls = (B[96 + (i & 7)] >> (4 * (i >> 3))) & 0x0F;
        int hs = (B[104 + (i & 3)] >> (2 * (i >> 2))) & 3;
        *q = lo - ((hb ^ 1) << 2);
        *sc = (int)(int8_t)(ls | (hs << 4)) - 32;
        break;
    }
    case GG_Q4_K: { /* dequant.py:180-195 */
        int sb = e >> 5;
        *q = (B[16 + 32 * (e >> 6) + (e & 31)] >> (4 * (sb & 1))) & 0x0F;
        k_scale_min(B + 4, sb, sc, mn);
        break;
    }
    case GG_Q5_K: { /* dequant.py:159-178 */
        int sb = e >> 5;
        int lo = (B[48 + 32 * (e >> 6) + (e & 31)] >> (4 * (sb & 1))) & 0x0F;
        int hi = (B[16 + (e & 31)] >> sb) & 1;
        *q = lo | (hi << 4);
        k_scale_min(B + 4, sb, sc, mn);
        break;
    }
    case GG_Q6_K: { /* dequant.py:141-157 */
        int h = e >> 7, r = e & 127;
        int lo = (B[64 * h + (r & 63)] >> (4 * (r >> 6))) & 0x0F;
        int hi = (B[128 + 32 * h + (r & 31)] >> (2 * (r >> 5))) & 3;
        *q = (int)(int8_t)(lo | (hi << 4)) - 32;
        *sc = (int8_t)B[192 + (e >> 4)];
        break;
    }
    case GG_IQ4_NL: /* dequant.py:243-256 */
        *q = IQ4_VALUES[(B[2 + (e & 15)] >> (4 * (e >> 4))) & 0x0F];
        break;
    case GG_IQ4_XS: { /* dequant.py:258-285 */
        int i = e >> 5;
        uint32_t sh = rd16(B + 2);
        int ls = (B[4 + (i >> 1)] >> (4 * (i & 1))) & 0x0F;
        int hs = (int)((sh >> (2 * i)) & 3u);
        *q = IQ4_VALUES[(B[8 + 16 * i + (e & 15)] >> (4 * ((e >> 4) & 1))) & 0x0F];
        *sc = (int)(int8_t)(ls | (hs << 4)) - 32;
        break;
    }
    default:
        *q = 0;
        break;
    }
}

/* the two fp16 header fields of a block: d (scale) and the second one (m / dmin), 0 if absent */
static inline void block_header(int type, const uint8_t *B, uint16_t *d, uint16_t *d2)
{
    *d2 = 0;
    switch (type) {
    case GG_Q4_0: case GG_Q5_0: case GG_Q8_0: case GG_IQ4_NL: case GG_IQ4_XS:
        *d = rd16(B); break;
    case GG_Q4_1: case GG_Q5_1: case GG_Q4_K: case GG_Q5_K:
        *d = rd16(B); *d2 = rd16(B + 2); break;
    case GG_Q2_K: *d = rd16(B + 80); *d2 = rd16(B + 82); break;
    case GG_Q3_K: *d = rd16(B + 108); break;
    case GG_Q6_K: *d = rd16(B + 208); break;
    default: *d = 0; break;
    }
}

/*
 * Float step of one element, op order exactly as the reference's torch chain:
 *   legacy       d*q                      (dequant.py:69,101,123,256)
 *   legacy+m     (d*q) + m                (dequant.py:85,113)
 *   K scale      (d*sc)*q                 (dequant.py:147-157, 212-219, 278-285)
 *   K scale+min  (d*sc)*q - (dmin*mn)     (dequant.py:170-178, 189-195, 229-236)
 */
static inline float float_step(int type, int math, float d, float d2, int q, int sc, int mn)
{
    switch (type) {
    case GG_Q4_0: case GG_Q5_0: case GG_Q8_0: case GG_IQ4_NL:
        return rnd(math, d * (float)q);
    case GG_Q4_1: case GG_Q5_1:
        return rnd(math, rnd(math, d * (float)q) + d2);
    case GG_Q3_K: case GG_Q6_K: case GG_IQ4_XS: {
        float dl = rnd(math, d * (float)sc);
        return rnd(math, dl * (float)q);
    }
    case GG_Q2_K: case GG_Q4_K: case GG_Q5_K: {
        float dl = rnd(math, d * (float)sc);
        float ml = rnd(math, d2 * (float)mn);
        return rnd(math, rnd(math, dl * (float)q) - ml);
    }
    default:
        return 0.0f;
    }
}

/*
 * dequant.py:15-44 for one packed tensor: n_blocks blocks -> n_blocks*block_size
 * values.  math_dtype = dtype the float ops run in (DT_F16 is the reference
 * default), out_dtype = dtype of the final `.to(dtype)`.
 * Returns 0, or -1 for an unknown type.
 */
int ggor_dequant(int type, const uint8_t *packed, int64_t n_blocks, void *out, int out_dtype, int math_dtype)
{
    int bs, ts;
    if (ggor_type_info(type, &bs, &ts) != 0) return -1;
    if (out_dtype < 0 || out_dtype > 2 || math_dtype < 0 || math_dtype > 2) return -2;

    if (type == GG_BF16) { /* dequant.py:61-62: always widened to fp32 first, then cast */
        int64_t i;
#pragma omp parallel for schedule(static)
        for (i = 0; i < n_blocks; ++i) store_out(out, i, out_dtype, b2f(rd16(packed + 2 * i)));
        return 0;
    }

    int64_t b;
#pragma omp parallel for schedule(static)
    for (b = 0; b < n_blocks; ++b) {
        const uint8_t *B = packed + b * (int64_t)ts;
        uint16_t dh, d2h;
        block_header(type, B, &dh, &d2h);
        /* `d.view(float16).to(dtype)`: the header is first cast to the math dtype */
        float d = rnd(math_dtype, h2f(dh));
        float d2 = rnd(math_dtype, h2f(d2h));
        /* the sub-block scale / min are constant over aligned runs of 16 elements for every format: the two
         * products d*sc and dmin*mn (each rounded once, as in the reference) are computed once per run */
        for (int e0 = 0; e0 < bs; e0 += 16) {
            int q, sc, mn;
            unpack_elem(type, B, e0, &q, &sc, &mn);
            const float dl = rnd(math_dtype, d * (float)sc);
            const float ml = rnd(math_dtype, d2 * (float)mn);
            for (int e = e0; e < e0 + 16 && e < bs; ++e) {
                int s2, m2;
                unpack_elem(type, B, e, &q, &s2, &m2);
                float v;
                switch (type) {
                case GG_Q4_0: case GG_Q5_0: case GG_Q8_0: case GG_IQ4_NL:
                    v = rnd(math_dtype, d * (float)q); break;
                case GG_Q4_1: case GG_Q5_1:
                    v = rnd(math_dtype, rnd(math_dtype, d * (float)q) + d2); break;
                case GG_Q3_K: case GG_Q6_K: case GG_IQ4_XS:
                    v = rnd(math_dtype, dl * (float)q); break;
                default: /* Q2_K, Q4_K, Q5_K */
                    v = rnd(math_dtype, rnd(math_dtype, dl * (float)q) - ml); break;
                }
                store_out(out, b * (int64_t)bs + e, out_dtype, v);
            }
        }
    }
    return 0;
}

/* integer unpack only: q / sc / mn per element as int16 (each array n_blocks*block_size) */
int ggor_unpack_int(int type, const uint8_t *packed, int64_t n_blocks, int16_t *q_out, int16_t *sc_out, int16_t *mn_out)
{
    int bs, ts;
    if (ggor_type_info(type, &bs, &ts) != 0 || type == GG_BF16) return -1;
    int64_t b;
#pragma omp parallel for schedule(static)
    for (b = 0; b < n_blocks; ++b) {
        const uint8_t *B = packed + b * (int64_t)ts;
        for (int e = 0; e < bs; ++e) {
            int q, sc, mn;
            unpack_elem(type, B, e, &q, &sc, &mn);
            int64_t i = b * (int64_t)bs + e;
            if (q_out) q_out[i] = (int16_t)q;
            if (sc_out) sc_out[i] = (int16_t)sc;
            if (mn_out) mn_out[i] = (int16_t)mn;
        }
    }
    return 0;
}

/*
 * ops.py:242-244 restated for the Linear that consumes the weight:
 *   W = dequant(packed) in math dtype -> cast to act dtype (dequant.py:23)
 *   y[m,n] = act( sum_k x[m,k] * W[n,k]  (+ bias[n]) )
 * x / bias / y are in act_dtype (bias may be NULL).  Accumulation is binary32 in
 * k order -- a GEMM library accumulates in a different order, which is why the
 * Linear contract is a relative tolerance (1e-3) and not bit equality.
 */
int ggor_linear(int type, const uint8_t *packed, int64_t N, int64_t K, const void *X, int64_t M,
                int act_dtype, int math_dtype, const void *bias, void *Y)
{
    int bs, ts;
    if (ggor_type_info(type, &bs, &ts) != 0) return -1;
    if (K % bs != 0) return -3;
    int64_t row_bytes = K / bs * ts;
    int64_t n;
    int rc = 0;
#pragma omp parallel
    {
        float *w = (float *)__builtin_malloc((size_t)K * sizeof(float));
        uint16_t *wq = (uint16_t *)__builtin_malloc((size_t)K * sizeof(float));
#pragma omp for schedule(static)
        for (n = 0; n < N; ++n) {
            /* dequantise row n into act dtype, then widen to fp32 for the dot product */
            if (act_dtype == DT_F32) {
                ggor_dequant(type, packed + n * row_bytes, K / bs, w, DT_F32, math_dtype);
            } else {
                ggor_dequant(type, packed + n * row_bytes, K / bs, wq, act_dtype, math_dtype);
                for (int64_t k = 0; k < K; ++k) w[k] = act_dtype == DT_F16 ? h2f(wq[k]) : b2f(wq[k]);
            }
            for (int64_t m = 0; m < M; ++m) {
                float acc = 0.0f;
                for (int64_t k = 0; k < K; ++k) {
                    float xv;
                    if (act_dtype == DT_F32) xv = ((const float *)X)[m * K + k];
                    else if (act_dtype == DT_F16) xv = h2f(((const uint16_t *)X)[m * K + k]);
                    else xv = b2f(((const uint16_t *)X)[m * K + k]);
                    acc += xv * w[k];
                }
                if (bias) {
                    float bv;
                    if (act_dtype == DT_F32) bv = ((const float *)bias)[n];
                    else if (act_dtype == DT_F16) bv = h2f(((const uint16_t *)bias)[n]);
                    else bv = b2f(((const uint16_t *)bias)[n]);
                    acc += bv;
                }
                store_out(Y, m * N + n, act_dtype, acc);
            }
        }
        __builtin_free(w);
        __builtin_free(wq);
    }
    return rc;
}

int ggor_num_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

void ggor_set_num_threads(int n)
{
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
#else
    (void)n;
#endif
}
