// blocks.cuh -- per-format unpack of GGUF quantised blocks (device side).
//
// One struct per ggml type (the keys of the reference's dispatch table, dequant.py:287-301).
// Every struct exposes the same interface so the standalone dequant kernel, the row-gather
// kernel, the fused GEMV and the fused tcgen05 GEMM all share one unpack implementation:
//
//   BS, TS      block size (elements) and type size (bytes)          gguf-py GGML_QUANT_SIZES
//   BIAS        q4() returns u = q + BIAS as unsigned bytes (q = integer entering the multiply)
//   KIND        float step:  0  d*q            1  d*q + m
//                            2  (d*sc)*q       3  (d*sc)*q - (dmin*mn)
//   q4(blk,e0)  four consecutive elements e0..e0+3 (e0 % 4 == 0) as four biased bytes
//   scales()    integer sub-block scale / min of the group containing e0 (constant over
//               any aligned run of 8 elements for every format)
//   d_bits / d2_bits   raw fp16 header fields
//
// `blk` points at the first byte of the block; A_BLK = its compile-time known alignment
// (gcd(TS,16) when the tile base is 16-byte aligned).  Everything here is integer work and
// is bit-exact against oracle/gguf_oracle.c::unpack_elem and the reference.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace ggufb200 {

enum : int {
    T_Q4_0 = 2, T_Q4_1 = 3, T_Q5_0 = 6, T_Q5_1 = 7, T_Q8_0 = 8, T_Q2_K = 10, T_Q3_K = 11, T_Q4_K = 12,
    T_Q5_K = 13, T_Q6_K = 14, T_IQ4_NL = 20, T_IQ4_XS = 23, T_BF16 = 30
};

// spread the low four bits of t over the low bit of four bytes (bit i -> byte i)
GG_HD uint32_t spread4(uint32_t t) { return ((t & 0xFu) * 0x00204081u) & 0x01010101u; }

// dequant.py:241 value table, stored biased by +127 so it fits unsigned bytes
GG_HD uint32_t iq4_lookup4(uint32_t idx4)
{
    // entries 0..15 of (KVALUES + 127):  0 23 44 62 | 78 92 105 117 | 128 140 152 165 | 180 196 216 240
    const uint32_t t0 = 0x3E2C1700u, t1 = 0x75695C4Eu, t2 = 0xA5988C80u, t3 = 0xF0D8C4B4u;
    // prmt can index 8 bytes; pick from the low or the high half of the table by bit 3 of each index
    uint32_t sel = (idx4 & 0x07070707u);
    sel = (sel | (sel >> 4)) & 0x00FF00FFu;          // pack nibbles: byte0|byte1 -> low byte, byte2|byte3 -> byte 2
    sel = (sel | (sel >> 8)) & 0x0000FFFFu;          // four selector nibbles in the low 16 bits
    uint32_t lo = prmt(t0, t1, sel);
    uint32_t hi = prmt(t2, t3, sel);
    uint32_t m = ((idx4 >> 3) & 0x01010101u) * 0xFFu;  // 0xFF per byte whose index >= 8
    return (lo & ~m) | (hi & m);
}

template <int QT> struct Block;

// ---------------------------------------------------------------- legacy 32-element blocks
template <> struct Block<T_Q4_0> {  // dequant.py:115-123   [d f16][qs 16]
    static constexpr int BS = 32, TS = 18, BIAS = 8, KIND = 0, A_BLK = 2;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<2>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *) { return 0; }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        return (ld32<2>(b + 2 + (e0 & 15)) >> (4 * (e0 >> 4))) & 0x0F0F0F0Fu;
    }
    static GG_HD void scales(const uint8_t *, int, int &sc, int &mn) { sc = 1; mn = 0; }
};
template <> struct Block<T_Q4_1> {  // dequant.py:103-113   [d][m][qs 16]
    static constexpr int BS = 32, TS = 20, BIAS = 0, KIND = 1, A_BLK = 4;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<4>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *b) { return ld16<2>(b + 2); }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        return (ld32<4>(b + 4 + (e0 & 15)) >> (4 * (e0 >> 4))) & 0x0F0F0F0Fu;
    }
    static GG_HD void scales(const uint8_t *, int, int &sc, int &mn) { sc = 1; mn = 0; }
};
template <> struct Block<T_Q5_0> {  // dequant.py:87-101   [d][qh u32][qs 16]
    static constexpr int BS = 32, TS = 22, BIAS = 16, KIND = 0, A_BLK = 2;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<2>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *) { return 0; }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        uint32_t qh = ld32<2>(b + 2);
        uint32_t lo = (ld32<2>(b + 6 + (e0 & 15)) >> (4 * (e0 >> 4))) & 0x0F0F0F0Fu;
        return lo | (spread4(qh >> e0) << 4);
    }
    static GG_HD void scales(const uint8_t *, int, int &sc, int &mn) { sc = 1; mn = 0; }
};
template <> struct Block<T_Q5_1> {  // dequant.py:71-85   [d][m][qh u32][qs 16]
    static constexpr int BS = 32, TS = 24, BIAS = 0, KIND = 1, A_BLK = 8;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<8>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *b) { return ld16<2>(b + 2); }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        uint32_t qh = ld32<4>(b + 4);
        uint32_t lo = (ld32<4>(b + 8 + (e0 & 15)) >> (4 * (e0 >> 4))) & 0x0F0F0F0Fu;
        return lo | (spread4(qh >> e0) << 4);
    }
    static GG_HD void scales(const uint8_t *, int, int &sc, int &mn) { sc = 1; mn = 0; }
};
template <> struct Block<T_Q8_0> {  // dequant.py:65-69   [d][int8 x 32]
    static constexpr int BS = 32, TS = 34, BIAS = 128, KIND = 0, A_BLK = 2;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<2>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *) { return 0; }
    static GG_HD uint32_t q4(const uint8_t *b, int e0) { return ld32<2>(b + 2 + e0) ^ 0x80808080u; }
    static GG_HD void scales(const uint8_t *, int, int &sc, int &mn) { sc = 1; mn = 0; }
};
template <> struct Block<T_IQ4_NL> {  // dequant.py:243-256   layout of Q4_0, values through the table
    static constexpr int BS = 32, TS = 18, BIAS = 127, KIND = 0, A_BLK = 2;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<2>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *) { return 0; }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        return iq4_lookup4((ld32<2>(b + 2 + (e0 & 15)) >> (4 * (e0 >> 4))) & 0x0F0F0F0Fu);
    }
    static GG_HD void scales(const uint8_t *, int, int &sc, int &mn) { sc = 1; mn = 0; }
};

// ---------------------------------------------------------------- K-quants, 256-element super-blocks
// dequant.py:129-139: eight 6-bit (scale, min) pairs in 12 bytes s[0..11]
// branch-free: the three little-endian words w0 = s[0..3], w1 = s[4..7], w2 = s[8..11]
GG_HD void k_scale_min(const uint8_t *s, int j, int &sc, int &mn)
{
    const uint32_t *w = reinterpret_cast<const uint32_t *>(s);   // blk + 4 is 4-byte aligned for Q4_K / Q5_K
    const int sh = 8 * (j & 3);
    const uint32_t a = (w[0] >> sh) & 0xFFu, b = (w[1] >> sh) & 0xFFu, c = (w[2] >> sh) & 0xFFu;
    const bool hi = j >= 4;
    sc = hi ? (int)((c & 0x0Fu) | ((a >> 6) << 4)) : (int)(a & 63u);
    mn = hi ? (int)((c >> 4) | ((b >> 6) << 4)) : (int)(b & 63u);
}

template <> struct Block<T_Q2_K> {  // dequant.py:221-238   [scales 16][qs 64][d][dmin]
    static constexpr int BS = 256, TS = 84, BIAS = 0, KIND = 3, A_BLK = 4;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<4>(b + 80); }
    static GG_HD uint32_t d2_bits(const uint8_t *b) { return ld16<2>(b + 82); }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        return (ld32<4>(b + 16 + 32 * (e0 >> 7) + (e0 & 31)) >> (2 * ((e0 >> 5) & 3))) & 0x03030303u;
    }
    static GG_HD void scales(const uint8_t *b, int e0, int &sc, int &mn)
    {
        uint32_t s = b[e0 >> 4];
        sc = s & 0x0F;
        mn = s >> 4;
    }
};
template <> struct Block<T_Q3_K> {  // dequant.py:197-219   [hmask 32][qs 64][scales 12][d]
    static constexpr int BS = 256, TS = 110, BIAS = 4, KIND = 2, A_BLK = 2;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<2>(b + 108); }
    static GG_HD uint32_t d2_bits(const uint8_t *) { return 0; }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        uint32_t lo = (ld32<2>(b + 32 + 32 * (e0 >> 7) + (e0 & 31)) >> (2 * ((e0 >> 5) & 3))) & 0x03030303u;
        uint32_t hb = (ld32<2>(b + (e0 & 31)) >> (e0 >> 5)) & 0x01010101u;
        return lo + (hb << 2);  // q = lo - 4*(hb^1) = lo + 4*hb - 4
    }
    static GG_HD void scales(const uint8_t *b, int e0, int &sc, int &mn)
    {
        int i = e0 >> 4;
        uint32_t ls = (b[96 + (i & 7)] >> (4 * (i >> 3))) & 0x0F;
        uint32_t hs = (b[104 + (i & 3)] >> (2 * (i >> 2))) & 3;
        sc = (int)(ls | (hs << 4)) - 32;
        mn = 0;
    }
};
template <> struct Block<T_Q4_K> {  // dequant.py:180-195   [d][dmin][scales 12][qs 128]
    static constexpr int BS = 256, TS = 144, BIAS = 0, KIND = 3, A_BLK = 16;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<16>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *b) { return ld16<2>(b + 2); }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        return (ld32<4>(b + 16 + 32 * (e0 >> 6) + (e0 & 31)) >> (4 * ((e0 >> 5) & 1))) & 0x0F0F0F0Fu;
    }
    static GG_HD void scales(const uint8_t *b, int e0, int &sc, int &mn)
    {
        k_scale_min(b + 4, e0 >> 5, sc, mn);
    }
};
template <> struct Block<T_Q5_K> {  // dequant.py:159-178   [d][dmin][scales 12][qh 32][qs 128]
    static constexpr int BS = 256, TS = 176, BIAS = 0, KIND = 3, A_BLK = 16;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<16>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *b) { return ld16<2>(b + 2); }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        int sb = e0 >> 5;
        uint32_t lo = (ld32<4>(b + 48 + 32 * (e0 >> 6) + (e0 & 31)) >> (4 * (sb & 1))) & 0x0F0F0F0Fu;
        uint32_t hi = (ld32<4>(b + 16 + (e0 & 31)) >> sb) & 0x01010101u;
        return lo | (hi << 4);
    }
    static GG_HD void scales(const uint8_t *b, int e0, int &sc, int &mn)
    {
        k_scale_min(b + 4, e0 >> 5, sc, mn);
    }
};
template <> struct Block<T_Q6_K> {  // dequant.py:141-157   [ql 128][qh 64][scales i8 16][d]
    static constexpr int BS = 256, TS = 210, BIAS = 32, KIND = 2, A_BLK = 2;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<2>(b + 208); }
    static GG_HD uint32_t d2_bits(const uint8_t *) { return 0; }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        int h = e0 >> 7, r = e0 & 127;
        uint32_t lo = (ld32<2>(b + 64 * h + (r & 63)) >> (4 * (r >> 6))) & 0x0F0F0F0Fu;
        uint32_t hi = (ld32<2>(b + 128 + 32 * h + (r & 31)) >> (2 * (r >> 5))) & 0x03030303u;
        return lo | (hi << 4);
    }
    static GG_HD void scales(const uint8_t *b, int e0, int &sc, int &mn)
    {
        sc = (int)(int8_t)b[192 + (e0 >> 4)];
        mn = 0;
    }
};
template <> struct Block<T_IQ4_XS> {  // dequant.py:258-285   [d][scales_h u16][scales_l 4][qs 128]
    static constexpr int BS = 256, TS = 136, BIAS = 127, KIND = 2, A_BLK = 8;
    static GG_HD uint32_t d_bits(const uint8_t *b) { return ld16<8>(b); }
    static GG_HD uint32_t d2_bits(const uint8_t *) { return 0; }
    static GG_HD uint32_t q4(const uint8_t *b, int e0)
    {
        int i = e0 >> 5;
        uint32_t idx = (ld32<4>(b + 8 + 16 * i + (e0 & 15)) >> (4 * ((e0 >> 4) & 1))) & 0x0F0F0F0Fu;
        return iq4_lookup4(idx);
    }
    static GG_HD void scales(const uint8_t *b, int e0, int &sc, int &mn)
    {
        int i = e0 >> 5;
        uint32_t sh = ld16<2>(b + 2);
        uint32_t ls = (b[4 + (i >> 1)] >> (4 * (i & 1))) & 0x0F;
        uint32_t hs = (sh >> (2 * i)) & 3;
        sc = (int)(ls | (hs << 4)) - 32;
        mn = 0;
    }
};

// ---------------------------------------------------------------- host dispatch over the formats and dtypes
// The only place that maps a ggml type code to its Block<T>: returns f(Block<T>{}) for the 12 block formats and `other`
// for anything else (BF16, unknown codes).  A switch of direct calls, resolved at compile time: it sits on the host path of
// every Linear call, whose cost matters at short activations.
template <class R, class F> R with_block(int type, R other, F &&f)
{
    switch (type) {
    case T_Q4_0: return f(Block<T_Q4_0>{});
    case T_Q4_1: return f(Block<T_Q4_1>{});
    case T_Q5_0: return f(Block<T_Q5_0>{});
    case T_Q5_1: return f(Block<T_Q5_1>{});
    case T_Q8_0: return f(Block<T_Q8_0>{});
    case T_Q2_K: return f(Block<T_Q2_K>{});
    case T_Q3_K: return f(Block<T_Q3_K>{});
    case T_Q4_K: return f(Block<T_Q4_K>{});
    case T_Q5_K: return f(Block<T_Q5_K>{});
    case T_Q6_K: return f(Block<T_Q6_K>{});
    case T_IQ4_NL: return f(Block<T_IQ4_NL>{});
    case T_IQ4_XS: return f(Block<T_IQ4_XS>{});
    }
    return other;
}

template <int D> using DType = std::integral_constant<int, D>;

// f(DType<d>{}) for a dtype code d in {kF16, kBF16, kF32}, GGUFB200_E_DTYPE for anything else
template <class F> int with_dtype(int dtype, F &&f)
{
    switch (dtype) {
    case kF16: return f(DType<kF16>{});
    case kBF16: return f(DType<kBF16>{});
    case kF32: return f(DType<kF32>{});
    }
    return GGUFB200_E_DTYPE;
}

// f(DType<act>{}) for an activation dtype: bf16, otherwise fp16 (callers have validated `act`)
template <class F> int with_act(int act, F &&f)
{
    return act == kBF16 ? f(DType<kBF16>{}) : f(DType<kF16>{});
}

// K elements of one span, the unit in which the fused kernels stage packed weight rows
constexpr int kSpanK = 256;

template <class Q> struct SpanOf {
    static constexpr int BYTES = (kSpanK / Q::BS) * Q::TS;      // packed bytes of one row's span
    // Row pitch of a staged span in shared memory (and of the re-packed span-major layout, repack.cu).  A span whose byte
    // count is a multiple of 16 keeps it (the canonical rows can then be staged by a 2-D tensor map, which writes rows
    // densely); the others are padded to the next ODD multiple of 16: 16-byte aligned rows whose 16-byte reads at
    // lane = row are bank-conflict free (Q2_K 84 -> 112, Q3_K 110 -> 112, IQ4_XS 136 -> 144, Q6_K 210 -> 240).
    static constexpr int PAD16 = (BYTES + 15) / 16 * 16;
    static constexpr int PITCH = BYTES % 16 == 0 ? BYTES : ((PAD16 / 16) % 2 == 1 ? PAD16 : PAD16 + 16);
};

// ---------------------------------------------------------------- float step shared by every consumer
// The multiplier / offset pair (a, b) of the float step is constant over a GROUP of consecutive elements:
//   KIND 0: a = d              KIND 1: a = d, b = m          (GROUP = the 32-element block)
//   KIND 2: a = d*sc           KIND 3: a = d*sc, b = dmin*mn (GROUP = 32 for Q4_K/Q5_K/IQ4_XS, 16 for Q2_K/Q3_K/Q6_K)
// Consumers that walk a whole group (standalone dequant, fused GEMM) compute it once per group.
template <class Q> struct GroupOf {
    static constexpr int value = (Q::BS == 32) ? 32 : ((Q::TS == 144 || Q::TS == 176 || Q::TS == 136) ? 32 : 16);
};

template <int MATH> struct GroupScale {
    typename Math<MATH>::T2 a, b;
};

template <class Q, int MATH> GG_HD GroupScale<MATH> group_scale(const uint8_t *blk, int e0)
{
    using M = Math<MATH>;
    GroupScale<MATH> g;
    typename M::T d = M::from_h(Q::d_bits(blk));
    if constexpr (Q::KIND == 0) {
        g.a = M::bcast(d);
        g.b = g.a;
    } else if constexpr (Q::KIND == 1) {
        g.a = M::bcast(d);
        g.b = M::bcast(M::from_h(Q::d2_bits(blk)));
    } else {
        int sc, mn;
        Q::scales(blk, e0, sc, mn);
        g.a = M::bcast(M::mul(d, M::from_int(sc)));
        if constexpr (Q::KIND == 3) g.b = M::bcast(M::mul(M::from_h(Q::d2_bits(blk)), M::from_int(mn)));
        else g.b = g.a;
    }
    return g;
}

// N consecutive elements (N = 4 or 8, e0 % N == 0, all inside one group) -> N/2 pairs in the math dtype,
// op order and per-op rounding exactly as the reference (see oracle/gguf_oracle.c::float_step).
template <class Q, int MATH, int N>
GG_HD void dequant_elems(const uint8_t *blk, int e0, const GroupScale<MATH> &g, typename Math<MATH>::T2 (&out)[N / 2])
{
    using M = Math<MATH>;
    static_assert(N == 4 || N == 8, "run length");
#pragma unroll
    for (int j = 0; j < N / 4; ++j) {
        typename M::T2 lo, hi;
        M::cvt4(Q::q4(blk, e0 + 4 * j), Q::BIAS, lo, hi);
        lo = M::mul2(g.a, lo);
        hi = M::mul2(g.a, hi);
        if constexpr (Q::KIND == 1) {
            lo = M::add2(lo, g.b);
            hi = M::add2(hi, g.b);
        } else if constexpr (Q::KIND == 3) {
            lo = M::sub2(lo, g.b);
            hi = M::sub2(hi, g.b);
        }
        out[2 * j] = lo;
        out[2 * j + 1] = hi;
    }
}

// ---------------------------------------------------------------- specialised 16-element producers (fused GEMM hot formats)
// Sixteen consecutive elements (e0 % 16 == 0) of one block as eight packed activation-dtype pairs, fp16 reference math.
// Same operations and roundings as group_scale + dequant_elems, but with the whole header fetched by one 16-byte load, the
// quants by one 16-byte load and (d,dmin) x (sc,mn) as a single half2 multiply.  `blk` must be 16-byte aligned.
template <class Q, int ACT> struct Fast16 {
    static constexpr bool available = false;
};

template <int ACT> GG_HD uint32_t pack_h2_to_act(__half2 v)
{
    if constexpr (ACT == kF16) {
        return *reinterpret_cast<uint32_t *>(&v);
    } else {
        float2 f = __half22float2(v);
        __nv_bfloat162 b = __floats2bfloat162_rn(f.x, f.y);
        return *reinterpret_cast<uint32_t *>(&b);
    }
}

template <int ACT> struct Fast16<Block<T_Q4_K>, ACT> {
    static constexpr bool available = true;
    static GG_HD void run(const uint8_t *blk, int e0, uint32_t (&out)[8])
    {
        const uint4 h = *reinterpret_cast<const uint4 *>(blk);                 // d | dmin<<16, scales[0..11]
        const int sb = e0 >> 5;                                               // sub-block 0..7
        const uint4 qw = *reinterpret_cast<const uint4 *>(blk + 16 + 32 * (e0 >> 6) + (e0 & 16));
        // 6-bit scale / min of the sub-block (dequant.py:129-139), branch-free on the three scale words
        const int sh = 8 * (sb & 3);
        const uint32_t a = (h.y >> sh) & 0xFFu, b = (h.z >> sh) & 0xFFu, c = (h.w >> sh) & 0xFFu;
        const bool hi4 = sb >= 4;
        const uint32_t sc = hi4 ? ((c & 0x0Fu) | ((a >> 6) << 4)) : (a & 63u);
        const uint32_t mn = hi4 ? ((c >> 4) | ((b >> 6) << 4)) : (b & 63u);
        // (sc, mn) -> exact fp16 pair through the 1024+u exponent pattern, then (d*sc, dmin*mn) in ONE rounded half2 multiply
        uint32_t scm_bits = sc | (mn << 16) | 0x64006400u;
        const __half2 k1024 = __half2half2(__ushort_as_half((unsigned short)0x6400u));
        const __half2 scm = __hsub2_rn(*reinterpret_cast<__half2 *>(&scm_bits), k1024);
        uint32_t dm_bits = h.x;
        const __half2 DM = __hmul2_rn(*reinterpret_cast<__half2 *>(&dm_bits), scm);
        const __half2 D2 = __low2half2(DM), M2 = __high2half2(DM);
        // odd sub-blocks live in the high nibbles.  Instead of shifting them down, keep q << 4 in place and build the fp16
        // pattern 0x5400 | (q << 4) = 64 + q (ulp 1/16 at 64) -- the low-nibble case is the usual 0x6400 | q = 1024 + q
        const bool hi = (sb & 1) != 0;
        const uint32_t mask = hi ? 0xF0F0F0F0u : 0x0F0F0F0Fu;
        const uint32_t magic = hi ? 0x54545454u : 0x64646464u;
        const __half2 kmagic = __half2half2(__ushort_as_half((unsigned short)(hi ? 0x5400u : 0x6400u)));
        const uint32_t w[4] = {qw.x, qw.y, qw.z, qw.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t v = w[i] & mask;
            uint32_t l = prmt(v, magic, 0x4140u), u = prmt(v, magic, 0x4342u);
            __half2 lo = __hsub2_rn(*reinterpret_cast<__half2 *>(&l), kmagic);
            __half2 up = __hsub2_rn(*reinterpret_cast<__half2 *>(&u), kmagic);
            lo = __hsub2_rn(__hmul2_rn(D2, lo), M2);
            up = __hsub2_rn(__hmul2_rn(D2, up), M2);
            out[2 * i] = pack_h2_to_act<ACT>(lo);
            out[2 * i + 1] = pack_h2_to_act<ACT>(up);
        }
    }
};

template <int ACT> struct Fast16<Block<T_Q8_0>, ACT> {
    static constexpr bool available = true;
    // a 34-byte block is only 2-byte aligned: assemble the sixteen int8 from 16-bit loads
    static GG_HD void run(const uint8_t *blk, int e0, uint32_t (&out)[8])
    {
        const uint16_t *p16 = reinterpret_cast<const uint16_t *>(blk);
        const __half2 D2 = __half2half2(__ushort_as_half(p16[0]));
        const __half2 k1152 = __half2half2(__ushort_as_half((unsigned short)(0x6400u + 128u)));
        const uint16_t *q = p16 + 1 + (e0 >> 1);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t v = ((uint32_t)q[2 * i] | ((uint32_t)q[2 * i + 1] << 16)) ^ 0x80808080u;   // int8 + 128 as bytes
            uint32_t l = prmt(v, 0x64646464u, 0x4140u), u = prmt(v, 0x64646464u, 0x4342u);
            __half2 lo = __hmul2_rn(D2, __hsub2_rn(*reinterpret_cast<__half2 *>(&l), k1152));
            __half2 up = __hmul2_rn(D2, __hsub2_rn(*reinterpret_cast<__half2 *>(&u), k1152));
            out[2 * i] = pack_h2_to_act<ACT>(lo);
            out[2 * i + 1] = pack_h2_to_act<ACT>(up);
        }
    }
};

template <class Q, int MATH, int N>
GG_HD void dequant_run(const uint8_t *blk, int e0, typename Math<MATH>::T2 (&out)[N / 2])
{
    const GroupScale<MATH> g = group_scale<Q, MATH>(blk, e0);
    dequant_elems<Q, MATH, N>(blk, e0, g, out);
}

}  // namespace ggufb200
