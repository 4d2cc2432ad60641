// produce.cuh -- W producers of the TMEM-fed fused Linear kernel (gemm4.cu): one thread turns 64 consecutive k of ONE
// packed weight row into 32 packed fp16 pairs, ready for tcgen05.st into the A-operand columns of tensor memory.
//
// `span` points at the row's packed bytes of one 256-wide K-span (eight 32-element blocks or one 256-element
// super-block), 16-byte aligned (the kernel stages spans in shared memory with the TMA engine); `kq` = 0..3 selects
// the 64-wide quarter.  The result is delivered in two halves of 16 registers (elements 0..31 and 32..63 of the
// quarter) through emit(half, regs) so that only 16 output registers are live at a time.
//
// Numerics (DESIGN.md section 3): the INTEGER unpack is the one of blocks.cuh / the reference, bit-exact.
//   * Producer<Q>          generic, every format: the reference's float sequence with its per-op fp16 rounding
//                          (dequant.py: d*sc, *q, -dmin*mn each rounded) -> W is bit-identical to the reference's
//                          fp16 weight.
//   * FastProducer<Q>      hot formats: the sub-block products D = fp16(d*sc), M = fp16(dmin*mn) are the reference's,
//                          the per-element step is ONE fused multiply-add fp16(D*q - M) (single rounding instead of
//                          two: the correctly rounded value of the step), hand-scheduled loads.  The Linear stays within 1e-3 of the reference's.
// W is handed to the tensor core as fp16 whatever the activation dtype is (kind::f16 takes A = f16 with B = bf16), so
// no fp16 -> bf16 conversion of the weight exists in this path.
//
// All functions are __host__ __device__ so tests/host_functors.cu can run them on the CPU against the oracle.
#pragma once
#include "blocks.cuh"

namespace ggufb200 {

// 16-byte / 4-byte loads of a staged span.  On the device the span always lives in shared memory (gemm4.cu): say so, or
// the compiler emits generic loads (LD.E.128 + address-space resolution) instead of LDS.128.
GG_HD uint4 ld_span16(const uint8_t *p)
{
#ifdef __CUDA_ARCH__
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(p)));
    return v;
#else
    return *reinterpret_cast<const uint4 *>(p);
#endif
}
GG_HD uint32_t ld_span4(const uint8_t *p)
{
#ifdef __CUDA_ARCH__
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)));
    return v;
#else
    return *reinterpret_cast<const uint32_t *>(p);
#endif
}

GG_HD uint32_t h2_bits(__half2 v) { return *reinterpret_cast<uint32_t *>(&v); }
GG_HD __half2 bits_h2(uint32_t v) { return *reinterpret_cast<__half2 *>(&v); }

// ------------------------------------------------------------------ generic: reference rounding sequence, any format
template <class Q> struct Producer {
    static constexpr bool fast = false;
    template <class Emit> static GG_HD void run64(const uint8_t *span, int kq, Emit &&emit)
    {
        constexpr int GROUP = GroupOf<Q>::value;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int k = kq * 64 + half * 32;                    // position inside the span
            const uint8_t *blk = span + (k / Q::BS) * Q::TS;
            const int e0 = k % Q::BS;
            const GroupScale<kF16> g0 = group_scale<Q, kF16>(blk, e0);
            GroupScale<kF16> g1 = g0;
            if constexpr (GROUP == 16) g1 = group_scale<Q, kF16>(blk, e0 + 16);
            uint32_t o[16];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                __half2 v[4];
                dequant_elems<Q, kF16, 8>(blk, e0 + c * 8, (GROUP == 16 && c >= 2) ? g1 : g0, v);
#pragma unroll
                for (int j = 0; j < 4; ++j) o[4 * c + j] = h2_bits(v[j]);
            }
            emit(half, o);
        }
    }
};

// FMA = true: the per-element step of Q4_K / Q5_K is one fused multiply-add (the `fast` contract); false: multiply, round,
// subtract, round -- the reference's sequence, bit-identical weight (the other hand-written producers have a single-rounding
// float step in the reference already and ignore the flag).
template <class Q, bool FMA = true> struct FastProducer : Producer<Q> {};   // formats without a hand-written producer use the generic one



GG_HD __half2 h2_fma(__half2 a, __half2 b, __half2 c)
{
#ifdef __CUDA_ARCH__
    return __hfma2(a, b, c);
#else
    // host stand-in: fp16 products / sums of these magnitudes are exact in binary64, one rounding to fp16
    const float2 fa = __half22float2(a), fb = __half22float2(b), fc = __half22float2(c);
    const double x = (double)fa.x * (double)fb.x + (double)fc.x, y = (double)fa.y * (double)fb.y + (double)fc.y;
    return __halves2half2(__double2half(x), __double2half(y));
#endif
}

template <bool FMA> GG_HD __half2 k_step(__half2 q, __half2 D, __half2 nM)
{
    if constexpr (FMA) return h2_fma(q, D, nM);
    else return __hadd2_rn(__hmul2_rn(D, q), nM);        // fp16(fp16(D*q) - M): x + (-M) == x - M exactly
}

// (sc, mn) bytes -> (d*sc, dmin*mn) as one rounded half2 product, exactly the reference's fp16(d*sc), fp16(dmin*mn)
GG_HD __half2 k_dm(uint32_t dm_bits, uint32_t sc, uint32_t mn)
{
    const __half2 k1024 = __half2half2(__ushort_as_half((unsigned short)0x6400u));
    const __half2 scm = __hsub2_rn(bits_h2((sc & 0xFFu) | ((mn & 0xFFu) << 16) | 0x64006400u), k1024);
    return __hmul2_rn(bits_h2(dm_bits), scm);
}

// the two 6-bit (scale, min) pairs of sub-blocks 2kq and 2kq+1 from the three scale words (dequant.py:129-139),
// returned as two bytes each: sc = sc0 | sc1 << 8, mn likewise
GG_HD void k_scale_pair(uint32_t w0, uint32_t w1, uint32_t w2, int kq, uint32_t &sc, uint32_t &mn)
{
    const int sh = 16 * (kq & 1);
    const uint32_t a = (w0 >> sh) & 0xFFFFu, b = (w1 >> sh) & 0xFFFFu, c = (w2 >> sh) & 0xFFFFu;
    if (kq < 2) {
        sc = a & 0x3F3Fu;
        mn = b & 0x3F3Fu;
    } else {
        sc = (c & 0x0F0Fu) | ((a >> 2) & 0x3030u);
        mn = ((c >> 4) & 0x0F0Fu) | ((b >> 2) & 0x3030u);
    }
}

// four unsigned bytes (values < 256 in the low-nibble case, q << 4 in the in-place high-nibble case) -> two half2 of
// exact integers:  LOW: 0x6400 | u = 1024 + u;  HIGH nibble kept in place: 0x5400 | (q << 4) = 64 + q
template <bool HIGH> GG_HD void bytes_to_h2(uint32_t v, __half2 &lo, __half2 &hi)
{
    const uint32_t magic = HIGH ? 0x54545454u : 0x64646464u;
    const __half2 off = __half2half2(__ushort_as_half((unsigned short)(HIGH ? 0x5400u : 0x6400u)));
    lo = __hsub2_rn(bits_h2(prmt(v, magic, 0x4140u)), off);
    hi = __hsub2_rn(bits_h2(prmt(v, magic, 0x4342u)), off);
}

// ------------------------------------------------------------------ Q4_K  (dequant.py:180-195)
template <bool FMA> struct FastProducer<Block<T_Q4_K>, FMA> {
    static constexpr bool fast = true;
    template <class Emit> static GG_HD void run64(const uint8_t *blk, int kq, Emit &&emit)
    {
        const uint4 h = ld_span16(blk);                       // d | dmin << 16, scales[12]
        const uint4 qa = ld_span16(blk + 16 + 32 * kq);       // bytes 0..15 of the 64-element group
        const uint4 qb = ld_span16(blk + 32 + 32 * kq);       // bytes 16..31
        uint32_t sc, mn;
        k_scale_pair(h.y, h.z, h.w, kq, sc, mn);
        const __half2 dm0 = k_dm(h.x, sc, mn), dm1 = k_dm(h.x, sc >> 8, mn >> 8);
        const uint32_t w[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
        {   // sub-block 2kq: low nibbles
            const __half2 D = __low2half2(dm0), nM = __hneg2(__high2half2(dm0));
            uint32_t o[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                __half2 a, b;
                bytes_to_h2<false>(w[i] & 0x0F0F0F0Fu, a, b);
                o[2 * i] = h2_bits(k_step<FMA>(a, D, nM));
                o[2 * i + 1] = h2_bits(k_step<FMA>(b, D, nM));
            }
            emit(0, o);
        }
        {   // sub-block 2kq+1: high nibbles, converted in place (64 + q)
            const __half2 D = __low2half2(dm1), nM = __hneg2(__high2half2(dm1));
            uint32_t o[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                __half2 a, b;
                bytes_to_h2<true>(w[i] & 0xF0F0F0F0u, a, b);
                o[2 * i] = h2_bits(k_step<FMA>(a, D, nM));
                o[2 * i + 1] = h2_bits(k_step<FMA>(b, D, nM));
            }
            emit(1, o);
        }
    }
};

// ------------------------------------------------------------------ Q5_K  (dequant.py:159-178)
template <bool FMA> struct FastProducer<Block<T_Q5_K>, FMA> {
    static constexpr bool fast = true;
    template <class Emit> static GG_HD void run64(const uint8_t *blk, int kq, Emit &&emit)
    {
        const uint4 h = ld_span16(blk);
        const uint4 ha = ld_span16(blk + 16), hb = ld_span16(blk + 32);   // qh[32]
        const uint4 qa = ld_span16(blk + 48 + 32 * kq);
        const uint4 qb = ld_span16(blk + 64 + 32 * kq);
        uint32_t sc, mn;
        k_scale_pair(h.y, h.z, h.w, kq, sc, mn);
        const __half2 dm0 = k_dm(h.x, sc, mn), dm1 = k_dm(h.x, sc >> 8, mn >> 8);
        const uint32_t w[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
        const uint32_t qh[8] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const __half2 dm = half ? dm1 : dm0;
            const __half2 D = __low2half2(dm), nM = __hneg2(__high2half2(dm));
            const int sb = 2 * kq + half;
            uint32_t o[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const uint32_t lo = (half ? (w[i] >> 4) : w[i]) & 0x0F0F0F0Fu;
                const uint32_t u = lo | (((qh[i] >> sb) & 0x01010101u) << 4);      // 5-bit value per byte
                __half2 a, b;
                bytes_to_h2<false>(u, a, b);
                o[2 * i] = h2_bits(k_step<FMA>(a, D, nM));
                o[2 * i + 1] = h2_bits(k_step<FMA>(b, D, nM));
            }
            emit(half, o);
        }
    }
};

// ------------------------------------------------------------------ Q8_0  (dequant.py:65-69)
// eight 34-byte blocks per span; block b starts at 34*b (4-byte aligned for even b, 2 mod 4 for odd b).  d*x has a single
// rounding in the reference as well, so this producer is bit-exact; it only replaces the 2-byte loads of the generic one
// by aligned 4-byte words.
template <bool FMA> struct FastProducer<Block<T_Q8_0>, FMA> {
    static constexpr bool fast = true;
    template <class Emit> static GG_HD void run64(const uint8_t *span, int kq, Emit &&emit)
    {
        const __half2 k1152 = __half2half2(__ushort_as_half((unsigned short)(0x6400u + 128u)));
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            // blocks 2kq (offset 68kq, 4-byte aligned) and 2kq+1 (offset 68kq + 34 = 2 mod 4)
            const uint8_t *p = span + 68 * kq + (half ? 32 : 0);
            uint32_t o[16];
            if (half == 0) {
                // word 0 = d | x0 x1 << 16; words 1..7 = x2..x29; word 8 low half = x30 x31
                uint32_t wd[9];
#pragma unroll
                for (int i = 0; i < 9; ++i) wd[i] = ld_span4(p + 4 * i);
                const __half2 D = __half2half2(__ushort_as_half((unsigned short)(wd[0] & 0xFFFFu)));
#pragma unroll
                for (int i = 0; i < 9; ++i) wd[i] ^= 0x80808080u;
#pragma unroll
                for (int j = 0; j < 16; ++j) {   // pair j = elements 2j, 2j+1 = bytes 2 + 2j, 3 + 2j of the block
                    const int byte = 2 + 2 * j;
                    const uint32_t sel = (byte & 2) ? 0x4342u : 0x4140u;
                    const __half2 x = __hsub2_rn(bits_h2(prmt(wd[byte >> 2], 0x64646464u, sel)), k1152);
                    o[j] = h2_bits(__hmul2_rn(D, x));
                }
            } else {
                // p = block start - 2: word 0 high half = d; words 1..8 = x0..x31
                uint32_t wd[9];
#pragma unroll
                for (int i = 0; i < 9; ++i) wd[i] = ld_span4(p + 4 * i);
                const __half2 D = __half2half2(__ushort_as_half((unsigned short)(wd[0] >> 16)));
#pragma unroll
                for (int i = 1; i < 9; ++i) wd[i] ^= 0x80808080u;
#pragma unroll
                for (int j = 0; j < 16; ++j) {   // pair j = bytes 4 + 2j, 5 + 2j relative to p
                    const int byte = 4 + 2 * j;
                    const uint32_t sel = (byte & 2) ? 0x4342u : 0x4140u;
                    const __half2 x = __hsub2_rn(bits_h2(prmt(wd[byte >> 2], 0x64646464u, sel)), k1152);
                    o[j] = h2_bits(__hmul2_rn(D, x));
                }
            }
            emit(half, o);
        }
    }
};

// ------------------------------------------------------------------ Q4_0  (dequant.py:115-123)
// eight 18-byte blocks per span; d*(q-8) has a single rounding in the reference: bit-exact, aligned word loads.
// A 64-wide quarter = blocks 2kq, 2kq+1 = 36 bytes at offset 36kq (4-byte aligned): [d0 qs0[16]] [d1 qs1[16]].
template <bool FMA> struct FastProducer<Block<T_Q4_0>, FMA> {
    static constexpr bool fast = true;
    template <class Emit> static GG_HD void run64(const uint8_t *span, int kq, Emit &&emit)
    {
        uint32_t wd[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) wd[i] = ld_span4(span + 36 * kq + 4 * i);
        const __half2 k1032 = __half2half2(__ushort_as_half((unsigned short)(0x6400u + 8u)));
        const __half2 k72 = __half2half2(__ushort_as_half((unsigned short)0x5480u));      // 64 + 8
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            // block `half`: d at byte 18*half, qs at 18*half + 2 .. +17.  Element e < 16: low nibble of qs[e]; e >= 16: high nibble of qs[e-16]
            const int base = 18 * half;
            const uint32_t dbits = (wd[base >> 2] >> (8 * (base & 3))) & 0xFFFFu;
            const __half2 D = __half2half2(__ushort_as_half((unsigned short)dbits));
            uint32_t o[16];
#pragma unroll
            for (int j = 0; j < 8; ++j) {      // pair j of the low-nibble half: bytes base+2+2j, +3+2j
                const int byte = base + 2 + 2 * j;
                const uint32_t sel = (byte & 2) ? 0x4342u : 0x4140u;
                const uint32_t word = wd[byte >> 2];
                const __half2 lo = __hsub2_rn(bits_h2(prmt(word & 0x0F0F0F0Fu, 0x64646464u, sel)), k1032);
                const __half2 hi = __hsub2_rn(bits_h2(prmt(word & 0xF0F0F0F0u, 0x54545454u, sel)), k72);
                o[j] = h2_bits(__hmul2_rn(D, lo));
                o[8 + j] = h2_bits(__hmul2_rn(D, hi));
            }
            emit(half, o);
        }
    }
};

// ------------------------------------------------------------------ Q6_K  (dequant.py:141-157)
// [ql 128][qh 64][scales i8 16][d]; 210-byte blocks are only 2-byte aligned in the canonical layout, so this producer is
// used with the re-packed (16-byte aligned, padded) span layout only.  (d*sc) and (*q) round separately in the reference;
// here q*(d*sc) is one rounded product of the reference's fp16(d*sc) -- the same single multiply, hence bit-exact.
template <bool FMA> struct FastProducer<Block<T_Q6_K>, FMA> {
    static constexpr bool fast = true;
    template <class Emit> static GG_HD void run64(const uint8_t *blk, int kq, Emit &&emit)
    {
        // quarter kq covers elements 64kq..64kq+63: h = kq >> 1 (128-half), r0 = 64 * (kq & 1)
        const int hh = kq >> 1, up = kq & 1;
        // ql bytes 64h + (r & 63), nibble r >> 6 -> for this quarter: all 64 bytes ql[64h .. 64h+63], nibble `up`
        // qh bytes 128 + 32h + (r & 31), 2-bit field r >> 5 -> fields 2*up (first 32 elements) and 2*up + 1 (last 32)
        const uint8_t *ql = blk + 64 * hh;
        const uint4 h0 = ld_span16(blk + 128 + 32 * hh), h1 = ld_span16(blk + 144 + 32 * hh);
        const uint32_t hw[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        const uint32_t sw = ld_span4(blk + 192 + 4 * kq);     // four int8 scales of this quarter
        const __half d = __ushort_as_half((unsigned short)(ld_span4(blk + 208) & 0xFFFFu));    // bytes 210, 211 are row padding of the span layout
        const __half2 k1056 = __half2half2(__ushort_as_half((unsigned short)(0x6400u + 32u)));
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const uint4 l0 = ld_span16(ql + 32 * half), l1 = ld_span16(ql + 32 * half + 16);
            const uint32_t lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
            // scales: elements 0..15 of this 32-run use scale 2*half, 16..31 use 2*half+1
            const int s0 = (int)(int8_t)(sw >> (16 * half)), s1 = (int)(int8_t)(sw >> (16 * half + 8));
            const __half2 D0 = __half2half2(__hmul_rn(d, __int2half_rn(s0))), D1 = __half2half2(__hmul_rn(d, __int2half_rn(s1)));
            const int fsh = 2 * (2 * up + half);
            uint32_t o[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const uint32_t lo = (up ? (lw[i] >> 4) : lw[i]) & 0x0F0F0F0Fu;
                const uint32_t u = lo | (((hw[i] >> fsh) & 0x03030303u) << 4);     // q + 32 per byte
                const __half2 D = i < 4 ? D0 : D1;
                o[2 * i] = h2_bits(__hmul2_rn(D, __hsub2_rn(bits_h2(prmt(u, 0x64646464u, 0x4140u)), k1056)));
                o[2 * i + 1] = h2_bits(__hmul2_rn(D, __hsub2_rn(bits_h2(prmt(u, 0x64646464u, 0x4342u)), k1056)));
            }
            emit(half, o);
        }
    }
};

// ---------------------------------------------------------------- A-stage ownership of the TMEM-fed kernel (gemm4.cu)
// The ring of A stages in tensor memory has a multiple of 4 stages and relies on ONE writer group per stage: producer group g
// (0..3) writes exactly the k-blocks whose GLOBAL index is == g (mod 4), so the parity wait on a stage's `empty` barrier can
// never be satisfied by a phase two uses old.  `it0` = global index of the item's first k-block (not a multiple of 4 once an
// earlier item of this CTA pair carried a LoRA k-block).
GG_HD int g4_group_quarter(int g, int it0) { return (g - it0) & 3; }                    // the group's quarter of every span of the item
GG_HD int g4_lora_group(int it0, int nspans) { return (it0 + 4 * nspans) & 3; }         // the group that writes the LoRA k-block

}  // namespace ggufb200
