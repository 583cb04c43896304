// Device building blocks of the two integer-pipe searches: the full-row kernel (search.cu) and the
// windowed one (search_range.cu). Descriptor loads, the carry-save Hamming trees and the IMAD helper;
// the exactness argument for the cost << 16 | column keys is in search.cu's header comment.
#pragma once

#include "kernels.cuh"

namespace bicos_b200 {
namespace {

__device__ __forceinline__ uint32_t xor3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__device__ __forceinline__ uint32_t maj3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

template<int K>
struct Desc {
    uint32_t w[K];
};

template<int K>
__device__ __forceinline__ Desc<K> load_desc(const uint32_t* p) {
    Desc<K> d;
    if constexpr (K == 1) {
        d.w[0] = *p;
    } else if constexpr (K == 2) {
        const uint2 v = *reinterpret_cast<const uint2*>(p);
        d.w[0] = v.x;
        d.w[1] = v.y;
    } else {
#pragma unroll
        for (int q = 0; q < K / 4; ++q) {
            const uint4 v = reinterpret_cast<const uint4*>(p)[q];
            d.w[4 * q + 0] = v.x;
            d.w[4 * q + 1] = v.y;
            d.w[4 * q + 2] = v.z;
            d.w[4 * q + 3] = v.w;
        }
    }
    return d;
}

struct Csa {
    uint32_t s, c; // ones and twos of a + b + c, bit position by bit position
};

__device__ __forceinline__ Csa csa(uint32_t a, uint32_t b, uint32_t c) {
    return { xor3(a, b, c), maj3(a, b, c) };
}

// a * m + c as one IMAD with m a run-time 1 or 2 (SearchArgs::one / two): ptxas would otherwise emit
// part of the popcount sums as IADD3 / LEA, i.e. on the ALU pipe the LOP3s already fill, while the FMA
// pipe idles.
__device__ __forceinline__ uint32_t mad(uint32_t a, uint32_t m, uint32_t c) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(m), "r"(c));
    return d;
}

struct Weights {
    uint32_t one, two, shl16; // 1, 2, 65536
};

// popcount(l ^ r) over K words (reference ham(), bicos.hpp:29-48). Every carry-save adder trades one
// POPC (8 issue cycles of the 16-lane XU pipe per warp) for two LOP3 (2 x 2 cycles of the ALU pipe).
// From 256 bits on the ALU pipe is the busier one; `light` pairs skip the last adder and spend one more
// POPC instead. Measured (tools/search_tune, MIX = light pairs per thread): no mix beats MIX = 0 at
// 256 bits (0.857 / 0.831 / 0.841 T pairs/s for MIX 0 / 1 / 2) and the differences at 384 / 512 bits
// are below 1 %, so the full trees are the default and `light` stays a tuning knob.
template<int K>
__device__ __forceinline__ uint32_t hamming(const Desc<K>& l, const Desc<K>& r, bool light, const Weights w) {
    uint32_t x[K];
#pragma unroll
    for (int k = 0; k < K; ++k)
        x[k] = l.w[k] ^ r.w[k];
    if constexpr (K == 1) {
        return __popc(x[0]);
    } else if constexpr (K == 2) {
        return __popc(x[0]) + __popc(x[1]);
    } else if constexpr (K == 4) {
        // full adder over three words: ones in s, twos in c -> 3 POPC instead of 4
        const Csa a = csa(x[0], x[1], x[2]);
        return __popc(a.s) + __popc(x[3]) + 2 * __popc(a.c);
    } else if constexpr (K == 8) {
        const Csa a = csa(x[0], x[1], x[2]), b = csa(x[3], x[4], x[5]), c = csa(a.s, b.s, x[6]);
        const uint32_t ones = mad(__popc(c.s), w.one, __popc(x[7]));
        if (light) // 3 adders, 5 POPC
            return mad(mad(mad(__popc(a.c), w.one, __popc(b.c)), w.one, __popc(c.c)), w.two, ones);
        const Csa t = csa(a.c, b.c, c.c); // 4 adders, 4 POPC: ones c.s x7, twos t.s, fours t.c
        return mad(mad(__popc(t.c), w.two, __popc(t.s)), w.two, ones);
    } else if constexpr (K == 12) {
        const Csa a = csa(x[0], x[1], x[2]), b = csa(x[3], x[4], x[5]), c = csa(x[6], x[7], x[8]), d = csa(x[9], x[10], x[11]);
        const Csa e = csa(a.s, b.s, c.s);
        const uint32_t ones = mad(__popc(e.s), w.one, __popc(d.s));
        const uint32_t de = mad(__popc(d.c), w.one, __popc(e.c));
        if (light) // 5 adders, 7 POPC
            return mad(mad(mad(mad(__popc(a.c), w.one, __popc(b.c)), w.one, __popc(c.c)), w.one, de), w.two, ones);
        const Csa t = csa(a.c, b.c, c.c); // 6 adders, 6 POPC: twos t.s d.c e.c, fours t.c
        return mad(mad(mad(__popc(t.c), w.two, __popc(t.s)), w.one, de), w.two, ones);
    } else {
        static_assert(K == 16, "descriptor widths: 1, 2, 4, 8, 12 or 16 words");
        const Csa a = csa(x[0], x[1], x[2]), b = csa(x[3], x[4], x[5]), c = csa(x[6], x[7], x[8]), d = csa(x[9], x[10], x[11]),
                  e = csa(x[12], x[13], x[14]);
        const Csa f = csa(a.s, b.s, c.s), g = csa(d.s, e.s, x[15]);
        const uint32_t ones = mad(__popc(f.s), w.one, __popc(g.s));
        const uint32_t defg = mad(mad(mad(__popc(d.c), w.one, __popc(e.c)), w.one, __popc(f.c)), w.one, __popc(g.c));
        if (light) // 7 adders, 9 POPC
            return mad(mad(mad(mad(__popc(a.c), w.one, __popc(b.c)), w.one, __popc(c.c)), w.one, defg), w.two, ones);
        const Csa t = csa(a.c, b.c, c.c); // 8 adders, 8 POPC: twos t.s d.c e.c f.c g.c, fours t.c
        return mad(mad(mad(__popc(t.c), w.two, __popc(t.s)), w.one, defg), w.two, ones);
    }
}

} // namespace
} // namespace bicos_b200
