// ac_sym.cuh -- the presentation symmetry group G on packed keys (ac_keys.cuh), for orbit search.
//
// G has order 16.  Element g = (r, s, a, b), index 8r + 4s + 2a + b, acts on a state by
//     s: swap x <-> y,  then  a: invert x,  then  b: invert y  (on every letter),  then  r: swap the relators.
// G acts on the AC' graph by automorphisms: a fixed permutation pi_g of the 12 move ids satisfies
//     acmove(pi_g(m), g.state) = g.acmove(m, state)
// with or without cyclic reduction, for rejected and raising moves too (the length cap and the free and
// cyclic reductions only compare letters for equality and inverseness).  The 8 trivial presentations are
// one orbit, so breadth-first search over orbits finds the exact distance to them.
//
// Canonical form (part of the search contract: it fixes the stored states and their visited order):
// the smallest of the 16 images of a key, comparing words in the order k[W-1], ..., k[0], k[2W-1], ...,
// k[W] as unsigned integers.  In row terms that orders states by (len r0, r0 read from its last letter to
// its first, len r1, r1 likewise), letters by their codes y=0, x=1, y^-1=2, x^-1=3; the order is the same
// for W = 1 and W = 2.  Among the elements giving that image, canonical() returns the smallest index.
#pragma once
#include <cstdint>

#include "ac_keys.cuh"

namespace acs {

// composition: sym_mul(g, h) is the element of "h, then g".  The relator swaps add; a swap of the
// generators moves an inversion of x before it to an inversion of y after it.
__host__ __device__ __forceinline__ int sym_mul(int g, int h) {
    const int sg = (g >> 2) & 1, ah = (h >> 1) & 1, bh = h & 1;
    const int a = ((g >> 1) & 1) ^ (sg ? bh : ah), b = (g & 1) ^ (sg ? ah : bh);
    return ((g ^ h) & 12) | (a << 1) | b;
}
__host__ __device__ __forceinline__ int sym_inv(int g) {
    return (g & 4) ? ((g & 12) | ((g & 1) << 1) | ((g >> 1) & 1)) : g;
}
// pi_g(m): one 12-nibble row per element (move m in nibble m)
__host__ __device__ __forceinline__ int sym_pi(int g, int m) {
    const uint64_t T[16] = {
        0xBA9876543210ull, 0xB6587A943210ull, 0x7A94B6583210ull, 0x7654BA983210ull,
        0x587A94B63210ull, 0x987654BA3210ull, 0x54BA98763210ull, 0x94B6587A3210ull,
        0x49A7856B0123ull, 0x456789AB0123ull, 0x89AB45670123ull, 0x856B49A70123ull,
        0x6789AB450123ull, 0xA7856B490123ull, 0x6B49A7850123ull, 0xAB4567890123ull,
    };
    return (int)((T[g] >> (4 * m)) & 15);
}

// 01-mask of the letters of one 64-bit word of a relator: bit 0 of each of the first n letters of the word
__host__ __device__ __forceinline__ uint64_t sym_low_bits(int n) {
    n = n < 0 ? 0 : (n > 32 ? 32 : n);
    return n == 32 ? 0x5555555555555555ull : (0x5555555555555555ull & ((1ull << (2 * n)) - 1ull));
}

// the letter map (s, a, b) of g applied to one relator's W words holding len letters
template <int W>
__host__ __device__ __forceinline__ void sym_letters(uint64_t* w, int len, int g) {
    const uint64_t s = (g & 4) ? ~0ull : 0ull, a = (g & 2) ? ~0ull : 0ull, b = (g & 1) ? ~0ull : 0ull;
#pragma unroll
    for (int i = 0; i < W; ++i) {
        const uint64_t lo = sym_low_bits(len - 32 * i);  // padding has code 0 (= y): leave it alone
        const uint64_t v = w[i] ^ (lo & s);
        const uint64_t x = v & lo;  // bit 0 set: an x letter
        w[i] = v ^ (((x & a) | ((lo ^ x) & b)) << 1);
    }
}

// g.q
template <int W>
__host__ __device__ __forceinline__ Key<W> sym_apply(const Key<W>& q, int g) {
    Key<W> o;
    const int h = (g >> 3) & 1;
#pragma unroll
    for (int i = 0; i < W; ++i) {
        o.k[i] = q.k[h * W + i];
        o.k[W + i] = q.k[(1 - h) * W + i];
    }
    sym_letters<W>(o.k, key_len<W>(o, 0), g);
    sym_letters<W>(o.k + W, key_len<W>(o, 1), g);
    return o;
}

// a < b in the canonical order
template <int W>
__host__ __device__ __forceinline__ bool sym_less(const Key<W>& a, const Key<W>& b) {
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int i = W - 1; i >= 0; --i)
            if (a.k[h * W + i] != b.k[h * W + i]) return a.k[h * W + i] < b.k[h * W + i];
    return false;
}

// the canonical form c = g.q of q, and g (the smallest element giving c)
template <int W>
__host__ __device__ __forceinline__ Key<W> canonical(const Key<W>& q, int& g_out) {
    const int l0 = key_len<W>(q, 0), l1 = key_len<W>(q, 1);
    Key<W> best = q;
    int bg = 0;
#pragma unroll 1
    for (int g = 0; g < 8; ++g) {  // letter maps; each gives the images g and g + 8 (relators swapped)
        Key<W> t = q;
        if (g) {
            sym_letters<W>(t.k, l0, g);
            sym_letters<W>(t.k + W, l1, g);
            if (sym_less<W>(t, best) || (g < bg && key_eq<W>(t, best))) {
                best = t;
                bg = g;
            }
        }
        Key<W> u;
#pragma unroll
        for (int i = 0; i < W; ++i) {
            u.k[i] = t.k[W + i];
            u.k[W + i] = t.k[i];
        }
        if (sym_less<W>(u, best) || (8 + g < bg && key_eq<W>(u, best))) {
            best = u;
            bg = 8 + g;
        }
    }
    g_out = bg;
    return best;
}

}  // namespace acs
