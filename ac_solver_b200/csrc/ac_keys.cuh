// ac_keys.cuh -- packed search-node keys shared by the device searches (pbfs.cu, sbfs.cu, greedy.cu).
//
// A node key is the exact, canonical image of a padded int8 presentation: W 64-bit words per
// relator (2-bit letter codes of ac_core.cuh) with the relator length in the top 6 bits of the
// last word.  W = 1 (16-byte keys) for max_relator_length <= 29, W = 2 (32 bytes) up to 61.
// Equality of keys == equality of the reference's state tuples (breadth_first.py:87,
// greedy.py:102), so the visited sets built on them are exact, not probabilistic.
#pragma once
#include <cstdint>
#include <cstring>

#include "ac_core.cuh"

namespace acs {

constexpr uint64_t kNone = ~0ull;
constexpr uint64_t kIdxMask = (1ull << 40) - 1;  // table slot = 24-bit fingerprint | 40-bit (index + 1)

// ---- node keys: W 64-bit words per relator, length in the top 6 bits of the last word ----
constexpr int kKeyLenShift = 58;  // 2 bits per letter below it: 29 letters per word, 61 in two
constexpr int kMaxKeyMrl = 61;    // the longest relator a key holds (searches refuse wider rows)

// words per relator for relators of up to mrl letters (1 <= mrl <= kMaxKeyMrl)
__host__ __device__ constexpr int key_words(int mrl) { return mrl <= kKeyLenShift / 2 ? 1 : 2; }
// words per node record: the 2W key words, the parent link and one word the engine chooses
__host__ __device__ constexpr int node_words(int W) { return 2 * W + 2; }

template <int W>
struct Key {
    uint64_t k[2 * W];
};

// length of relator h of a key stored as 2W words (W at run time: records of either width)
__host__ __device__ __forceinline__ int key_len(const uint64_t* k, int W, int h) {
    return (int)(k[h * W + W - 1] >> kKeyLenShift);
}
template <int W>
__host__ __device__ __forceinline__ int key_len(const Key<W>& q, int h) {
    return key_len(q.k, W, h);
}
template <int W>
__host__ __device__ __forceinline__ int key_total_len(const Key<W>& q) {
    return key_len<W>(q, 0) + key_len<W>(q, 1);
}

template <int W>
__host__ __device__ __forceinline__ bool key_eq(const Key<W>& a, const Key<W>& b) {
    uint64_t d = 0;
#pragma unroll
    for (int i = 0; i < 2 * W; ++i) d |= a.k[i] ^ b.k[i];
    return d == 0;
}
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return x;
}
template <int W>
__host__ __device__ __forceinline__ uint64_t key_hash(const Key<W>& a) {
    uint64_t h = 0x9e3779b97f4a7c15ull;
#pragma unroll
    for (int i = 0; i < 2 * W; ++i) h = mix64(h ^ a.k[i]) + 0x9e3779b97f4a7c15ull * (uint64_t)(i + 1);
    return mix64(h);
}
template <int W>
__device__ __forceinline__ Key<W> make_key(const Rel<2 * W>& r0, const Rel<2 * W>& r1) {
    Key<W> q;
#pragma unroll
    for (int i = 0; i < W; ++i) {
        q.k[i] = (uint64_t)r0.b.w[2 * i] | ((uint64_t)r0.b.w[2 * i + 1] << 32);
        q.k[W + i] = (uint64_t)r1.b.w[2 * i] | ((uint64_t)r1.b.w[2 * i + 1] << 32);
    }
    q.k[W - 1] |= (uint64_t)r0.len << kKeyLenShift;
    q.k[2 * W - 1] |= (uint64_t)r1.len << kKeyLenShift;
    return q;
}
template <int W>
__device__ __forceinline__ void split_key(const Key<W>& q, Rel<2 * W>& r0, Rel<2 * W>& r1) {
#pragma unroll
    for (int i = 0; i < W; ++i) {
        r0.b.w[2 * i] = (uint32_t)q.k[i];
        r0.b.w[2 * i + 1] = (uint32_t)(q.k[i] >> 32);
        r1.b.w[2 * i] = (uint32_t)q.k[W + i];
        r1.b.w[2 * i + 1] = (uint32_t)(q.k[W + i] >> 32);
    }
    r0.len = key_len<W>(q, 0);
    r1.len = key_len<W>(q, 1);
    r0.b.w[2 * W - 1] &= (1u << 26) - 1;
    r1.b.w[2 * W - 1] &= (1u << 26) - 1;
}
template <int W>
__device__ __forceinline__ Key<W> load_key(const uint64_t* keys, uint64_t idx) {
    Key<W> q;
    if constexpr (W == 1) {
        const ulonglong2 v = reinterpret_cast<const ulonglong2*>(keys)[idx];
        q.k[0] = v.x;
        q.k[1] = v.y;
    } else {
        const ulonglong2 v0 = reinterpret_cast<const ulonglong2*>(keys)[2 * idx];
        const ulonglong2 v1 = reinterpret_cast<const ulonglong2*>(keys)[2 * idx + 1];
        q.k[0] = v0.x;
        q.k[1] = v0.y;
        q.k[2] = v1.x;
        q.k[3] = v1.y;
    }
    return q;
}
template <int W>
__device__ __forceinline__ void store_key(uint64_t* keys, uint64_t idx, const Key<W>& q) {
    if constexpr (W == 1) {
        reinterpret_cast<ulonglong2*>(keys)[idx] = make_ulonglong2(q.k[0], q.k[1]);
    } else {
        reinterpret_cast<ulonglong2*>(keys)[2 * idx] = make_ulonglong2(q.k[0], q.k[1]);
        reinterpret_cast<ulonglong2*>(keys)[2 * idx + 1] = make_ulonglong2(q.k[2], q.k[3]);
    }
}

// host-side packing of a root presentation.  A bad letter (outside {+-1,+-2}) is reported at once;
// otherwise a relator that is not zero right-padded outranks an empty one (utils.py:13-54 rejects both).
enum class RootCheck { ok, bad_letter, not_padded, empty };
template <int W>
inline RootCheck pack_root(const int8_t* p, int mrl, Key<W>& key, int lens[2]) {
    std::memset(&key, 0, sizeof(key));
    bool padded = true, empty = false;
    for (int h = 0; h < 2; ++h) {
        int len = 0;
        bool seen_zero = false;
        for (int t = 0; t < mrl; ++t) {
            const int v = p[h * mrl + t];
            if (v == 0) {
                seen_zero = true;
                continue;
            }
            if (v < -2 || v > 2) return RootCheck::bad_letter;
            if (seen_zero) padded = false;
            const uint64_t code = (uint64_t)(((v < 0) ? 2 : 0) | (v & 1));
            const int bit = 2 * len;
            key.k[h * W + bit / 64] |= code << (bit % 64);
            ++len;
        }
        lens[h] = len;
        key.k[h * W + W - 1] |= (uint64_t)len << kKeyLenShift;
        if (len == 0) empty = true;
    }
    return !padded ? RootCheck::not_padded : empty ? RootCheck::empty : RootCheck::ok;
}

// the same as a bool: false for a bad letter, and `valid` only for a root that packed cleanly
// (the valid flag of acs_sbfs_pack_root)
template <int W>
inline bool pack_root(const int8_t* p, int mrl, Key<W>& key, int lens[2], bool& valid) {
    const RootCheck rc = pack_root<W>(p, mrl, key, lens);
    valid = rc == RootCheck::ok;
    return rc != RootCheck::bad_letter;
}

// one node record (node_words(W) words) on the host
template <int W>
inline void node_pack(const Key<W>& key, int64_t link, int64_t tag, uint64_t* out) {
    for (int i = 0; i < 2 * W; ++i) out[i] = key.k[i];
    out[2 * W] = (uint64_t)link;
    out[2 * W + 1] = (uint64_t)tag;
}

// n records of `stride` words (2W for flat key arrays, node_words(W) for node records) -> int8 rows in
// record order; with gid_out, also word 2W + 1 of each node record (pbfs: the node's global id)
template <int W>
__global__ void records_unpack_kernel(const uint64_t* recs, int stride, int64_t* gid_out, int8_t* out, uint64_t n,
                                      int mrl) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t* p = recs + i * stride;
    Key<W> q;
#pragma unroll
    for (int j = 0; j < W; ++j) {
        const ulonglong2 v = reinterpret_cast<const ulonglong2*>(p)[j];
        q.k[2 * j] = v.x;
        q.k[2 * j + 1] = v.y;
    }
    Rel<2 * W> r0, r1;
    split_key<W>(q, r0, r1);
    unpack_bytes<2 * W>(out + i * 2 * mrl, r0, mrl);
    unpack_bytes<2 * W>(out + i * 2 * mrl + mrl, r1, mrl);
    if (gid_out) gid_out[i] = (int64_t)p[2 * W + 1];
}

}  // namespace acs
