// bfs_common.cuh -- device helpers shared by the breadth-first engines (pbfs.cu, mbfs.cu):
// node store layout, the visited-table hash and bucket load, the move-skip rule and block scans.
#pragma once
#include <cstdint>

#include "ac_core.cuh"
#include "ac_keys.cuh"

namespace acs {

constexpr int kScanT = 256, kScanPer = 8, kScanBlock = kScanT * kScanPer;  // words per scan block

// node store: key words, then (parent global id << 4 | action) or -1, then one more word
// (pbfs: the node's global id; mbfs: the search the node belongs to)
template <int W>
__device__ __forceinline__ Key<W> node_key(const uint64_t* nodes, uint64_t idx) {
    Key<W> q;
    const ulonglong2* p = reinterpret_cast<const ulonglong2*>(nodes + idx * node_words(W));
#pragma unroll
    for (int i = 0; i < W; ++i) {
        const ulonglong2 v = p[i];
        q.k[2 * i] = v.x;
        q.k[2 * i + 1] = v.y;
    }
    return q;
}
template <int W>
__device__ __forceinline__ void node_load(const uint64_t* nodes, uint64_t idx, Key<W>& q, int64_t& parent, int64_t& gid) {
    const ulonglong2* p = reinterpret_cast<const ulonglong2*>(nodes + idx * node_words(W));
#pragma unroll
    for (int i = 0; i < W; ++i) {
        const ulonglong2 v = p[i];
        q.k[2 * i] = v.x;
        q.k[2 * i + 1] = v.y;
    }
    const ulonglong2 t = p[W];
    parent = (int64_t)t.x;
    gid = (int64_t)t.y;
}
template <int W>
__device__ __forceinline__ void node_store(uint64_t* nodes, uint64_t idx, const Key<W>& q, int64_t parent, int64_t gid) {
    uint64_t* p = nodes + idx * node_words(W);
    if constexpr (W == 1) {  // one 256-bit store: one memory request per node
        asm volatile("st.global.v4.u64 [%0], {%1,%2,%3,%4};" ::"l"(p), "l"(q.k[0]), "l"(q.k[1]), "l"((uint64_t)parent),
                     "l"((uint64_t)gid)
                     : "memory");
    } else {
        ulonglong2* v = reinterpret_cast<ulonglong2*>(p);
        v[0] = make_ulonglong2(q.k[0], q.k[1]);
        v[1] = make_ulonglong2(q.k[2], q.k[3]);
        v[2] = make_ulonglong2((uint64_t)parent, (uint64_t)gid);
    }
}

// ---- hashing: slot = low bits, committed fingerprint = bits 41..63, tentative fp = bits 58..63,
// owner from a separately mixed product (must be independent of the slot bits, see sbfs.cu) ----
template <int W>
__host__ __device__ __forceinline__ uint64_t pb_hash(const Key<W>& q) {
    uint64_t h = q.k[0] * 0x9E3779B97F4A7C15ull;
    h ^= h >> 32;
#pragma unroll
    for (int i = 1; i < 2 * W; ++i) {
        h = (h + q.k[i]) * 0xD6E8FEB86659FD93ull;
        h ^= h >> 29;
    }
    h *= 0xC4CEB9FE1A85EC53ull;
    h ^= h >> 32;
    return h;
}

template <int W>
__device__ __forceinline__ Key<W> load_key_cg(const uint64_t* keys, uint64_t idx) {
    Key<W> q;
#pragma unroll
    for (int i = 0; i < W; ++i) {
        const ulonglong2 v = __ldcg(reinterpret_cast<const ulonglong2*>(keys) + W * idx + i);
        q.k[2 * i] = v.x;
        q.k[2 * i + 1] = v.y;
    }
    return q;
}

// Moves that need not be generated from a node, given the link (parent gid << 4 | action) that created it: their
// children are certainly duplicates of candidates with a SMALLER id, so they can never win a slot, start a new
// minimal length, be the first solved child or move the budget cut -- skipping them changes nothing observable.
//  * back edge (searches without cyclic reduction): the move that undoes the creating move leads to the parent.
//    Inverse pairs: r1<-r1 r0 / r1<-r1 r0^-1 (0,2); r0<-r0 r1^-1 / r0<-r0 r1 (1,3); conjugation by g / g^-1.
//  * commuting conjugations: ids 4..11 conjugate r0 (odd ids) or r1 (even ids), and the two act on different
//    relators independently (length cap, free / cyclic reduction are per relator).  For B = S.m' and a conjugation
//    m < m' of the OTHER relator, B.m = (S.m).m'; the state S.m was discovered no later than S's expansion with an
//    id below B's, so it is expanded before B and generates the same child under a smaller candidate id.
// Not for children of the root: a caller-supplied root need not be a normal form, and its children are the first
// fully simplified states.  The argument only uses FIFO order within one search.
template <bool TRUSTED>
__device__ __forceinline__ uint32_t skip_moves(int64_t pl, bool cyc) {
    if (!TRUSTED || pl < 16) return 0u;
    const int mp = (int)(pl & 15);
    uint32_t skip = 0;
    if (!cyc) skip |= 1u << ((0x7654BA981032ull >> (4 * mp)) & 15);
    if (mp >= 4) skip |= ((mp & 1) ? 0x550u : 0xAA0u) & ((1u << mp) - 1u);
    return skip;
}

// one 256-bit load of a 4-slot bucket (a 32-byte sector): ONE memory request.  Measured on B200
// (scripts/microbench/random_access.cu): the chip sustains ~37 G random load requests/s whether
// a request carries 8 or 32 bytes, and two 16-byte loads of one sector cost two requests.
__device__ __forceinline__ void load_bucket(const uint64_t* p, uint64_t (&v)[4]) {
    asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
}

// exclusive block scan over kScanT threads; `total` = sum over the block
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t& total) {
    __shared__ uint32_t ws[kScanT / 32];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, x, off);
        if (lane >= off) x += t;
    }
    __syncthreads();
    if (lane == 31) ws[wid] = x;
    __syncthreads();
    uint32_t before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kScanT / 32; ++w) {
        const uint32_t s = ws[w];
        if (w < (int)wid) before += s;
        tot += s;
    }
    total = tot;
    return before + x - v;
}

}  // namespace acs
