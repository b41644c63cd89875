// goalset.cuh -- a device-resident set of states keyed by the state alone (goalset.cu), and the
// lookup the batched engine (mbfs.cu) runs on the states its searches generate.
//
// Entries use the engine's node layout: key words, the link (parent entry << 4 | action) or -1, and
// the index of the entry's root (the row, or the search that committed it).  The index is an exact
// open-addressing table of 4-slot buckets, slot = 23-bit fingerprint << 40 | (entry + 1), at most
// half full.  When a state occurs more than once, the smallest entry index holds its slot.
//
// A symmetric set holds canonical forms (ac_sym.cuh) and answers "is any image of this state in the set?":
// goal_find canonicalizes the query first.  Its entries carry the element g with stored = g.(generated state)
// in bits 32..35 of the root word (the layout of an orbit search's nodes, mbfs.cu).
#pragma once
#include <cstdint>

#include <cuda_runtime.h>

#include "ac_keys.cuh"
#include "ac_sym.cuh"
#include "bfs_common.cuh"

namespace acs {

constexpr uint64_t kGsIdx = (1ull << 40) - 1;

struct GoalView {
    const uint64_t* nodes;  // [n_entries][2W+2]
    const uint64_t* table;  // [tmask+1]
    uint64_t tmask;
    int symmetric;  // entries are canonical forms: queries are canonicalized before the lookup
};

// kept out of line so that the lookups of exact sets do not carry its registers
template <int W>
__device__ __noinline__ Key<W> goal_canonical(const Key<W> q) {
    int g;
    return canonical<W>(q, g);
}

// entry index of state q (of its canonical form in a symmetric set), or -1
template <int W>
__device__ __forceinline__ int64_t goal_find(const GoalView& G, Key<W> q) {
    if (G.symmetric) q = goal_canonical<W>(q);
    const uint64_t h = pb_hash<W>(q), fp = h >> 41;
    uint64_t base = (h & G.tmask) & ~3ull;
    for (uint64_t n = 0; n <= G.tmask; n += 4, base = (base + 4) & G.tmask) {
        uint64_t v[4];
        load_bucket(G.table + base, v);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (v[j] == 0) return -1;
            if ((v[j] >> 40) != fp) continue;
            const uint64_t e = (v[j] & kGsIdx) - 1;
            if (key_eq<W>(node_key<W>(G.nodes, e), q)) return (int64_t)e;
        }
    }
    return -1;
}

}  // namespace acs

// host side of a goal set (shared by goalset.cu and mbfs.cu)
struct acs_goalset {
    int device = 0, mrl = 0, W = 1, cyclical = 0, symmetric = 0;
    int64_t n_entries = 0, n_states = 0;
    uint64_t* nodes = nullptr;  // [max(n_entries, 1)][2W+2]
    uint64_t* table = nullptr;  // [tcap]
    uint64_t tcap = 0;
    acs::GoalView view() const { return acs::GoalView{nodes, table, tcap - 1, symmetric}; }
};

namespace acs {
// Allocates and fills the index of g's nodes (g->nodes holds n_entries entries) and counts its distinct
// states.  Returns ACS_OK or an error code with the message set.
int goalset_index(acs_goalset* g, cudaStream_t s);
// ACS_OK when an engine of max_relator_length mrl, `cyclical` flag and device `device` can search with goal set g
// (an orbit search needs a symmetric set); otherwise an error code with the text "<who>_set_goals: ..."
int goalset_check(const acs_goalset* g, int mrl, int cyclical, int device, bool orbit, const char* who);
// Frees what g owns and g itself.
void goalset_free(acs_goalset* g);
}  // namespace acs
