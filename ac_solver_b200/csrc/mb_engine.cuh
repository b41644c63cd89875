// mb_engine.cuh -- the state and the kernels of the batched breadth-first engine (mbfs.cu) that the
// batched beam search (beam.cu) runs unchanged: per-search records, the chunk's segments and record log,
// root init, expansion into the log, the winner-only goal test and the path walk.  See mbfs.cu for the design.
#pragma once
#include <cstdint>

#include <cuda_runtime.h>

#include "ac_core.cuh"
#include "ac_keys.cuh"
#include "ac_sym.cuh"
#include "bfs_common.cuh"
#include "goalset.cuh"

namespace acs {

// per segment: solving child, raising child, first child of each total length < 128, first goal child
// (candidate id << 32 | goal entry)
constexpr int kMbCtrl = 131;
constexpr int kMbSol = 0, kMbErr = 1, kMbLen0 = 2, kMbGoal = 130;
constexpr uint64_t kMbNode = 1ull << 39, kMbIdx = kMbNode - 1;
constexpr uint64_t kMbTomb = 1ull << 63;  // fingerprints are 23 bits: never equal to a tombstone's
constexpr int kMbStage = 128;             // records staged per warp before a flush to the log
constexpr uint32_t kMbSymShift = 28;      // orbit search: a staged record's search id carries g in its top 4 bits

enum : int { MB_IERR_TABLE_FULL = 1, MB_IERR_SLAB_FULL = 2 };

// per-search state
struct MbSearch {
    int64_t budget, slab, cap, n_nodes, head, level_end, n_expanded, sol_gid, err_code;
    int32_t min_len, levels, done, solved, budget_hit, status, n_minlen;
    int32_t sol_len;  // total length of the state that ended a solved search: 2, or a goal state's
    int32_t minlen_log[128];
};

// run state (the host polls a lagging copy of it)
struct MbState {
    int64_t Ftot, n_seg, used, chunks, chunk_cap;
    uint64_t tmask;
    int32_t mrl, cyclical, n_search, done, ierr;
    int32_t explore;  // 1: the length-2 rule is off, searches end at a goal, their budget or exhaustion
};

struct MbEngine {
    MbState* st;
    MbSearch* srch;       // [n_search]
    uint64_t* nodes;      // [sum cap][2W+2]: key words, parent link, search id
    uint64_t* table;      // [tmask+1]
    uint64_t* log_keys;   // [rec_cap][2W]
    uint32_t* log_c;      // [rec_cap]
    uint32_t* log_s;      // [rec_cap]
    uint64_t* rec_slot;   // [rec_cap] table slot a record claimed
    unsigned long long* cursor;
    uint32_t* bitmap;     // [bitmap_words]
    uint2* rt;            // [bitmap_words + 1] {winners before the word, its bits}
    uint32_t* bsums;      // [nblk]
    unsigned long long* ctrl;  // [n_search][kMbCtrl], indexed by segment
    int32_t* seg_search;  // [n_search]
    int64_t* seg_head;    // [n_search]
    int64_t* seg_off;     // [n_search + 1]
    int64_t* seg_limit;   // [n_search] chunk candidate id limit of the commit
    int64_t* seg_base;    // [n_search] global node index of the segment's first winner, minus its rank
    int32_t* seg_of;      // [n_search] segment of a search in the current chunk
    int64_t rec_cap;
    GoalView goals;       // the goal set, if one is set
    int64_t* goal_hit;    // [n_search] goal entry a search stopped at, or -1 (allocated with the first goal set)
    uint8_t* log_g;       // [rec_cap] orbit search: the element that canonicalized each record
    const uint8_t* root_g;  // [n_search] orbit search: the element that canonicalized each root
    int32_t* goal_hit_g;  // [n_search] u with u.(end state of the returned path) = the goal entry's state, or -1
};

template <int W>
__device__ __forceinline__ uint64_t mb_hash(const Key<W>& q, uint32_t s) {
    return mix64(pb_hash<W>(q) ^ ((uint64_t)(s + 1) * 0x9E3779B97F4A7C15ull));
}

__device__ __forceinline__ int mb_segment(const int64_t* seg_off, int n_seg, int64_t p) {
    int lo = 0, hi = n_seg - 1;  // last k with seg_off[k] <= p
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(seg_off + mid) <= p) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ uint64_t mb_rank(const uint2* rt, uint64_t c) {
    const uint2 e = rt[c >> 5];
    return e.x + __popc(e.y & ((1u << (c & 31)) - 1u));
}

// ---- the segment event rule (decide kernels) ---------------------------------------------------------
struct MbEvent {
    bool solved, goal;  // a solving or goal child ends the search (goal: the goal test fired)
    int status;         // or a raising child: the reference's status
    uint64_t offset;    // the event's candidate offset from the segment's first candidate id
};

// The event that ends a segment's search among its candidates c0 + [0, limit), which lowers limit to the event:
// the first solving child `sol` (~0: none), a goal child before it (on the solving child itself the solve wins),
// then a raising child before either.
__device__ __forceinline__ MbEvent mb_event(const unsigned long long* red, unsigned long long sol, uint64_t c0,
                                            uint64_t& limit) {
    MbEvent ev{false, false, 0, 0};
    const unsigned long long err = red[kMbErr], goal = red[kMbGoal];
    if (sol != ~0ull && sol - c0 < limit) {
        ev.offset = limit = sol - c0;
        ev.solved = true;
    }
    if (goal != ~0ull && (goal >> 32) - c0 < limit) {
        ev.offset = limit = (goal >> 32) - c0;
        ev.solved = ev.goal = true;
    }
    if (err != ~0ull && (err >> 2) - c0 < limit) {  // the reference raises here, before anything later
        ev.offset = limit = (err >> 2) - c0;
        ev.status = (int)(err & 3);
        ev.solved = ev.goal = false;
    }
    return ev;
}

// The counters of a search that event ev of its segment (first candidate id 12 * head) ended, and the goal
// entry it stopped at
__device__ __forceinline__ void mb_end_at(const MbEngine& E, MbSearch& M, int s, const unsigned long long* red,
                                          const MbEvent& ev, uint64_t head) {
    const uint64_t c = 12 * head + ev.offset;
    M.n_expanded = (int64_t)(c / 12 + 1);
    if (ev.status) {
        M.status = ev.status;
        M.err_code = (int64_t)((c << 2) | (uint64_t)ev.status);
        return;
    }
    M.solved = 1;
    M.sol_gid = (int64_t)c;
    M.sol_len = 2;
    if (ev.goal) {
        const uint64_t e = red[kMbGoal] & 0xFFFFFFFFull;
        const int W = key_words(E.st->mrl);
        const uint64_t* q = E.goals.nodes + e * node_words(W);  // the goal state's key
        M.sol_len = key_len(q, W, 0) + key_len(q, W, 1);
        E.goal_hit[s] = (int64_t)e;
    }
}

// "New minimal length found" events in the reference's order, up to the segment's event: the first child of each
// new minimal total length among candidates c0 + [0, limit), and the solving child itself
__device__ __forceinline__ void mb_minlen_log(MbSearch& M, const unsigned long long* red, uint64_t c0, uint64_t limit,
                                              bool solved) {
    const uint64_t c_limit = limit + (solved ? 1 : 0);
    int min_len = M.min_len;
    for (;;) {
        unsigned long long best = ~0ull;
        int bestL = -1;
        for (int L = 0; L < min_len && L < 128; ++L) {
            const unsigned long long g = red[kMbLen0 + L];
            if (g != ~0ull && g - c0 < c_limit && g < best) {
                best = g;
                bestL = L;
            }
        }
        if (bestL < 0) break;
        min_len = bestL;
        if (M.n_minlen < 128) M.minlen_log[M.n_minlen++] = bestL;
    }
    M.min_len = min_len;
}

// ---- init: roots into their slabs and the table ----------------------------------------------
template <int W>
__global__ void mb_init_kernel(const MbEngine E, const uint64_t* roots) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= E.st->n_search || E.srch[s].done) return;
    Key<W> q;
#pragma unroll
    for (int i = 0; i < 2 * W; ++i) q.k[i] = roots[(size_t)s * 2 * W + i];
    const uint64_t idx = (uint64_t)E.srch[s].slab;
    node_store<W>(E.nodes, idx, q, -1, (int64_t)s | (E.root_g ? (int64_t)E.root_g[s] << 32 : 0));
    const uint64_t h = mb_hash<W>(q, (uint32_t)s), tmask = E.st->tmask;
    const uint64_t v = ((h >> 41) << 40) | kMbNode | (idx + 1);
    // slot by slot from the start of the 4-slot bucket: the order in which mb_insert_kernel probes
    for (uint64_t t = (h & tmask) & ~3ull, n = 0; n <= tmask; t = (t + 1) & tmask, ++n)
        if (atomicCAS((unsigned long long*)&E.table[t], 0ull, (unsigned long long)v) == 0ull) return;
    atomicOr(&E.st->ierr, MB_IERR_TABLE_FULL);
}

// ---- expand ----------------------------------------------------------------------------------------
template <int W>
__host__ __device__ constexpr int mb_stage_bytes_per_warp() {
    return kMbStage * (16 * W + 4 + 4);
}
extern __shared__ __align__(16) unsigned char mb_smem[];

template <int W, bool SYM>
__device__ __forceinline__ void mb_flush(const MbEngine& E, const ulonglong2* sk, const uint32_t* sc, const uint32_t* ss,
                                         uint32_t n, int lane) {
    unsigned long long pos = 0;
    if (lane == 0) pos = atomicAdd(E.cursor, (unsigned long long)n);
    pos = __shfl_sync(0xFFFFFFFFu, pos, 0);
    ulonglong2* dk = reinterpret_cast<ulonglong2*>(E.log_keys) + pos * W;
    for (uint32_t idx = lane; idx < n; idx += 32) {  // the log holds 12 records per parent: never full
#pragma unroll
        for (int i = 0; i < W; ++i) dk[(size_t)idx * W + i] = sk[idx * W + i];
        E.log_c[pos + idx] = sc[idx];
        if constexpr (SYM) {
            E.log_s[pos + idx] = ss[idx] & ((1u << kMbSymShift) - 1u);
            E.log_g[pos + idx] = (uint8_t)(ss[idx] >> kMbSymShift);
        } else {
            E.log_s[pos + idx] = ss[idx];
        }
    }
    __syncwarp();
}

// FIFO: the parents are expanded in FIFO order, which the move-skip rule (bfs_common.cuh) needs
template <int W, bool TRUSTED, bool SYM, bool FIFO = true>
__global__ void __launch_bounds__(256) mb_expand_kernel(const MbEngine E) {
    const MbState* st = E.st;
    if (st->done) return;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    unsigned char* p = mb_smem + wib * mb_stage_bytes_per_warp<W>();
    ulonglong2* sk = reinterpret_cast<ulonglong2*>(p);
    uint32_t* sc = reinterpret_cast<uint32_t*>(p + kMbStage * 16 * W);
    uint32_t* ss = sc + kMbStage;
    const int64_t F = st->Ftot;
    const int n_seg = (int)st->n_seg;
    const int mrl = st->mrl;
    const bool cyc = st->cyclical != 0;
    const int64_t gw = (int64_t)blockIdx.x * wpb + wib, nw = (int64_t)gridDim.x * wpb;
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t staged = 0;  // warp-uniform
    for (int64_t base = 32 * gw; base < F; base += 32 * nw) {
        const int64_t j = base + lane;
        const bool valid = j < F;
        Key<W> pk;
#pragma unroll
        for (int i = 0; i < 2 * W; ++i) pk.k[i] = 0;
        uint32_t skip = 0, s = 0;
        int k = 0, min_len = 0;
        if (valid) {
            k = mb_segment(E.seg_off, n_seg, j);
            s = (uint32_t)__ldg(E.seg_search + k);
            const MbSearch& M = E.srch[s];
            min_len = M.min_len;
            int64_t pl, tag;
            node_load<W>(E.nodes, (uint64_t)(M.slab + __ldg(E.seg_head + k) + (j - __ldg(E.seg_off + k))), pk, pl, tag);
            if constexpr (!SYM && FIFO) skip = skip_moves<TRUSTED>(pl, cyc);
        }
        unsigned long long* ctrl = E.ctrl + (int64_t)k * kMbCtrl;
        Rel<2 * W> p0, p1;
        split_key<W>(pk, p0, p1);
        const uint32_t cbase = (uint32_t)(j * 12);
#pragma unroll 4
        for (int a = 0; a < 12; ++a) {
            Rel<2 * W> r0 = p0, r1 = p1;
            bool emit = false;
            Key<W> child;
            int g = 0;
#pragma unroll
            for (int i = 0; i < 2 * W; ++i) child.k[i] = 0;
            if (valid && !((skip >> a) & 1u)) {
                bool co;
                const int stt = apply_move<2 * W, TRUSTED>(r0, r1, a, mrl, cyc, co);
                const unsigned long long c = cbase + a;
                if (stt != ST_OK) {
                    atomicMin(&ctrl[kMbErr], (c << 2) | (unsigned)stt);
                } else {
                    const int L = r0.len + r1.len;
                    if (L < min_len) atomicMin(&ctrl[kMbLen0 + L], c);
                    if (L == 2) atomicMin(&ctrl[kMbSol], c);  // before the visited test
                    child = make_key<W>(r0, r1);
                    if constexpr (SYM) child = canonical<W>(child, g);
                    emit = !key_eq<W>(child, pk);
                }
            }
            const uint32_t act = __ballot_sync(0xFFFFFFFFu, emit);
            if (emit) {
                const uint32_t q = staged + __popc(act & lt);
#pragma unroll
                for (int i = 0; i < W; ++i) sk[q * W + i] = make_ulonglong2(child.k[2 * i], child.k[2 * i + 1]);
                sc[q] = cbase + a;
                ss[q] = SYM ? s | ((uint32_t)g << kMbSymShift) : s;
            }
            staged += __popc(act);
            if (staged > kMbStage - 32) {
                __syncwarp();
                mb_flush<W, SYM>(E, sk, sc, ss, staged, lane);
                staged = 0;
            }
        }
    }
    if (staged) {
        __syncwarp();
        mb_flush<W, SYM>(E, sk, sc, ss, staged, lane);
    }
}

// ---- goal test (only with a goal set) ----------------------------------------------------------------
// The reference tests a child against the goal set after the length-2 test and before the visited test.
// Only the final winners of the bitmap need a lookup: a child whose state its search has already visited
// cannot be a goal, because that state was generated under a smaller candidate id and the search would
// have stopped there (roots are tested at init); a child that lost its slot to a smaller candidate id of
// the same state is preceded by that candidate.  The first goal child per segment goes to its control slot.
template <int W>
__global__ void __launch_bounds__(256) mb_goal_kernel(const MbEngine E) {
    const MbState* st = E.st;
    if (st->done) return;
    const unsigned long long n = *E.cursor;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t c = __ldcg(E.log_c + i);
        if (!((__ldcg(E.bitmap + (c >> 5)) >> (c & 31)) & 1u)) continue;
        const int64_t e = goal_find<W>(E.goals, load_key_cg<W>(E.log_keys, i));
        if (e < 0) continue;
        const int k = E.seg_of[__ldcg(E.log_s + i)];
        atomicMin(&E.ctrl[(int64_t)k * kMbCtrl + kMbGoal], ((unsigned long long)c << 32) | (unsigned long long)e);
    }
}

// a root in the goal set is a hit at depth 0: one visited node, nothing expanded
template <int W>
__global__ void mb_goal_roots_kernel(const MbEngine E) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= E.st->n_search || E.srch[s].done) return;
    MbSearch& M = E.srch[s];
    const int64_t e = goal_find<W>(E.goals, node_key<W>(E.nodes, (uint64_t)M.slab));
    if (e < 0) return;
    M.solved = 1;
    M.done = 1;
    M.sol_gid = -1;
    M.n_expanded = 0;
    M.sol_len = M.min_len;
    E.goal_hit[s] = e;
}

// ---- results -----------------------------------------------------------------------------------------
// path of every solved search: (action, total length) pairs from the root, then (solving action, 2) -- or
// (action, the goal state's total length) after a goal child, or nothing more when the root is a goal.
// Orbit search: the walk from the node back to the root stashes each node's element beside its action,
// then a forward pass turns the moves on stored states c_k into moves on the actual states a_k = h_k.c_k:
// h_0 = g_0^-1, the actual move of (m_k, g_k+1) is pi_{h_k}(m_k), and h_k+1 = h_k.g_k+1^-1.
template <int W, bool SYM>
__global__ void mb_path_kernel(const MbEngine E, int32_t* paths, int path_cap, int32_t* path_len) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= E.st->n_search) return;
    const MbSearch& M = E.srch[s];
    path_len[s] = 0;
    if (!M.solved) return;
    int32_t* path = paths + (size_t)s * path_cap * 2;
    const bool at_root = M.sol_gid < 0;
    const int64_t node = at_root ? 0 : M.sol_gid / 12;
    int depth = 0;
    for (int64_t g = node; g >= 0; ++depth) {
        Key<W> k;
        int64_t pl, tag;
        node_load<W>(E.nodes, (uint64_t)(M.slab + g), k, pl, tag);
        g = pl < 0 ? -1 : (pl >> 4);
    }
    path_len[s] = depth + (at_root ? 0 : 1);
    if (!at_root && depth < path_cap) {
        path[2 * depth] = (int32_t)(M.sol_gid % 12);
        path[2 * depth + 1] = M.sol_len;
    }
    int pos = depth - 1;
    for (int64_t g = node; g >= 0; --pos) {
        Key<W> k;
        int64_t pl, tag;
        node_load<W>(E.nodes, (uint64_t)(M.slab + g), k, pl, tag);
        if (pos < path_cap) {
            path[2 * pos] = pl < 0 ? -1 : (int32_t)(pl & 15);
            if constexpr (SYM) path[2 * pos] = (path[2 * pos] & 0xFF) | (int32_t)(((uint64_t)tag >> 32) & 15) << 8;
            path[2 * pos + 1] = key_total_len<W>(k);
        }
        g = pl < 0 ? -1 : (pl >> 4);
    }
    int hk = 0;  // orbit search: the frame of the path's last stored node
    if constexpr (SYM) {
        int h = 0;
        const int n = depth < path_cap ? depth : path_cap;
        for (int i = 0; i < n; ++i) {
            const int v = path[2 * i], el = v >> 8;
            if (i == 0) {
                h = sym_inv(el);
                path[0] = -1;
            } else {
                path[2 * i] = sym_pi(h, v & 0xFF);
                h = sym_mul(h, sym_inv(el));
            }
        }
        if (!at_root && depth < path_cap) path[2 * depth] = sym_pi(h, path[2 * depth]);
        hk = h;
    }
    // the element of a goal hit: u.(actual end state) = the entry's state -- the identity for an exact set
    if (E.goal_hit_g && E.goal_hit[s] >= 0) {
        Key<W> q = node_key<W>(E.nodes, (uint64_t)(M.slab + node));
        if (!at_root) {
            Rel<2 * W> r0, r1;
            split_key<W>(q, r0, r1);
            bool co;
            apply_move<2 * W, false>(r0, r1, (int)(M.sol_gid % 12), E.st->mrl, E.st->cyclical != 0, co);
            q = make_key<W>(r0, r1);
        }
        if constexpr (SYM) q = sym_apply<W>(q, hk);
        int u = 0;
        if (E.goals.symmetric) canonical<W>(q, u);
        E.goal_hit_g[s] = u;
    }
}

}  // namespace acs
