// greedy.cu -- batched greedy (best-first) search of the AC graph, bit-exact with the
// reference's greedy_search() (ac_solver/search/greedy.py:15-121, relative to /root/reference).
//
// The reference pops the minimum of a heap keyed (total_length, depth, state tuple) -- the
// tuple compares element-wise as signed ints with the padding zeros taking part
// (greedy.py:104-113) -- expands its 12 children in action order, returns at the first child
// of total length 2 (before the visited test), pushes unseen children, and tests the node
// budget after each node.  Keys are distinct, so the pop sequence is a property of the key
// order alone and any correct priority queue reproduces it.
//
// B200 formulation: ONE WARP PER SEARCH, many searches per launch (BASELINE config 3 runs
// ~1190 independent presentations); all state lives in HBM pools indexed by search.
//   pop     32-ary implicit heap: a sift-down level loads 32 children (one coalesced 256 B
//           read) plus their keys, and a 5-step shuffle tournament picks the minimum under the
//           exact (length, depth, state) order -> 4 levels for 1e6 entries.
//   expand  lanes 0..11 apply the 12 moves to the popped node (ac_core.cuh).
//   dedup   exact open-addressing table private to the search (slot = 24-bit fingerprint |
//           40-bit index+1, keys always compared); the 12 lanes probe in parallel and settle
//           slot conflicts by lane order, so duplicates inside one expansion keep the lower
//           action, as the sequential reference does.
//   append  new nodes are numbered in action order (ballot + popc), so the node array is the
//           reference's insertion order; then pushed (sift-up, <= 4 levels).
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "ac_core.cuh"
#include "ac_keys.cuh"
#include "acs_internal.h"
#include "goalset.cuh"

namespace acs {

constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kHeapArity = 32;

struct GreedyRec {  // per-search result record (device -> host)
    int32_t solved, status, budget_hit, n_minlen;
    uint64_t n_nodes, n_expanded, n_moves, heap_left;
    uint64_t final_node;
    int32_t final_action, final_len;
    int32_t rounds, engine;  // bucket rounds executed; 1 = bucket kernel, 2 = heap kernel (fallback or forced)
    int32_t minlen_log[128];
    int64_t goal;  // goal entry the search stopped at, or -1 (written by the goal instantiations only)
};

struct GreedyArgs {
    uint64_t* keys;    // [S][cap][2W]
    uint64_t* parent;  // [S][cap]
    uint32_t* depth;   // [S][cap]
    uint64_t* heap;    // [S][cap]   entry = ((len << 24 | depth) << 32) | node index
    uint64_t* table;   // [S][tcap]
    const uint64_t* roots;  // [S][2W] packed root keys
    GreedyRec* rec;    // [S]
    uint64_t cap, tcap, budget;
    int n_search, mrl, cyclical;
    int fallback_only;  // run only the searches the bucket kernel handed back (status kGbFallback)
};

// signed order of the letters: -2 < -1 < +1 < +2  <->  codes 2 < 3 < 1 < 0
__device__ __forceinline__ int letter_rank(uint32_t code) { return (0x4B >> (2 * code)) & 3; }

// three-way compare of two relators as zero-padded signed tuples
template <int N>
__device__ __forceinline__ int rel_cmp(const Rel<N>& a, const Rel<N>& b) {
    const int d = ctz<N>(a.b ^ b.b) >> 1;
    const int m = min(a.len, b.len);
    if (d < m) return letter_rank(get_code<N>(a.b, d)) < letter_rank(get_code<N>(b.b, d)) ? -1 : 1;
    if (a.len == b.len) return 0;
    // one word is a proper prefix of the other: a padding zero meets a letter at position m
    if (a.len < b.len) return (get_code<N>(b.b, m) & 2u) ? 1 : -1;  // 0 vs b[m]: b[m] < 0  =>  a > b
    return (get_code<N>(a.b, m) & 2u) ? -1 : 1;
}
template <int W>
__device__ __forceinline__ bool key_less(const Key<W>& a, const Key<W>& b) {
    Rel<2 * W> a0, a1, b0, b1;
    split_key<W>(a, a0, a1);
    split_key<W>(b, b0, b1);
    const int c = rel_cmp<2 * W>(a0, b0);
    if (c) return c < 0;
    return rel_cmp<2 * W>(a1, b1) < 0;
}
// heap order: (total length, depth) in the high word, then the state tuple
template <int W>
__device__ __forceinline__ bool entry_less(uint64_t e1, const Key<W>& k1, uint64_t e2, const Key<W>& k2) {
    const uint32_t h1 = (uint32_t)(e1 >> 32), h2 = (uint32_t)(e2 >> 32);
    if (h1 != h2) return h1 < h2;
    return key_less<W>(k1, k2);
}

template <int W>
__device__ __forceinline__ Key<W> shfl_key(const Key<W>& k, int src) {
    Key<W> r;
#pragma unroll
    for (int i = 0; i < 2 * W; ++i) r.k[i] = __shfl_sync(kFull, k.k[i], src);
    return r;
}
template <int W>
__device__ __forceinline__ Key<W> shfl_xor_key(const Key<W>& k, int off) {
    Key<W> r;
#pragma unroll
    for (int i = 0; i < 2 * W; ++i) r.k[i] = __shfl_xor_sync(kFull, k.k[i], off);
    return r;
}

// GOAL: the goal test of DESIGN.md §K9 against G -- a root in the set is a hit at depth 0, and a generated
// child in the set ends the search like a solving child, after the length-2 test (the solve wins on the same
// child) and before the visited test
template <int W, bool GOAL>
__global__ void __launch_bounds__(32) greedy_kernel(const GreedyArgs A, const GoalView G) {
    const int sidx = blockIdx.x;
    if (sidx >= A.n_search) return;
    if (A.fallback_only && A.rec[sidx].status != 99) return;
    const int lane = threadIdx.x;
    uint64_t* keys = A.keys + (uint64_t)sidx * A.cap * 2 * W;
    uint64_t* parent = A.parent + (uint64_t)sidx * A.cap;
    uint32_t* depth = A.depth + (uint64_t)sidx * A.cap;
    uint64_t* heap = A.heap + (uint64_t)sidx * A.cap;
    uint64_t* table = A.table + (uint64_t)sidx * A.tcap;
    const uint64_t tmask = A.tcap - 1;
    GreedyRec* rec = A.rec + sidx;

    // ---- root ----
    Key<W> root;
#pragma unroll
    for (int i = 0; i < 2 * W; ++i) root.k[i] = A.roots[(uint64_t)sidx * 2 * W + i];
    const int L0 = key_total_len<W>(root);
    if (lane == 0) {
        store_key<W>(keys, 0, root);
        parent[0] = kNone;
        depth[0] = 0;
        const uint64_t h = key_hash<W>(root);
        table[h & tmask] = ((h >> 40) << 40) | 1ull;
        heap[0] = ((uint64_t)((uint32_t)L0 << 24)) << 32;
    }
    __syncwarp();
    uint64_t n_nodes = 1, hn = 1, n_expanded = 0, n_moves = 0;
    int min_len = L0, n_minlen = 0;
    int solved = 0, status = 0, budget_hit = 0;
    uint64_t cur = 0;
    int final_action = 11, final_len = L0;
    int64_t goal_entry = -1;
    if constexpr (GOAL) {
        goal_entry = goal_find<W>(G, root);
        if (goal_entry >= 0) {  // path [(-1, L0)]: nothing expanded
            solved = 1;
            final_action = -1;
        }
    }

    while (hn > 0 && !(GOAL && solved)) {
        // ================= pop the minimum =================
        const uint64_t top = __ldcg(&heap[0]);
        cur = top & 0xFFFFFFFFull;
        const uint32_t cur_depth = (uint32_t)(top >> 32) & 0xFFFFFFu;
        --hn;
        if (hn > 0) {
            const uint64_t last = __ldcg(&heap[hn]);
            const Key<W> lastkey = load_key_cg<W>(keys, last & 0xFFFFFFFFull);
            uint64_t i = 0;
            for (;;) {
                const uint64_t c0 = kHeapArity * i + 1;
                if (c0 >= hn) break;
                const uint64_t ci = c0 + lane;
                uint64_t e = ~0ull;
                Key<W> k;
#pragma unroll
                for (int t = 0; t < 2 * W; ++t) k.k[t] = 0;
                if (ci < hn) {
                    e = __ldcg(&heap[ci]);
                    k = load_key_cg<W>(keys, e & 0xFFFFFFFFull);
                }
                int best = lane;
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {  // butterfly tournament: all lanes get the min
                    const uint64_t oe = __shfl_xor_sync(kFull, e, off);
                    const Key<W> ok = shfl_xor_key<W>(k, off);
                    const int ob = __shfl_xor_sync(kFull, best, off);
                    const bool take = (oe != ~0ull) && (e == ~0ull || entry_less<W>(oe, ok, e, k));
                    if (take) {
                        e = oe;
                        k = ok;
                        best = ob;
                    }
                }
                if (!entry_less<W>(e, k, last, lastkey)) break;
                if (lane == 0) __stcg(&heap[i], e);
                i = c0 + best;
            }
            if (lane == 0) __stcg(&heap[i], last);
            __syncwarp();
        }
        ++n_expanded;

        // ================= expand: lanes 0..11 =================
        const Key<W> pk = load_key_cg<W>(keys, cur);
        Key<W> child = pk;
        int st = ST_OK, L = 0;
        if (lane < 12) {
            Rel<2 * W> r0, r1;
            split_key<W>(pk, r0, r1);
            bool co;
            st = cur ? apply_move<2 * W, true>(r0, r1, lane, A.mrl, A.cyclical != 0, co)
                     : apply_move<2 * W, false>(r0, r1, lane, A.mrl, A.cyclical != 0, co);
            child = make_key<W>(r0, r1);
            L = r0.len + r1.len;
        }
        const unsigned err_mask = __ballot_sync(kFull, lane < 12 && st != ST_OK);
        const unsigned sol_mask = __ballot_sync(kFull, lane < 12 && st == ST_OK && L == 2);
        // every OK child is looked up: a visited or duplicate child is never the first goal, so the extra
        // lookups cannot change the outcome
        int64_t ge = -1;
        if (GOAL && lane < 12 && st == ST_OK) ge = goal_find<W>(G, child);
        const unsigned goal_mask = GOAL ? __ballot_sync(kFull, ge >= 0) : 0u;
        const unsigned ev_mask = err_mask | sol_mask | goal_mask;
        const int first_event = ev_mask ? (__ffs(ev_mask) - 1) : 12;
        const bool ev_solved = first_event < 12 && ((sol_mask >> first_event) & 1u);  // the solve wins on the same child
        const bool ev_goal = GOAL && first_event < 12 && !ev_solved && ((goal_mask >> first_event) & 1u);
        const bool ev_error = first_event < 12 && !ev_solved && !ev_goal;
        // children the reference evaluates: actions 0..first_event (the raising one has no length)
        const int n_eval = ev_error ? first_event : min(first_event + 1, 12);
        n_moves += (uint64_t)min(first_event + 1, 12);

        // "New minimal length found" in action order (greedy.py:82-85)
        {
            int pm = lane < n_eval ? L : 0x7FFFFFFF;
#pragma unroll
            for (int off = 1; off < 16; off <<= 1) {
                const int t = __shfl_up_sync(kFull, pm, off);
                if (lane >= off) pm = min(pm, t);
            }
            int excl = __shfl_up_sync(kFull, pm, 1);
            if (lane == 0) excl = 0x7FFFFFFF;
            const bool ev = lane < n_eval && L < min(min_len, excl);
            unsigned evm = __ballot_sync(kFull, ev);
            while (evm) {
                const int b = __ffs(evm) - 1;
                evm &= evm - 1;
                const int v = __shfl_sync(kFull, L, b);
                if (lane == 0 && n_minlen < 128) rec->minlen_log[n_minlen] = v;
                ++n_minlen;
            }
            const int allmin = __shfl_sync(kFull, pm, 15);  // prefix min over lanes 0..15 (>= 12 are +inf)
            min_len = min(min_len, allmin);
        }
        final_len = __shfl_sync(kFull, L, 11);
        if (ev_error) {
            status = __shfl_sync(kFull, st, first_event);
            break;
        }

        // ================= dedup + insert (children before the event) =================
        const uint64_t h = key_hash<W>(child);
        const uint64_t fp = h >> 40;
        uint64_t s = h & tmask;
        bool pending = lane < first_event && !key_eq<W>(child, pk);
        bool is_new = false;
        if (lane < 12) store_key<W>(keys, n_nodes + lane, child);  // tentative key storage for compares
        __syncwarp();
        while (__any_sync(kFull, pending)) {
            bool found_empty = false;
            if (pending) {
                for (;;) {
                    const uint64_t c = __ldcg(&table[s]);
                    if (c == 0) {
                        found_empty = true;
                        break;
                    }
                    if ((c >> 40) == fp) {
                        const Key<W> other = load_key_cg<W>(keys, (c & kIdxMask) - 1);
                        if (key_eq<W>(other, child)) {
                            pending = false;  // already visited (or an earlier action of this node)
                            break;
                        }
                    }
                    s = (s + 1) & tmask;
                }
            }
            // two lanes on the same empty slot: the lower action takes it, the other re-probes
            bool lose = false;
#pragma unroll
            for (int b = 0; b < 12; ++b) {
                const uint64_t sb = __shfl_sync(kFull, s, b);
                const bool fb = __shfl_sync(kFull, (int)found_empty, b) != 0;
                if (b < lane && fb && sb == s) lose = true;
            }
            if (found_empty && !lose) {
                __stcg(&table[s], (fp << 40) | (n_nodes + lane + 1));
                is_new = true;
                pending = false;
            }
            __syncwarp();
        }
        const unsigned new_mask = __ballot_sync(kFull, is_new);
        const int rank = __popc(new_mask & ((1u << lane) - 1u));
        const int n_new = __popc(new_mask);
        __syncwarp();
        if (is_new) {  // final numbering in action order == the reference's insertion order
            const uint64_t idx = n_nodes + rank;
            store_key<W>(keys, idx, child);
            parent[idx] = (cur << 4) | (uint64_t)lane;
            depth[idx] = cur_depth + 1;
            __stcg(&table[s], (fp << 40) | (idx + 1));
        }
        __syncwarp();

        // ================= push the new nodes =================
        for (unsigned m = new_mask; m; m &= m - 1) {
            const int b = __ffs(m) - 1;
            const Key<W> nk = shfl_key<W>(child, b);
            const int nL = __shfl_sync(kFull, L, b);
            const int nr = __shfl_sync(kFull, rank, b);
            const uint64_t ne = ((uint64_t)(((uint32_t)nL << 24) | (cur_depth + 1)) << 32) | (n_nodes + nr);
            uint64_t i = hn;
            while (i > 0) {
                const uint64_t p = (i - 1) / kHeapArity;
                const uint64_t pe = __ldcg(&heap[p]);
                const Key<W> pkey = load_key_cg<W>(keys, pe & 0xFFFFFFFFull);
                if (!entry_less<W>(ne, nk, pe, pkey)) break;
                if (lane == 0) __stcg(&heap[i], pe);
                i = p;
            }
            if (lane == 0) __stcg(&heap[i], ne);
            ++hn;
            __syncwarp();
        }
        n_nodes += n_new;

        if (ev_solved) {
            solved = 1;
            final_action = first_event;
            final_len = 2;
            break;
        }
        if (GOAL && ev_goal) {
            solved = 1;
            final_action = first_event;
            final_len = __shfl_sync(kFull, L, first_event);
            goal_entry = __shfl_sync(kFull, ge, first_event);
            break;
        }
        if (n_nodes >= A.budget) {  // greedy.py:115-119, after all 12 children
            budget_hit = 1;
            break;
        }
    }
    if (lane == 0) {
        rec->solved = solved;
        rec->status = status;
        rec->budget_hit = budget_hit;
        rec->n_minlen = min(n_minlen, 128);
        rec->n_nodes = n_nodes;
        rec->n_expanded = n_expanded;
        rec->n_moves = n_moves;
        rec->heap_left = hn;
        rec->final_node = cur;
        rec->final_action = solved ? final_action : 11;
        rec->final_len = final_len;
        rec->rounds = 0;
        rec->engine = 2;
        if constexpr (GOAL) rec->goal = goal_entry;
    }
}

}  // namespace acs
#include "greedy_bucket.cuh"
namespace acs {

// path of every search: chain of its final node, then (final_action, final_len) -- nothing more when the
// search stopped at its root (a root in the goal set, final_action -1)
template <int W>
__global__ void greedy_path_kernel(const GreedyArgs A, int32_t* paths, int path_cap, int32_t* path_len) {
    const int sidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (sidx >= A.n_search) return;
    const uint64_t* keys = A.keys + (uint64_t)sidx * A.cap * 2 * W;
    const uint64_t* parent = A.parent + (uint64_t)sidx * A.cap;
    const GreedyRec& rec = A.rec[sidx];
    int32_t* path = paths + (size_t)sidx * path_cap * 2;
    int d = 0;
    for (uint64_t q = rec.final_node;; q = parent[q] >> 4) {
        ++d;
        if (parent[q] == kNone) break;
    }
    const bool at_root = rec.final_action < 0;
    path_len[sidx] = d + (at_root ? 0 : 1);
    int pos = d - 1;
    for (uint64_t q = rec.final_node;; q = parent[q] >> 4, --pos) {
        const Key<W> k = load_key<W>(keys, q);
        const bool root = parent[q] == kNone;
        if (pos < path_cap) {
            path[2 * pos] = root ? -1 : (int)(parent[q] & 15);
            path[2 * pos + 1] = key_total_len<W>(k);
        }
        if (root) break;
    }
    if (!at_root && d < path_cap) {
        path[2 * d] = rec.final_action;
        path[2 * d + 1] = rec.final_len;
    }
}

// the element of every goal hit: u with u.(the state the search stopped at) = the entry's state (the identity
// for an exact set), or -1 for a search that did not stop at a goal
template <int W>
__global__ void greedy_goal_elem_kernel(const GreedyArgs A, int symmetric, int32_t* out) {
    const int sidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (sidx >= A.n_search) return;
    const GreedyRec& rec = A.rec[sidx];
    if (rec.goal < 0) {
        out[sidx] = -1;
        return;
    }
    Key<W> q = load_key<W>(A.keys + (uint64_t)sidx * A.cap * 2 * W, rec.final_node);
    if (rec.final_action >= 0) {
        Rel<2 * W> r0, r1;
        split_key<W>(q, r0, r1);
        bool co;
        apply_move<2 * W, false>(r0, r1, rec.final_action, A.mrl, A.cyclical != 0, co);
        q = make_key<W>(r0, r1);
    }
    int u = 0;
    if (symmetric) canonical<W>(q, u);
    out[sidx] = u;
}

}  // namespace acs

// ---------------------------------------------------------------------------------------
using namespace acs;

struct acs_greedy {
    int device = 0, mrl = 0, W = 1, cyclical = 0, n_search = 0;
    int64_t budget = 0;
    uint64_t cap = 0, tcap = 0;
    uint64_t *keys = nullptr, *parent = nullptr, *heap = nullptr, *table = nullptr, *roots = nullptr;
    uint32_t* depth = nullptr;
    GreedyRec* rec = nullptr;
    GbArgs gb{};  // pools of the bucket kernel
    bool use_bucket = true;
    int n_fallback = 0;
    int32_t *d_paths = nullptr, *d_path_len = nullptr, *d_goal_g = nullptr;
    int path_cap = 0;
    std::vector<int32_t> h_goal_g;  // greedy_goal_elem_kernel of the last run with goals
    std::vector<GreedyRec> h_rec;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    const acs_goalset* goals = nullptr;  // acs_greedy_set_goals
    bool ran = false, ran_with_goals = false;
};

extern "C" void acs_greedy_destroy(acs_greedy* g) {
    if (!g) return;
    cudaSetDevice(g->device);
    if (g->stream) {
        cudaStreamSynchronize(g->stream);
        cudaStreamDestroy(g->stream);
    }
    if (g->ev0) cudaEventDestroy(g->ev0);
    if (g->ev1) cudaEventDestroy(g->ev1);
    cudaFree(g->keys);
    cudaFree(g->parent);
    cudaFree(g->heap);
    cudaFree(g->table);
    cudaFree(g->roots);
    cudaFree(g->depth);
    cudaFree(g->rec);
    cudaFree(g->gb.segs);
    cudaFree(g->gb.sortbuf);
    cudaFree(g->gb.cand_key);
    cudaFree(g->gb.cand_meta);
    cudaFree(g->gb.cand_slot);
    cudaFree(g->gb.round_tab);
    cudaFree(g->d_paths);
    cudaFree(g->d_path_len);
    cudaFree(g->d_goal_g);
    delete g;
}

extern "C" int acs_greedy_create(int device, int n_search, int mrl, int64_t max_nodes, int cyclical, int path_cap,
                                 acs_greedy** out) {
    if (!out) return ACS_ERR_INVALID;
    *out = nullptr;
    if (const int rc = check_key_mrl(mrl, "greedy")) return rc;
    if (n_search < 1 || max_nodes < 0 || path_cap < 2 || max_nodes > (1ll << 24) - 32)
        return fail(ACS_ERR_INVALID, "greedy: need n_search >= 1, 0 <= max_nodes < 2^24 - 32, path_cap >= 2");
    if (const int rc = open_device(device, "greedy")) return rc;
    acs_greedy* g = new acs_greedy();
    g->device = device;
    g->mrl = mrl;
    g->W = key_words(mrl);
    g->cyclical = cyclical ? 1 : 0;
    g->n_search = n_search;
    g->budget = max_nodes;
    g->cap = (uint64_t)max_nodes + 16;  // overshoot <= 11, + 12 tentative key slots
    uint64_t t = 64;
    while (t < 2 * g->cap) t <<= 1;
    g->tcap = t;
    g->path_cap = path_cap;
    const uint64_t S = (uint64_t)n_search;
    ACS_ALLOC(g->keys, S * g->cap * 2 * g->W * sizeof(uint64_t), acs_greedy_destroy(g));
    ACS_ALLOC(g->parent, S * g->cap * sizeof(uint64_t), acs_greedy_destroy(g));
    ACS_ALLOC(g->depth, S * g->cap * sizeof(uint32_t), acs_greedy_destroy(g));
    ACS_ALLOC(g->heap, S * g->cap * sizeof(uint64_t), acs_greedy_destroy(g));
    ACS_ALLOC(g->table, S * g->tcap * sizeof(uint64_t), acs_greedy_destroy(g));
    ACS_ALLOC(g->roots, S * 2 * g->W * sizeof(uint64_t), acs_greedy_destroy(g));
    ACS_ALLOC(g->rec, S * sizeof(GreedyRec), acs_greedy_destroy(g));
    ACS_ALLOC(g->d_paths, S * (size_t)path_cap * 2 * sizeof(int32_t), acs_greedy_destroy(g));
    ACS_ALLOC(g->d_path_len, S * sizeof(int32_t), acs_greedy_destroy(g));
    {
        const char* e = std::getenv("ACS_GREEDY_KERNEL");  // "heap" forces the one-warp-per-search kernel
        g->use_bucket = !(e && std::string(e) == "heap");
    }
    if (g->use_bucket) {
        ACS_ALLOC(g->gb.segs, S * (size_t)kGbSegPool * sizeof(GbSeg), acs_greedy_destroy(g));
        ACS_ALLOC(g->gb.sortbuf, S * (size_t)kGbSortCap * gb_rec_words(g->W) * sizeof(uint64_t), acs_greedy_destroy(g));
        ACS_ALLOC(g->gb.cand_key, S * (size_t)kGbCand * 2 * g->W * sizeof(uint64_t), acs_greedy_destroy(g));
        ACS_ALLOC(g->gb.cand_meta, S * (size_t)kGbCand * sizeof(uint32_t), acs_greedy_destroy(g));
        ACS_ALLOC(g->gb.cand_slot, S * (size_t)kGbCand * sizeof(uint32_t), acs_greedy_destroy(g));
        ACS_ALLOC(g->gb.round_tab, S * (size_t)kGbRoundSlots * sizeof(uint64_t), acs_greedy_destroy(g));
        g->gb.frontier = reinterpret_cast<uint32_t*>(g->heap);  // the heap pool doubles as the frontier array
        g->gb.fcap = 2 * g->cap;
    }
    g->h_rec.resize(S);
    if (cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking) != cudaSuccess) {
        acs_greedy_destroy(g);
        return ACS_ERR_CUDA;
    }
    cudaEventCreate(&g->ev0);
    cudaEventCreate(&g->ev1);
    *out = g;
    return ACS_OK;
}

namespace {

template <int W, bool GOAL>
int greedy_run_impl(acs_greedy* g, const int8_t* h_pres, int32_t* h_paths, acs_search_result* res) {
    ACS_CUDA(cudaSetDevice(g->device));
    const int S = g->n_search;
    std::vector<uint64_t> roots((size_t)S * 2 * W);
    bool padded = true;
    for (int s = 0; s < S; ++s) {
        Key<W> k;
        int lens[2];
        // a mis-padded root cannot be represented; empty relators can (the first move raises)
        const RootCheck rc = pack_root<W>(h_pres + (size_t)s * 2 * g->mrl, g->mrl, k, lens);
        if (rc == RootCheck::bad_letter)
            return fail(ACS_ERR_UNSUPPORTED, "greedy: letters outside {+-1,+-2} are not supported by the packed search");
        padded = padded && rc != RootCheck::not_padded;
        std::memcpy(&roots[(size_t)s * 2 * W], k.k, sizeof(k.k));
    }
    if (!padded) return fail(ACS_ERR_INVALID, "greedy: presentation is not zero right-padded");
    cudaStream_t st = g->stream;
    ACS_CUDA(cudaMemcpyAsync(g->roots, roots.data(), roots.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    ACS_CUDA(cudaMemsetAsync(g->table, 0, (size_t)S * g->tcap * sizeof(uint64_t), st));
    GreedyArgs A{};
    A.keys = g->keys;
    A.parent = g->parent;
    A.depth = g->depth;
    A.heap = g->heap;
    A.table = g->table;
    A.roots = g->roots;
    A.rec = g->rec;
    A.cap = g->cap;
    A.tcap = g->tcap;
    A.budget = (uint64_t)g->budget;
    A.n_search = S;
    A.mrl = g->mrl;
    A.cyclical = g->cyclical;
    A.fallback_only = 0;
    const GoalView G = GOAL ? g->goals->view() : GoalView{nullptr, nullptr, 0};
    ACS_CUDA(cudaEventRecord(g->ev0, st));
    g->n_fallback = 0;
    if (g->use_bucket) {
        // pass 1: small bucket directory (several CTAs per SM); pass 2: the searches that outgrew it, with a
        // large directory (one CTA per SM); whatever still does not fit is re-run by the heap kernel
        // with goals, the goal slot follows the bucket directory
        auto smem_for = [](int buckets) {
            return ((sizeof(GbShared) + 15) / 16) * 16 + (size_t)buckets * sizeof(GbBucket) + (GOAL ? kGbGoalSmem : 0);
        };
        ACS_CUDA(cudaFuncSetAttribute(greedy_bucket_kernel<W, GOAL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem_for(kGbBuckets2)));
        // several CTAs per SM in pass 1: ask for the largest shared-memory carve-out
        ACS_CUDA(cudaFuncSetAttribute(greedy_bucket_kernel<W, GOAL>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                     (int)cudaSharedmemCarveoutMaxShared));
        const bool debug = std::getenv("ACS_GREEDY_DEBUG") != nullptr;
        for (int pass = 0; pass < 2; ++pass) {
            g->gb.max_buckets = pass == 0 ? kGbBuckets1 : kGbBuckets2;
            g->gb.retry_only = pass;
            cudaEvent_t e0 = pass == 0 ? g->ev0 : g->ev1;
            if (pass) ACS_CUDA(cudaEventRecord(e0, st));
            greedy_bucket_kernel<W, GOAL><<<S, kGbThreads, smem_for(g->gb.max_buckets), st>>>(A, g->gb, G);
            ACS_CUDA(cudaGetLastError());
            ACS_CUDA(cudaMemcpyAsync(g->h_rec.data(), g->rec, (size_t)S * sizeof(GreedyRec), cudaMemcpyDeviceToHost, st));
            ACS_CUDA(cudaStreamSynchronize(st));
            g->n_fallback = 0;
            for (int s = 0; s < S; ++s)
                if (g->h_rec[s].status == kGbFallback) {
                    ++g->n_fallback;
                    if (debug)
                        std::fprintf(stderr, "greedy: pass %d, search %d handed back (reason %d, %llu nodes)\n", pass, s,
                                     -g->h_rec[s].rounds, (unsigned long long)g->h_rec[s].n_nodes);
                    ACS_CUDA(cudaMemsetAsync(g->table + (size_t)s * g->tcap, 0, g->tcap * sizeof(uint64_t), st));
                }
            if (debug) std::fprintf(stderr, "greedy: bucket pass %d, %d searches, mrl %d: %d handed back\n", pass, S, g->mrl, g->n_fallback);
            if (!g->n_fallback) break;
        }
        if (g->n_fallback) {
            A.fallback_only = 1;
            greedy_kernel<W, GOAL><<<S, 32, 0, st>>>(A, G);
            ACS_CUDA(cudaGetLastError());
        }
    } else {
        greedy_kernel<W, GOAL><<<S, 32, 0, st>>>(A, G);
        ACS_CUDA(cudaGetLastError());
    }
    greedy_path_kernel<W><<<(S + 63) / 64, 64, 0, st>>>(A, g->d_paths, g->path_cap, g->d_path_len);
    ACS_CUDA(cudaGetLastError());
    ACS_CUDA(cudaEventRecord(g->ev1, st));
    if (GOAL) {
        if (!g->d_goal_g) ACS_CUDA(cudaMalloc((void**)&g->d_goal_g, (size_t)S * sizeof(int32_t)));
        greedy_goal_elem_kernel<W><<<(S + 63) / 64, 64, 0, st>>>(A, g->goals->symmetric, g->d_goal_g);
        ACS_CUDA(cudaGetLastError());
        g->h_goal_g.resize((size_t)S);
        ACS_CUDA(cudaMemcpyAsync(g->h_goal_g.data(), g->d_goal_g, (size_t)S * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    }
    ACS_CUDA(cudaMemcpyAsync(g->h_rec.data(), g->rec, (size_t)S * sizeof(GreedyRec), cudaMemcpyDeviceToHost, st));
    std::vector<int32_t> plen(S);
    ACS_CUDA(cudaMemcpyAsync(plen.data(), g->d_path_len, (size_t)S * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (h_paths)
        ACS_CUDA(cudaMemcpyAsync(h_paths, g->d_paths, (size_t)S * g->path_cap * 2 * sizeof(int32_t),
                                cudaMemcpyDeviceToHost, st));
    ACS_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, g->ev0, g->ev1);
    g->ran = true;
    g->ran_with_goals = GOAL;
    for (int s = 0; s < S; ++s) {
        const GreedyRec& r = g->h_rec[s];
        acs_search_result& o = res[s];
        std::memset(&o, 0, sizeof(o));
        o.solved = r.solved;
        o.status = r.status;
        o.budget_hit = r.budget_hit;
        o.path_len = r.status ? 0 : plen[s];
        o.n_visited = (int64_t)r.n_nodes;
        o.n_expanded = (int64_t)r.n_expanded;
        o.n_moves = (int64_t)r.n_moves;
        o.frontier_left = (int64_t)r.heap_left;
        o.n_levels = r.engine == 1 ? r.rounds : -1;  // bucket rounds; -1 = served by the heap kernel
        o.n_minlen = r.n_minlen;
        std::memcpy(o.minlen_log, r.minlen_log, sizeof(o.minlen_log));
        o.seconds_device = ms * 1e-3;
    }
    return ACS_OK;
}

}  // namespace

extern "C" int acs_greedy_run(acs_greedy* g, const int8_t* h_presentations, int32_t* h_paths,
                              acs_search_result* results) {
    if (!g || !h_presentations || !results) return ACS_ERR_INVALID;
    if (g->goals)
        return g->W == 1 ? greedy_run_impl<1, true>(g, h_presentations, h_paths, results)
                         : greedy_run_impl<2, true>(g, h_presentations, h_paths, results);
    return g->W == 1 ? greedy_run_impl<1, false>(g, h_presentations, h_paths, results)
                     : greedy_run_impl<2, false>(g, h_presentations, h_paths, results);
}

extern "C" int acs_greedy_visited(acs_greedy* g, int search, int8_t* h_out, int64_t cap_rows, int64_t* n_out) {
    if (!g || search < 0 || search >= g->n_search || (!h_out && cap_rows > 0)) return ACS_ERR_INVALID;
    ACS_CUDA(cudaSetDevice(g->device));
    const int64_t n = (int64_t)std::min<uint64_t>(g->h_rec[search].n_nodes, (uint64_t)std::max<int64_t>(cap_rows, 0));
    if (n_out) *n_out = n;
    return records_to_host(g->W, g->keys + (uint64_t)search * g->cap * 2 * g->W, 2 * g->W, n, g->mrl, h_out, nullptr,
                           g->stream);
}

extern "C" int acs_greedy_set_goals(acs_greedy* g, const acs_goalset* gs) {
    if (!g) return ACS_ERR_INVALID;
    if (gs) {
        if (gs->mrl != g->mrl)
            return fail(ACS_ERR_INVALID, "greedy_set_goals: the goal set's max_relator_length differs from the engine's");
        if (gs->cyclical != g->cyclical)
            return fail(ACS_ERR_INVALID, "greedy_set_goals: the goal set's cyclical flag differs from the engine's");
        if (gs->device != g->device) return fail(ACS_ERR_INVALID, "greedy_set_goals: the goal set lives on another device");
        if (gs->n_entries >= (int64_t)0xFFFFFFFF)  // the bucket kernel packs a hit's entry into 32 bits beside its candidate
            return fail(ACS_ERR_UNSUPPORTED, "greedy_set_goals: goal sets of 2^32 - 1 entries or more are not supported");
    }
    g->goals = gs;
    return ACS_OK;
}

extern "C" int acs_greedy_goal_hit_elements(acs_greedy* g, int32_t* h_elem) {
    if (!g || !h_elem) return ACS_ERR_INVALID;
    if (!g->ran) return fail(ACS_ERR_INVALID, "greedy: no completed run");
    for (int s = 0; s < g->n_search; ++s) h_elem[s] = g->ran_with_goals ? g->h_goal_g[s] : -1;
    return ACS_OK;
}

extern "C" int acs_greedy_goal_hits(acs_greedy* g, int64_t* h_entry) {
    if (!g || !h_entry) return ACS_ERR_INVALID;
    if (!g->ran) return fail(ACS_ERR_INVALID, "greedy: no completed run");
    for (int s = 0; s < g->n_search; ++s) h_entry[s] = g->ran_with_goals ? g->h_rec[s].goal : -1;
    return ACS_OK;
}
