// mbfs.cu -- batched breadth-first search: many independent searches of one max_relator_length
// and one `cyclical` flag advance together through the same kernel launches on one GPU.
//
// Contract: for every search, the result equals acs_bfs_run on that presentation (pbfs.cu, and so
// the reference's ac_solver/search/breadth_first.py:15-97): solved flag and path, counters,
// budget cut, raising row, "New minimal length" sequence and the visited array in FIFO order.
//
// Design.  Search s owns a slab of budget_s + 16 nodes (the reference overshoots its budget by at
// most 11: the test runs after a parent's 12 children), so a node's slab index is its FIFO id and
// parent links stay inside the slab.  A combined chunk concatenates one segment per active search:
// segment k covers parents [head_k, head_k + F_k) of search seg_search[k] (within its current
// level) at chunk offset off_k, and a child gets the candidate id c = 12*(off_k + gid - head_k) + a.
// Within a search that is the reference's order; across searches the (search, state) keys differ,
// so "smallest candidate id wins per (search, state)" is exact.  One chunk is
//
//   prep     reset the bitmap, the record cursor and the per-segment control minima
//   expand   one thread per parent, children appended to the chunk's record log (key, c, search)
//   insert   one shared exact open-addressing table keyed by (search, state): 32-byte buckets,
//            tentative slots point at log records, smallest c wins by CAS, XOR winner bitmap
//   scan     popcount prefix of the winner bitmap -> rank table
//   decide   one thread per segment: budget cut by binary search, solving / raising child,
//            minimal-length log, counters; a search that ends drops out
//   commit   winners below their segment's limit become nodes of their slab and their table slot
//            is re-pointed at the node; winners past the limit leave a tombstone
//   plan     next chunk: the active searches' level remainders, in search order, up to the
//            parents cap and the table's free room
//
// Table slots are fingerprint << 40 | tag | (index + 1): the tag bit 39 set means a committed node
// (global node index), clear a record of the current chunk's log.  The log is rewritten every
// chunk, so its size is bounded by 12 records per parent of one chunk.  The host enqueues chunks
// ahead of the device and reads only a lagging pinned copy of the run state.
//
// Orbit search (acs_bfs_batch_set_symmetric): the same engine over canonical states (ac_sym.cuh).  The
// root is stored as its canonical form, a child is canonicalized right after it is packed, and it is new
// when its canonical form is unseen.  Every node records the element g with stored = g.(generated state)
// in bits 32..35 of its search word; the path kernel turns the canonical-frame moves into moves of the
// input row.  The move-skip rule is off in this mode: its argument is about generated, not canonical, states.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "ac_core.cuh"
#include "ac_keys.cuh"
#include "ac_sym.cuh"
#include "acs_internal.h"
#include "bfs_common.cuh"
#include "goalset.cuh"
#include "mb_engine.cuh"

namespace acs {

// ---- plan: the next chunk's segments (one warp) --------------------------------------------------
__global__ void __launch_bounds__(32) mb_plan_kernel(const MbEngine E, int first) {
    MbState* st = E.st;
    if (st->done) return;
    const int lane = threadIdx.x;
    const int n = st->n_search;
    int64_t P = st->chunk_cap;
    if (first) {
        P = (int64_t)n;  // the roots, expanded without the normal-form shortcuts
    } else {
        // no room: more than 3/4 of the table holds nodes and tombstones -- stop with an error rather
        // than crawl on in tiny chunks
        const int64_t room = ((int64_t)(3 * ((st->tmask + 1) / 4)) - st->used) / 12;
        if (room < 1) {
            if (lane == 0) {
                atomicOr(&st->ierr, MB_IERR_TABLE_FULL);
                st->done = 1;
            }
            return;
        }
        P = room < P ? room : P;
    }
    const uint32_t lt = (1u << lane) - 1u;
    int64_t carryD = 0;
    int carryK = 0;
    for (int base = 0; base < n; base += 32) {
        const int s = base + lane;
        int64_t d = 0, head = 0;
        if (s < n && !E.srch[s].done) {
            const MbSearch& M = E.srch[s];
            head = M.head;
            // a third of the remaining budget at most: a search ends inside its last segment, and the winners
            // past its end stay in the table as tombstones; ~2.8 new states per parent keep them few
            const int64_t r = (M.budget - M.n_nodes) / 3 + 1;
            d = M.level_end - head;
            d = d < r ? d : r;
            d = d < P ? d : P;
        }
        int64_t x = d;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xFFFFFFFFu, x, o);
            if (lane >= o) x += t;
        }
        const int64_t D = carryD + x - d;
        const bool on = d > 0 && D < P;
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, on);
        if (on) {
            const int k = carryK + __popc(b & lt);
            E.seg_search[k] = s;
            E.seg_head[k] = head;
            E.seg_off[k] = D;
            E.seg_of[s] = k;
        }
        carryD += __shfl_sync(0xFFFFFFFFu, x, 31);
        carryK += __popc(b);
        if (carryD >= P) break;
    }
    if (lane == 0) {
        const int64_t F = carryD < P ? carryD : P;
        E.seg_off[carryK] = F;
        st->n_seg = carryK;
        st->Ftot = F;
        if (carryK == 0) st->done = 1;
    }
}

// ---- prep ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mb_prep_kernel(const MbEngine E) {
    const MbState* st = E.st;
    if (st->done) return;
    const int64_t nwords = (12 * st->Ftot + 31) / 32;
    const int64_t nctrl = st->n_seg * kMbCtrl;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += stride) E.bitmap[i] = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nctrl; i += stride) E.ctrl[i] = ~0ull;
    if (blockIdx.x == 0 && threadIdx.x == 0) *E.cursor = 0;
}


// ---- insert ----------------------------------------------------------------------------------------
template <int W>
__global__ void __launch_bounds__(256) mb_insert_kernel(const MbEngine E) {
    MbState* st = E.st;
    if (st->done) return;
    const unsigned long long n = *E.cursor;
    const uint64_t tmask = st->tmask;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const Key<W> key = load_key_cg<W>(E.log_keys, i);
        const uint32_t c = __ldcg(E.log_c + i), s = __ldcg(E.log_s + i);
        const uint64_t h = mb_hash<W>(key, s);
        const uint64_t fp23 = h >> 41;
        const uint64_t mine = (fp23 << 40) | (i + 1);
        uint64_t slot_base = (h & tmask) & ~3ull;
        uint64_t probes = 0;
        bool finished = false;
        while (!finished) {
            uint64_t vv[4];
            load_bucket(E.table + slot_base, vv);
#pragma unroll
            for (int jj = 0; jj < 4 && !finished; ++jj) {
                uint64_t cur = vv[jj];
                const uint64_t slot = slot_base + jj;
                unsigned long long* sp = (unsigned long long*)&E.table[slot];
                if (cur == 0) {
                    cur = atomicCAS(sp, 0ull, (unsigned long long)mine);
                    if (cur == 0) {  // first sighting of this (search, state): claim
                        E.rec_slot[i] = slot;
                        atomicXor(&E.bitmap[c >> 5], 1u << (c & 31));
                        finished = true;
                        break;
                    }
                }
                if ((cur >> 40) != fp23) continue;
                if (cur & kMbNode) {  // a committed node: visited if it is this search's state
                    Key<W> other;
                    int64_t pl, s2;
                    node_load<W>(E.nodes, (cur & kMbIdx) - 1, other, pl, s2);
                    if ((uint32_t)s2 != s || !key_eq<W>(other, key)) continue;
                    finished = true;
                    break;
                }
                uint64_t p2 = (cur & kMbIdx) - 1;
                if (__ldcg(E.log_s + p2) != s || !key_eq<W>(load_key_cg<W>(E.log_keys, p2), key)) continue;
                // a record of this chunk with the same (search, state): the smaller candidate id keeps the slot
                for (;;) {
                    const uint32_t c2 = __ldcg(E.log_c + p2);
                    if (c2 < c) break;
                    const uint64_t old = atomicCAS(sp, (unsigned long long)cur, (unsigned long long)mine);
                    if (old == cur) {  // displaced the holder: its claim bit flips back, mine flips on
                        E.rec_slot[i] = slot;
                        atomicXor(&E.bitmap[c2 >> 5], 1u << (c2 & 31));
                        atomicXor(&E.bitmap[c >> 5], 1u << (c & 31));
                        break;
                    }
                    cur = old;  // someone else replaced it meanwhile (same state): look again
                    p2 = (cur & kMbIdx) - 1;
                }
                finished = true;
            }
            if (!finished) {
                slot_base = (slot_base + 4) & tmask;
                probes += 4;
                if (probes > tmask) {  // cannot happen with the chunk sizing (table <= 3/4 full)
                    atomicOr(&st->ierr, MB_IERR_TABLE_FULL);
                    finished = true;
                }
            }
        }
    }
}


// ---- scan --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kScanT) mb_scan_sums_kernel(const MbEngine E) {
    const MbState* st = E.st;
    if (st->done) return;
    const int64_t nwords = (12 * st->Ftot + 31) / 32;
    const int64_t nblk = (nwords + kScanBlock - 1) / kScanBlock;
    for (int64_t b = blockIdx.x; b < nblk; b += gridDim.x) {
        uint32_t v = 0;
#pragma unroll
        for (int k = 0; k < kScanPer; ++k) {
            const int64_t i = b * kScanBlock + (int64_t)k * kScanT + threadIdx.x;
            if (i < nwords) v += __popc(__ldcg(E.bitmap + i));
        }
        uint32_t tot;
        block_excl_scan(v, tot);
        if (threadIdx.x == 0) E.bsums[b] = tot;
        __syncthreads();
    }
}
// single block: exclusive scan of the block sums in place; total to the sentinel rank-table entry
__global__ void __launch_bounds__(kScanT) mb_scan_top_kernel(const MbEngine E) {
    const MbState* st = E.st;
    if (st->done) return;
    const int64_t nwords = (12 * st->Ftot + 31) / 32;
    const int64_t nblk = (nwords + kScanBlock - 1) / kScanBlock;
    uint32_t carry = 0;
    for (int64_t base = 0; base < nblk; base += kScanT) {
        const int64_t i = base + threadIdx.x;
        const uint32_t v = i < nblk ? __ldcg(E.bsums + i) : 0u;
        uint32_t total;
        const uint32_t ex = block_excl_scan(v, total);
        if (i < nblk) E.bsums[i] = carry + ex;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) E.rt[nwords] = make_uint2(carry, 0u);
}
__global__ void __launch_bounds__(kScanT) mb_scan_final_kernel(const MbEngine E) {
    const MbState* st = E.st;
    if (st->done) return;
    const int64_t nwords = (12 * st->Ftot + 31) / 32;
    const int64_t nblk = (nwords + kScanBlock - 1) / kScanBlock;
    for (int64_t b = blockIdx.x; b < nblk; b += gridDim.x) {
        const int64_t first = b * kScanBlock + (int64_t)threadIdx.x * kScanPer;
        uint32_t w[kScanPer], sum = 0;
#pragma unroll
        for (int k = 0; k < kScanPer; ++k) {
            w[k] = first + k < nwords ? __ldcg(E.bitmap + first + k) : 0u;
            sum += __popc(w[k]);
        }
        uint32_t tot;
        uint32_t r = __ldcg(E.bsums + b) + block_excl_scan(sum, tot);
#pragma unroll
        for (int k = 0; k < kScanPer; ++k) {
            if (first + k < nwords) E.rt[first + k] = make_uint2(r, w[k]);
            r += __popc(w[k]);
        }
        __syncthreads();
    }
}

// ---- decide: one thread per segment, pbfs.cu's rules on the segment ---------------------------------
__global__ void __launch_bounds__(128) mb_decide_kernel(const MbEngine E) {
    MbState* st = E.st;
    if (st->done) return;
    const int64_t Ftot = st->Ftot;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k == 0) {  // every winner becomes a node or a tombstone
        const int64_t nwords = (12 * Ftot + 31) / 32;
        st->used += E.rt[nwords].x;
        st->chunks += 1;
    }
    if (k >= st->n_seg) return;
    const int s = E.seg_search[k];
    MbSearch& M = E.srch[s];
    const unsigned long long* red = E.ctrl + (int64_t)k * kMbCtrl;
    const uint64_t off = (uint64_t)E.seg_off[k], F = (uint64_t)E.seg_off[k + 1] - off;
    const uint64_t c0 = 12 * off, head = (uint64_t)M.head, n_nodes = (uint64_t)M.n_nodes;
    const uint64_t budget = (uint64_t)M.budget;
    const uint64_t r0 = mb_rank(E.rt, c0);
    const uint64_t total = mb_rank(E.rt, c0 + 12 * F) - r0;
    uint64_t limit = 12 * F;
    bool cut = false;
    uint64_t cut_p = 0;
    if (n_nodes + total >= budget) {
        // first segment-local parent p with n_nodes + #winners(parents <= p) >= budget (monotone in p)
        uint64_t lo = 0, hi = F - 1;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (n_nodes + mb_rank(E.rt, c0 + (mid + 1) * 12) - r0 >= budget) hi = mid;
            else lo = mid + 1;
        }
        cut = true;
        cut_p = lo;
        if (12 * (cut_p + 1) < limit) limit = 12 * (cut_p + 1);
    }
    const unsigned long long sol = st->explore ? ~0ull : red[kMbSol], err = red[kMbErr], goal = red[kMbGoal];
    bool sol_here = false, goal_here = false;
    int status = 0;
    uint64_t sol_l = 0, err_l = 0;
    if (sol != ~0ull && sol - c0 < limit) {  // solved at or before the cut parent
        sol_l = sol - c0;
        limit = sol_l;
        sol_here = true;
        cut = false;
    }
    if (goal != ~0ull && (goal >> 32) - c0 < limit) {  // a goal child; on the solving child itself the solve wins
        sol_l = (goal >> 32) - c0;
        limit = sol_l;
        sol_here = true;
        goal_here = true;
        cut = false;
    }
    if (err != ~0ull && (err >> 2) - c0 < limit) {  // the reference raises here, before anything later
        err_l = (err >> 2) - c0;
        limit = err_l;
        status = (int)(err & 3);
        sol_here = false;
        goal_here = false;
        cut = false;
    }
    // "New minimal length found" events in reference order
    const uint64_t c_limit = limit + (sol_here ? 1 : 0);
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
    const uint64_t cg = mb_rank(E.rt, c0 + limit) - r0;
    E.seg_limit[k] = (int64_t)(c0 + limit);
    E.seg_base[k] = M.slab + (int64_t)n_nodes - (int64_t)r0;
    if ((int64_t)(n_nodes + cg) > M.cap) atomicOr(&st->ierr, MB_IERR_SLAB_FULL);  // the commit drops the excess
    M.n_nodes = (int64_t)(n_nodes + cg);
    if (sol_here) {
        M.solved = 1;
        M.sol_gid = (int64_t)(12 * head + sol_l);
        M.n_expanded = M.sol_gid / 12 + 1;
        M.sol_len = 2;
        if (goal_here) {
            const uint64_t e = goal & 0xFFFFFFFFull;
            const int W = key_words(st->mrl);
            const uint64_t* q = E.goals.nodes + e * node_words(W);  // the goal state's key
            M.sol_len = key_len(q, W, 0) + key_len(q, W, 1);
            E.goal_hit[s] = (int64_t)e;
        }
    } else if (status) {
        M.status = status;
        M.err_code = (int64_t)(((12 * head + err_l) << 2) | (uint64_t)status);
        M.n_expanded = (int64_t)((12 * head + err_l) / 12 + 1);
    } else if (cut) {
        M.budget_hit = 1;
        M.n_expanded = (int64_t)(head + cut_p + 1);
    } else {
        M.n_expanded = (int64_t)(head + F);
    }
    M.head = (int64_t)(head + F);
    if (M.solved || M.budget_hit || M.status || M.head >= M.n_nodes) {
        M.done = 1;
    } else if (M.head == M.level_end) {
        M.level_end = M.n_nodes;
        M.levels += 1;
    }
}

// ---- commit ------------------------------------------------------------------------------------------
template <int W, bool SYM>
__global__ void __launch_bounds__(256) mb_commit_kernel(const MbEngine E) {
    const MbState* st = E.st;
    if (st->done) return;
    const unsigned long long n = *E.cursor;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t c = __ldcg(E.log_c + i);
        const uint2 e = E.rt[c >> 5];
        if (!((e.y >> (c & 31)) & 1u)) continue;  // an already visited state, or lost to an earlier candidate
        const uint32_t s = __ldcg(E.log_s + i);
        const int k = E.seg_of[s];
        const uint64_t slot = E.rec_slot[i];
        if ((int64_t)c >= E.seg_limit[k]) {  // past the end of its search
            E.table[slot] = kMbTomb;
            continue;
        }
        const int64_t idx = E.seg_base[k] + (int64_t)(e.x + __popc(e.y & ((1u << (c & 31)) - 1u)));
        const MbSearch& M = E.srch[s];
        if (idx >= M.slab + M.cap) {  // MB_IERR_SLAB_FULL was raised by decide
            E.table[slot] = kMbTomb;
            continue;
        }
        const Key<W> key = load_key_cg<W>(E.log_keys, i);
        const int64_t pgid = E.seg_head[k] + (int64_t)(c / 12) - E.seg_off[k];
        const int64_t tag = SYM ? (int64_t)s | ((int64_t)__ldcg(E.log_g + i) << 32) : (int64_t)s;
        node_store<W>(E.nodes, (uint64_t)idx, key, (pgid << 4) | (int64_t)(c % 12), tag);
        E.table[slot] = ((mb_hash<W>(key, s) >> 41) << 40) | kMbNode | (uint64_t)(idx + 1);
    }
}


// committed nodes of every search -> goal-set entries in (search, FIFO id) order; off [n_search + 1] holds
// each search's first entry, slab [n_search] its first node.  Parent links are rebased onto entry indices.
template <int W>
__global__ void mb_adopt_kernel(const uint64_t* nodes, const int64_t* off, const int64_t* slab, int n_search,
                                uint64_t* out, uint64_t n) {
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (uint64_t)gridDim.x * blockDim.x) {
        const int s = mb_segment(off, n_search, (int64_t)e);
        const int64_t first = __ldg(off + s);
        Key<W> k;
        int64_t pl, tag;
        node_load<W>(nodes, (uint64_t)(__ldg(slab + s) + ((int64_t)e - first)), k, pl, tag);
        node_store<W>(out, e, k, pl < 0 ? -1 : (((first + (pl >> 4)) << 4) | (pl & 15)), (int64_t)s | (tag & (15ll << 32)));
    }
}

}  // namespace acs

// ---------------------------------------------------------------------------------------------------------
using namespace acs;

namespace {
constexpr int kMbRing = 4, kMbLag = 2;

// sizes of an engine (shared by acs_bfs_batch_bytes and acs_bfs_batch_create)
struct MbPlan {
    int W;
    int64_t nodes, chunk, rec_cap, bitmap_words, nblk;
    uint64_t tcap;
    int64_t bytes;
};

int mb_plan(int n_search, int mrl, const int64_t* max_nodes, int64_t chunk_parents, MbPlan& P) {
    if (n_search < 1 || !max_nodes) return fail(ACS_ERR_INVALID, "bfs_batch: need at least one search");
    if (const int rc = check_key_mrl(mrl, "bfs_batch")) return rc;
    P.W = key_words(mrl);
    P.nodes = 0;
    for (int s = 0; s < n_search; ++s) {
        if (max_nodes[s] < 0) return fail(ACS_ERR_INVALID, "bfs_batch: negative node budget");
        P.nodes += max_nodes[s] + 16;
    }
    // the table stays <= 3/4 full: committed nodes, tombstones and one chunk's tentative claims
    uint64_t t = 1024;
    while (t < 5 * (uint64_t)P.nodes / 2) t <<= 1;
    P.tcap = t;
    if (P.nodes >= (int64_t)kMbIdx) return fail(ACS_ERR_UNSUPPORTED, "bfs_batch: too many nodes for one engine");
    // parents per chunk after the first: ~4 Mi (candidate ids are 32-bit)
    int64_t chunk = chunk_parents > 0 ? chunk_parents : (int64_t)1 << 22;
    chunk = std::min<int64_t>(chunk, std::max<int64_t>(P.nodes, 1024));
    chunk = std::min<int64_t>(chunk, ((int64_t)1 << 32) / 12 - 1);
    P.chunk = chunk;
    // the log and the bitmap also hold the first chunk, which expands every root
    const int64_t widest = std::max<int64_t>(chunk, n_search);
    if (widest > ((int64_t)1 << 32) / 12 - 1) return fail(ACS_ERR_UNSUPPORTED, "bfs_batch: too many searches");
    P.rec_cap = 12 * widest;
    P.bitmap_words = (12 * widest + 31) / 32 + 8;
    P.nblk = (P.bitmap_words + kScanBlock - 1) / kScanBlock + 1;
    const int64_t node_bytes = 8 * node_words(P.W);
    // per search: control minima, six segment arrays, the state and the root key
    const int64_t per_search = kMbCtrl * 8 + 4 + 8 + 8 + 8 + 8 + 4 + (int64_t)sizeof(MbSearch) + 16 * P.W;
    P.bytes = P.nodes * node_bytes + (int64_t)P.tcap * 8 + P.rec_cap * (16 * P.W + 4 + 4 + 8) + P.bitmap_words * 4 +
              (P.bitmap_words + 1) * 8 + P.nblk * 4 + (int64_t)n_search * per_search + 8 + 8 + (int64_t)sizeof(MbState);
    return ACS_OK;
}
}  // namespace

struct acs_bfs_batch {
    int device = 0, n_search = 0, mrl = 0, W = 1, cyclical = 0;
    MbPlan plan{};
    MbEngine E{};
    uint64_t* d_roots = nullptr;
    int32_t* d_paths = nullptr;
    int32_t* d_plen = nullptr;
    int d_path_cap = 0;
    std::vector<int64_t> budgets;
    std::vector<MbSearch> h_final;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ring_ev[kMbRing] = {};
    MbState* h_ring = nullptr;  // pinned [kMbRing]
    int sms = 148;
    int expand_blocks = 148, expand_blocks_sym = 148, expand_wpb = 8, insert_blocks = 148, commit_blocks = 148;
    size_t expand_smem = 0;
    bool ran = false;
    const acs_goalset* goals = nullptr;  // acs_bfs_batch_set_goals
    int explore = 0;                     // stop_at_trivial == 0
    bool adopted = false;                // the nodes went to a goal set (acs_goalset_from_bfs_batch)
    int symmetric = 0;                   // orbit search (acs_bfs_batch_set_symmetric)
    uint8_t* d_root_g = nullptr;         // [n_search] each root's element, with E.log_g allocated by set_symmetric
};

extern "C" {

int acs_bfs_batch_bytes(int n_search, int mrl, const int64_t* max_nodes, int64_t chunk_parents, int64_t* bytes_out) {
    if (!bytes_out) return ACS_ERR_INVALID;
    MbPlan P;
    const int rc = mb_plan(n_search, mrl, max_nodes, chunk_parents, P);
    if (rc != ACS_OK) return rc;
    *bytes_out = P.bytes;
    return ACS_OK;
}

void acs_bfs_batch_destroy(acs_bfs_batch* b) {
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->stream) {
        cudaStreamSynchronize(b->stream);
        cudaStreamDestroy(b->stream);
    }
    if (b->ev0) cudaEventDestroy(b->ev0);
    if (b->ev1) cudaEventDestroy(b->ev1);
    for (auto e : b->ring_ev)
        if (e) cudaEventDestroy(e);
    MbEngine& E = b->E;
    void* ptrs[] = {E.st, E.srch, E.nodes, E.table, E.log_keys, E.log_c, E.log_s, E.rec_slot, E.cursor, E.bitmap, E.rt,
                    E.bsums, E.ctrl, E.seg_search, E.seg_head, E.seg_off, E.seg_limit, E.seg_base, E.seg_of,
                    E.goal_hit, E.goal_hit_g, E.log_g, b->d_root_g, b->d_roots, b->d_paths, b->d_plen};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (b->h_ring) cudaFreeHost(b->h_ring);
    cudaGetLastError();
    delete b;
}

int acs_bfs_batch_create(int device, int n_search, int mrl, const int64_t* max_nodes, int cyclical, int64_t chunk_parents,
                         acs_bfs_batch** out) {
    if (!out) return ACS_ERR_INVALID;
    *out = nullptr;
    MbPlan P;
    const int rc = mb_plan(n_search, mrl, max_nodes, chunk_parents, P);
    if (rc != ACS_OK) return rc;
    if (const int rc2 = open_device(device, "bfs_batch")) return rc2;
    acs_bfs_batch* b = new acs_bfs_batch();
    b->device = device;
    b->n_search = n_search;
    b->mrl = mrl;
    b->W = P.W;
    b->cyclical = cyclical ? 1 : 0;
    b->plan = P;
    b->budgets.assign(max_nodes, max_nodes + n_search);
    auto bail = [&](int code, const std::string& m) {
        acs_bfs_batch_destroy(b);
        return fail(code, m);
    };
    MbEngine& E = b->E;
    E.rec_cap = P.rec_cap;
    ACS_ALLOC(E.st, sizeof(MbState), acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.srch, (size_t)n_search * sizeof(MbSearch), acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.nodes, (size_t)P.nodes * 8 * node_words(P.W), acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.table, (size_t)P.tcap * 8, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.log_keys, (size_t)P.rec_cap * 16 * P.W, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.log_c, (size_t)P.rec_cap * 4, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.log_s, (size_t)P.rec_cap * 4, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.rec_slot, (size_t)P.rec_cap * 8, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.cursor, 8, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.bitmap, (size_t)P.bitmap_words * 4, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.rt, (size_t)(P.bitmap_words + 1) * sizeof(uint2), acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.bsums, (size_t)P.nblk * 4, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.ctrl, (size_t)n_search * kMbCtrl * 8, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.seg_search, (size_t)n_search * 4, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.seg_head, (size_t)n_search * 8, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.seg_off, (size_t)(n_search + 1) * 8, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.seg_limit, (size_t)n_search * 8, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.seg_base, (size_t)n_search * 8, acs_bfs_batch_destroy(b));
    ACS_ALLOC(E.seg_of, (size_t)n_search * 4, acs_bfs_batch_destroy(b));
    ACS_ALLOC(b->d_roots, (size_t)n_search * 16 * P.W, acs_bfs_batch_destroy(b));
    if (cudaMallocHost((void**)&b->h_ring, kMbRing * sizeof(MbState)) != cudaSuccess)
        return bail(ACS_ERR_NOMEM, "bfs_batch: cudaMallocHost");
    if (cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(ACS_ERR_CUDA, "bfs_batch: cudaStreamCreate");
    cudaEventCreate(&b->ev0);
    cudaEventCreate(&b->ev1);
    for (auto& e : b->ring_ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) b->sms = prop.multiProcessorCount;
    b->expand_smem = (size_t)b->expand_wpb * (P.W == 1 ? mb_stage_bytes_per_warp<1>() : mb_stage_bytes_per_warp<2>());
    int per_sm = 1, per_sm_sym = 1, ib = 1, cb = 1;
    if (P.W == 1) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mb_expand_kernel<1, true, false>, 32 * b->expand_wpb, b->expand_smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_sym, mb_expand_kernel<1, true, true>, 32 * b->expand_wpb, b->expand_smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ib, mb_insert_kernel<1>, 256, 0);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cb, mb_commit_kernel<1, false>, 256, 0);
    } else {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mb_expand_kernel<2, true, false>, 32 * b->expand_wpb, b->expand_smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_sym, mb_expand_kernel<2, true, true>, 32 * b->expand_wpb, b->expand_smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ib, mb_insert_kernel<2>, 256, 0);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cb, mb_commit_kernel<2, false>, 256, 0);
    }
    cudaGetLastError();
    b->expand_blocks = b->sms * std::max(per_sm, 1);
    b->expand_blocks_sym = b->sms * std::max(per_sm_sym, 1);
    b->insert_blocks = b->sms * std::max(ib, 1);
    b->commit_blocks = b->sms * std::max(cb, 1);
    *out = b;
    return ACS_OK;
}

}  // extern "C"

namespace {

// Paths of the solved searches of the last run into h_paths [n_search, path_cap, 2]; plen gets every search's
// path length (0 if not solved).  A path longer than path_cap is an error, never truncated.
template <int W>
int mb_paths(acs_bfs_batch* b, int32_t* h_paths, int path_cap, std::vector<int32_t>& plen) {
    const int n = b->n_search;
    cudaStream_t s = b->stream;
    ACS_CUDA(cudaSetDevice(b->device));
    const int cap = std::max(path_cap, 1);  // the kernel writes the first pair of every solved path
    if (!b->d_paths || cap > b->d_path_cap) {
        if (b->d_paths) cudaFree(b->d_paths);
        b->d_paths = nullptr;
        b->d_path_cap = 0;
        ACS_CUDA(cudaMalloc((void**)&b->d_paths, (size_t)n * cap * 2 * sizeof(int32_t)));
        b->d_path_cap = cap;
    }
    if (!b->d_plen) ACS_CUDA(cudaMalloc((void**)&b->d_plen, (size_t)n * sizeof(int32_t)));
    if (b->symmetric) mb_path_kernel<W, true><<<(n + 127) / 128, 128, 0, s>>>(b->E, b->d_paths, cap, b->d_plen);
    else mb_path_kernel<W, false><<<(n + 127) / 128, 128, 0, s>>>(b->E, b->d_paths, cap, b->d_plen);
    ACS_CUDA(cudaGetLastError());
    plen.resize((size_t)n);
    ACS_CUDA(cudaMemcpyAsync(plen.data(), b->d_plen, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < n; ++i)
        if (plen[i] > path_cap)
            return fail(ACS_ERR_INVALID, "bfs_batch: a solution path is longer than path_cap (see path_len)");
    if (h_paths && path_cap > 0)
        ACS_CUDA(cudaMemcpy(h_paths, b->d_paths, (size_t)n * path_cap * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return ACS_OK;
}

template <int W>
int mb_run_impl(acs_bfs_batch* b, const int8_t* h_pres, int32_t* h_paths, int path_cap, acs_search_result* results) {
    const int n = b->n_search, mrl = b->mrl;
    MbEngine& E = b->E;
    if (b->adopted) return fail(ACS_ERR_INVALID, "bfs_batch: the engine's states were handed to a goal set");
    std::vector<MbSearch> init((size_t)n);
    std::vector<uint64_t> roots((size_t)n * 2 * W, 0);
    std::vector<uint8_t> root_g((size_t)n, 0);
    int64_t slab = 0, n_valid = 0;
    for (int s = 0; s < n; ++s) {
        MbSearch& M = init[s];
        std::memset(&M, 0, sizeof(M));
        M.budget = b->budgets[s];
        M.cap = b->budgets[s] + 16;
        M.slab = slab;
        slab += M.cap;
        M.n_nodes = 1;
        M.level_end = 1;
        M.sol_gid = -1;
        Key<W> root;
        int lens[2];
        const RootCheck rc = pack_root<W>(h_pres + (size_t)s * 2 * mrl, mrl, root, lens);
        if (rc == RootCheck::bad_letter)
            return fail(ACS_ERR_UNSUPPORTED, "bfs_batch: letters outside {+-1,+-2} are not supported by the packed search");
        if (rc != RootCheck::ok) {  // breadth_first.py:36-38 asserts is_array_valid_presentation
            M.status = ACS_ROW_ASSERT;
            M.done = 1;
            M.n_nodes = 0;
            continue;
        }
        M.min_len = lens[0] + lens[1];
        if (b->symmetric) {
            int g0 = 0;
            root = canonical<W>(root, g0);
            root_g[s] = (uint8_t)g0;
        }
        for (int i = 0; i < 2 * W; ++i) roots[(size_t)s * 2 * W + i] = root.k[i];
        ++n_valid;
    }
    MbState st{};
    st.chunk_cap = b->plan.chunk;
    st.tmask = b->plan.tcap - 1;
    st.mrl = mrl;
    st.cyclical = b->cyclical;
    st.n_search = n;
    st.used = n_valid;
    st.explore = b->explore;
    cudaStream_t s = b->stream;
    ACS_CUDA(cudaSetDevice(b->device));
    ACS_CUDA(cudaMemsetAsync(E.table, 0, b->plan.tcap * sizeof(uint64_t), s));
    if (E.goal_hit) ACS_CUDA(cudaMemsetAsync(E.goal_hit, 0xFF, (size_t)n * sizeof(int64_t), s));
    if (E.goal_hit_g) ACS_CUDA(cudaMemsetAsync(E.goal_hit_g, 0xFF, (size_t)n * sizeof(int32_t), s));
    b->h_ring[0] = st;  // pinned staging for the async upload
    ACS_CUDA(cudaMemcpyAsync(E.st, &b->h_ring[0], sizeof(MbState), cudaMemcpyHostToDevice, s));
    ACS_CUDA(cudaMemcpyAsync(E.srch, init.data(), init.size() * sizeof(MbSearch), cudaMemcpyHostToDevice, s));
    ACS_CUDA(cudaMemcpyAsync(b->d_roots, roots.data(), roots.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    if (b->symmetric) ACS_CUDA(cudaMemcpyAsync(b->d_root_g, root_g.data(), root_g.size(), cudaMemcpyHostToDevice, s));
    E.root_g = b->symmetric ? b->d_root_g : nullptr;
    ACS_CUDA(cudaStreamSynchronize(s));  // the staging copies above read host memory that goes out of scope
    ACS_CUDA(cudaEventRecord(b->ev0, s));
    mb_init_kernel<W><<<(n + 127) / 128, 128, 0, s>>>(E, b->d_roots);
    if (b->goals) mb_goal_roots_kernel<W><<<(n + 127) / 128, 128, 0, s>>>(E);
    mb_plan_kernel<<<1, 32, 0, s>>>(E, 1);
    ACS_CUDA(cudaGetLastError());
    const int decide_blocks = (n + 127) / 128;
    for (int64_t chunk = 0;; ++chunk) {
        if (chunk >= kMbLag) {
            ACS_CUDA(cudaEventSynchronize(b->ring_ev[(chunk - kMbLag) % kMbRing]));
            if (b->h_ring[(chunk - kMbLag) % kMbRing].done) break;
        }
        mb_prep_kernel<<<b->sms * 2, 256, 0, s>>>(E);
        const dim3 eg(b->symmetric ? b->expand_blocks_sym : b->expand_blocks), et(32 * b->expand_wpb);
        if (b->symmetric) {
            if (chunk == 0) mb_expand_kernel<W, false, true><<<eg, et, b->expand_smem, s>>>(E);
            else mb_expand_kernel<W, true, true><<<eg, et, b->expand_smem, s>>>(E);
        } else {
            if (chunk == 0) mb_expand_kernel<W, false, false><<<eg, et, b->expand_smem, s>>>(E);
            else mb_expand_kernel<W, true, false><<<eg, et, b->expand_smem, s>>>(E);
        }
        mb_insert_kernel<W><<<b->insert_blocks, 256, 0, s>>>(E);
        if (b->goals) mb_goal_kernel<W><<<b->insert_blocks, 256, 0, s>>>(E);
        mb_scan_sums_kernel<<<b->sms * 4, kScanT, 0, s>>>(E);
        mb_scan_top_kernel<<<1, kScanT, 0, s>>>(E);
        mb_scan_final_kernel<<<b->sms * 4, kScanT, 0, s>>>(E);
        mb_decide_kernel<<<decide_blocks, 128, 0, s>>>(E);
        if (b->symmetric) mb_commit_kernel<W, true><<<b->commit_blocks, 256, 0, s>>>(E);
        else mb_commit_kernel<W, false><<<b->commit_blocks, 256, 0, s>>>(E);
        mb_plan_kernel<<<1, 32, 0, s>>>(E, 0);
        ACS_CUDA(cudaGetLastError());
        ACS_CUDA(cudaMemcpyAsync(&b->h_ring[chunk % kMbRing], E.st, sizeof(MbState), cudaMemcpyDeviceToHost, s));
        ACS_CUDA(cudaEventRecord(b->ring_ev[chunk % kMbRing], s));
    }
    ACS_CUDA(cudaEventRecord(b->ev1, s));
    MbState fin{};
    b->h_final.resize((size_t)n);
    ACS_CUDA(cudaMemcpyAsync(&fin, E.st, sizeof(MbState), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaMemcpyAsync(b->h_final.data(), E.srch, (size_t)n * sizeof(MbSearch), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaStreamSynchronize(s));
    if (fin.ierr) {
        std::string m = "bfs_batch: internal error:";
        if (fin.ierr & MB_IERR_TABLE_FULL) m += " visited table full (more than 3/4 of its slots used)";
        if (fin.ierr & MB_IERR_SLAB_FULL) m += " node slab of a search full";
        return fail(ACS_ERR_CUDA, m);
    }
    b->ran = true;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, b->ev0, b->ev1);
    std::vector<int32_t> plen((size_t)n);
    const int rc = mb_paths<W>(b, h_paths, path_cap, plen);
    for (int i = 0; i < n; ++i) {
        const MbSearch& f = b->h_final[i];
        acs_search_result* r = results + i;
        std::memset(r, 0, sizeof(*r));
        r->solved = f.solved;
        r->status = f.status;
        r->budget_hit = f.budget_hit;
        r->path_len = plen[i];
        if (f.status == ACS_ROW_ASSERT && f.n_nodes == 0) {  // invalid root: the reference asserts before searching
            r->seconds_device = ms * 1e-3;
            continue;
        }
        r->n_visited = f.n_nodes;
        r->n_expanded = f.n_expanded;
        r->n_moves = f.solved ? f.sol_gid + 1 : (f.status ? (int64_t)(((uint64_t)f.err_code >> 2) + 1) : f.n_expanded * 12);
        r->frontier_left = f.n_nodes - f.n_expanded;
        r->n_levels = f.levels;
        r->n_minlen = f.n_minlen;
        for (int j = 0; j < f.n_minlen && j < 128; ++j) r->minlen_log[j] = f.minlen_log[j];
        r->seconds_device = ms * 1e-3;
    }
    return rc;
}

}  // namespace

extern "C" {

int acs_bfs_batch_run(acs_bfs_batch* b, const int8_t* h_presentations, int32_t* h_paths, int path_cap,
                      acs_search_result* results) {
    if (!b || !h_presentations || !results || path_cap < 0) return ACS_ERR_INVALID;
    return b->W == 1 ? mb_run_impl<1>(b, h_presentations, h_paths, path_cap, results)
                     : mb_run_impl<2>(b, h_presentations, h_paths, path_cap, results);
}

int acs_bfs_batch_paths(acs_bfs_batch* b, int32_t* h_paths, int path_cap) {
    if (!b || path_cap < 0 || (!h_paths && path_cap > 0)) return ACS_ERR_INVALID;
    if (!b->ran) return fail(ACS_ERR_INVALID, "bfs_batch: no completed run");
    std::vector<int32_t> plen;
    return b->W == 1 ? mb_paths<1>(b, h_paths, path_cap, plen) : mb_paths<2>(b, h_paths, path_cap, plen);
}

int acs_bfs_batch_visited(acs_bfs_batch* b, int search, int8_t* h_out, int64_t cap_rows, int64_t* n_out) {
    if (!b || search < 0 || search >= b->n_search || (!h_out && cap_rows > 0)) return ACS_ERR_INVALID;
    if (!b->ran) return fail(ACS_ERR_INVALID, "bfs_batch: no completed run");
    ACS_CUDA(cudaSetDevice(b->device));
    const MbSearch& f = b->h_final[search];
    const int64_t n = std::min<int64_t>(f.n_nodes, std::max<int64_t>(cap_rows, 0));
    if (n_out) *n_out = n;
    const uint64_t* slab = b->E.nodes + (size_t)f.slab * node_words(b->W);
    return records_to_host(b->W, slab, node_words(b->W), n, b->mrl, h_out, nullptr, b->stream);
}

}  // extern "C"

// ---- goal sets ---------------------------------------------------------------------------------------------
extern "C" {

int acs_bfs_batch_set_goals(acs_bfs_batch* b, const acs_goalset* g, int stop_at_trivial) {
    if (!b) return ACS_ERR_INVALID;
    if (g) {
        if (g->mrl != b->mrl)
            return fail(ACS_ERR_INVALID, "bfs_batch_set_goals: the goal set's max_relator_length differs from the engine's");
        if (g->cyclical != b->cyclical)
            return fail(ACS_ERR_INVALID, "bfs_batch_set_goals: the goal set's cyclical flag differs from the engine's");
        if (g->device != b->device)
            return fail(ACS_ERR_INVALID, "bfs_batch_set_goals: the goal set lives on another device");
        if (b->symmetric && !g->symmetric)  // an orbit search knows only the orbit of a child
            return fail(ACS_ERR_INVALID, "bfs_batch_set_goals: an orbit search needs a symmetric goal set");
        if (g->n_entries >= (int64_t)0xFFFFFFFF)  // a hit packs the entry into 32 bits beside its candidate id
            return fail(ACS_ERR_UNSUPPORTED, "bfs_batch_set_goals: goal sets of 2^32 - 1 entries or more are not supported");
        if (!b->E.goal_hit) {
            ACS_CUDA(cudaSetDevice(b->device));
            ACS_CUDA(cudaMalloc((void**)&b->E.goal_hit, (size_t)b->n_search * sizeof(int64_t)));
            ACS_CUDA(cudaMemset(b->E.goal_hit, 0xFF, (size_t)b->n_search * sizeof(int64_t)));
            ACS_CUDA(cudaMalloc((void**)&b->E.goal_hit_g, (size_t)b->n_search * sizeof(int32_t)));
            ACS_CUDA(cudaMemset(b->E.goal_hit_g, 0xFF, (size_t)b->n_search * sizeof(int32_t)));
        }
        b->E.goals = g->view();
    } else {
        b->E.goals = GoalView{nullptr, nullptr, 0, 0};
    }
    b->goals = g;
    b->explore = stop_at_trivial ? 0 : 1;
    return ACS_OK;
}

int acs_bfs_batch_goal_hits(acs_bfs_batch* b, int64_t* h_entry) {
    if (!b || !h_entry) return ACS_ERR_INVALID;
    if (!b->ran) return fail(ACS_ERR_INVALID, "bfs_batch: no completed run");
    if (!b->E.goal_hit) {
        std::fill(h_entry, h_entry + b->n_search, (int64_t)-1);
        return ACS_OK;
    }
    ACS_CUDA(cudaSetDevice(b->device));
    ACS_CUDA(cudaMemcpyAsync(h_entry, b->E.goal_hit, (size_t)b->n_search * sizeof(int64_t), cudaMemcpyDeviceToHost,
                            b->stream));
    ACS_CUDA(cudaStreamSynchronize(b->stream));
    return ACS_OK;
}

int acs_bfs_batch_goal_hit_elements(acs_bfs_batch* b, int32_t* h_elem) {
    if (!b || !h_elem) return ACS_ERR_INVALID;
    if (!b->ran) return fail(ACS_ERR_INVALID, "bfs_batch: no completed run");
    if (!b->E.goal_hit_g) {
        std::fill(h_elem, h_elem + b->n_search, -1);
        return ACS_OK;
    }
    ACS_CUDA(cudaSetDevice(b->device));
    ACS_CUDA(cudaMemcpyAsync(h_elem, b->E.goal_hit_g, (size_t)b->n_search * sizeof(int32_t), cudaMemcpyDeviceToHost,
                            b->stream));
    ACS_CUDA(cudaStreamSynchronize(b->stream));
    return ACS_OK;
}

int acs_goalset_from_bfs_batch(acs_bfs_batch* b, acs_goalset** out) {
    if (!b || !out) return ACS_ERR_INVALID;
    *out = nullptr;
    if (!b->ran) return fail(ACS_ERR_INVALID, "goalset_from_bfs_batch: the engine has no completed run");
    const int n = b->n_search;
    std::vector<int64_t> off((size_t)n + 1, 0), slab((size_t)n, 0);
    for (int s = 0; s < n; ++s) {
        off[s + 1] = off[s] + b->h_final[s].n_nodes;
        slab[s] = b->h_final[s].slab;
    }
    const int64_t total = off[n];
    ACS_CUDA(cudaSetDevice(b->device));
    ACS_CUDA(cudaStreamSynchronize(b->stream));
    // the engine is spent from here on: free its table and logs before the entries are allocated
    MbEngine& E = b->E;
    for (void** p : {(void**)&E.table, (void**)&E.log_keys, (void**)&E.log_c, (void**)&E.log_s, (void**)&E.rec_slot,
                     (void**)&E.bitmap, (void**)&E.rt, (void**)&E.bsums}) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    b->adopted = true;
    b->ran = false;
    acs_goalset* g = new acs_goalset();
    g->device = b->device;
    g->mrl = b->mrl;
    g->W = b->W;
    g->cyclical = b->cyclical;
    g->symmetric = b->symmetric;
    g->n_entries = total;
    int64_t* d_idx = nullptr;
    cudaError_t e = cudaMalloc((void**)&g->nodes, (size_t)std::max<int64_t>(total, 1) * 8 * node_words(b->W));
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_idx, (2 * (size_t)n + 1) * sizeof(int64_t));
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_idx, off.data(), off.size() * 8, cudaMemcpyHostToDevice, b->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(d_idx + n + 1, slab.data(), slab.size() * 8, cudaMemcpyHostToDevice, b->stream);
    if (e == cudaSuccess && total > 0) {
        const unsigned grid = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)b->sms * 8);
        if (b->W == 1) mb_adopt_kernel<1><<<grid, 256, 0, b->stream>>>(E.nodes, d_idx, d_idx + n + 1, n, g->nodes, (uint64_t)total);
        else mb_adopt_kernel<2><<<grid, 256, 0, b->stream>>>(E.nodes, d_idx, d_idx + n + 1, n, g->nodes, (uint64_t)total);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(b->stream);  // the host vectors above go out of scope
    if (d_idx) cudaFree(d_idx);
    if (e != cudaSuccess) {
        goalset_free(g);
        return cuda_fail(e, "goalset_from_bfs_batch");
    }
    cudaFree(E.nodes);
    E.nodes = nullptr;
    const int rc = goalset_index(g, b->stream);
    if (rc != ACS_OK) {
        goalset_free(g);
        return rc;
    }
    *out = g;
    return ACS_OK;
}

}  // extern "C"

// ---- orbit search ------------------------------------------------------------------------------------------
extern "C" {

int acs_bfs_batch_set_symmetric(acs_bfs_batch* b, int symmetric) {
    if (!b) return ACS_ERR_INVALID;
    if (symmetric) {
        if (b->goals && !b->goals->symmetric)
            return fail(ACS_ERR_INVALID, "bfs_batch_set_symmetric: an orbit search needs a symmetric goal set");
        if (b->n_search >= (1 << kMbSymShift))
            return fail(ACS_ERR_UNSUPPORTED, "bfs_batch_set_symmetric: orbit search supports fewer than 2^28 searches");
        if (!b->E.log_g) {
            ACS_CUDA(cudaSetDevice(b->device));
            ACS_CUDA(cudaMalloc((void**)&b->E.log_g, (size_t)b->E.rec_cap));
            ACS_CUDA(cudaMalloc((void**)&b->d_root_g, (size_t)b->n_search));
        }
    }
    b->symmetric = symmetric ? 1 : 0;
    return ACS_OK;
}

}  // extern "C"
