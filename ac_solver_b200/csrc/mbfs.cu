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
#include "mb_host.cuh"

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
    const MbEvent ev = mb_event(red, st->explore ? ~0ull : red[kMbSol], c0, limit);
    mb_minlen_log(M, red, c0, limit, ev.solved);
    const uint64_t cg = mb_rank(E.rt, c0 + limit) - r0;
    E.seg_limit[k] = (int64_t)(c0 + limit);
    E.seg_base[k] = M.slab + (int64_t)n_nodes - (int64_t)r0;
    if ((int64_t)(n_nodes + cg) > M.cap) atomicOr(&st->ierr, MB_IERR_SLAB_FULL);  // the commit drops the excess
    M.n_nodes = (int64_t)(n_nodes + cg);
    if (ev.solved || ev.status) {
        mb_end_at(E, M, s, red, ev, head);
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

struct acs_bfs_batch : MbHost {
    MbPlan plan{};
    MbEngine E{};
    int expand_blocks_sym = 148, commit_blocks = 148;
    int explore = 0;                     // stop_at_trivial == 0
    bool adopted = false;                // the nodes went to a goal set (acs_goalset_from_bfs_batch)
    int symmetric = 0;                   // orbit search (acs_bfs_batch_set_symmetric)
    uint8_t* d_root_g = nullptr;         // [n_search] each root's element, with E.log_g allocated by set_symmetric
};

// launch sizes from the kernels' occupancy
template <int W>
static void mb_size_launches(acs_bfs_batch* b) {
    b->expand_smem = (size_t)b->expand_wpb * mb_stage_bytes_per_warp<W>();
    b->expand_blocks = mb_blocks(*b, mb_expand_kernel<W, true, false>, 32 * b->expand_wpb, b->expand_smem);
    b->expand_blocks_sym = mb_blocks(*b, mb_expand_kernel<W, true, true>, 32 * b->expand_wpb, b->expand_smem);
    b->insert_blocks = mb_blocks(*b, mb_insert_kernel<W>, 256, 0);
    b->commit_blocks = mb_blocks(*b, mb_commit_kernel<W, false>, 256, 0);
    cudaGetLastError();
}

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
    mb_close(*b, b->E);
    if (b->d_root_g) cudaFree(b->d_root_g);
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
    mb_init(*b, device, n_search, mrl, P.W, cyclical, max_nodes);
    b->plan = P;
    MbEngine& E = b->E;
    auto alloc = [&]() -> int {
        if (const int r = mb_alloc(b, E, P.nodes, P.tcap, P.rec_cap, P.bitmap_words)) return r;
        ACS_ALLOC(E.rec_slot, (size_t)P.rec_cap * 8, (void)0);
        ACS_ALLOC(E.rt, (size_t)(P.bitmap_words + 1) * sizeof(uint2), (void)0);
        ACS_ALLOC(E.bsums, (size_t)P.nblk * 4, (void)0);
        return mb_open(*b, "bfs_batch");
    };
    if (const int r = alloc()) {
        acs_bfs_batch_destroy(b);
        return r;
    }
    if (P.W == 1) mb_size_launches<1>(b);
    else mb_size_launches<2>(b);
    *out = b;
    return ACS_OK;
}

}  // extern "C"

namespace {

template <int W>
int mb_run_impl(acs_bfs_batch* b, const int8_t* h_pres, int32_t* h_paths, int path_cap, acs_search_result* results) {
    const int n = b->n_search;
    MbEngine& E = b->E;
    if (b->adopted) return fail(ACS_ERR_INVALID, "bfs_batch: the engine's states were handed to a goal set");
    MbRoots R;  // slabs of budget + 16 nodes (see the design note)
    if (const int rc = mb_pack_roots<W>(*b, h_pres, 16, b->symmetric, "bfs_batch", R)) return rc;
    MbState st{};
    st.chunk_cap = b->plan.chunk;
    st.tmask = b->plan.tcap - 1;
    st.mrl = b->mrl;
    st.cyclical = b->cyclical;
    st.n_search = n;
    st.used = R.n_valid;
    st.explore = b->explore;
    if (const int rc = mb_run_begin<W>(*b, E, st, R, b->symmetric ? b->d_root_g : nullptr)) return rc;
    cudaStream_t s = b->stream;
    mb_plan_kernel<<<1, 32, 0, s>>>(E, 1);
    ACS_CUDA(cudaGetLastError());
    const int decide_blocks = (n + 127) / 128;
    for (int64_t chunk = 0;; ++chunk) {
        if (const int done = mb_ring_done(*b, chunk)) {
            if (done < 0) return done;
            break;
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
        if (const int rc = mb_ring_publish(*b, E, chunk)) return rc;
    }
    int ierr = 0;
    const int rc = mb_run_end<W>(*b, E, b->symmetric, "bfs_batch", h_paths, path_cap, results, ierr);
    if (ierr) {
        std::string m = "bfs_batch: internal error:";
        if (ierr & MB_IERR_TABLE_FULL) m += " visited table full (more than 3/4 of its slots used)";
        if (ierr & MB_IERR_SLAB_FULL) m += " node slab of a search full";
        return fail(ACS_ERR_CUDA, m);
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
    return mb_paths_again(*b, b->E, b->symmetric, "bfs_batch", h_paths, path_cap);
}

int acs_bfs_batch_visited(acs_bfs_batch* b, int search, int8_t* h_out, int64_t cap_rows, int64_t* n_out) {
    if (!b || search < 0 || search >= b->n_search || (!h_out && cap_rows > 0)) return ACS_ERR_INVALID;
    return mb_visited(*b, b->E, "bfs_batch", search, h_out, cap_rows, n_out);
}

}  // extern "C"

// ---- goal sets ---------------------------------------------------------------------------------------------
extern "C" {

int acs_bfs_batch_set_goals(acs_bfs_batch* b, const acs_goalset* g, int stop_at_trivial) {
    if (!b) return ACS_ERR_INVALID;
    if (g)
        if (const int rc = goalset_check(g, b->mrl, b->cyclical, b->device, b->symmetric, "bfs_batch")) return rc;
    if (const int rc = mb_set_goals(*b, b->E, g)) return rc;
    b->explore = stop_at_trivial ? 0 : 1;
    return ACS_OK;
}

int acs_bfs_batch_goal_hits(acs_bfs_batch* b, int64_t* h_entry) {
    if (!b || !h_entry) return ACS_ERR_INVALID;
    return mb_goal_hits<int64_t>(*b, b->E.goal_hit, h_entry, "bfs_batch");
}

int acs_bfs_batch_goal_hit_elements(acs_bfs_batch* b, int32_t* h_elem) {
    if (!b || !h_elem) return ACS_ERR_INVALID;
    return mb_goal_hits<int32_t>(*b, b->E.goal_hit_g, h_elem, "bfs_batch");
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
