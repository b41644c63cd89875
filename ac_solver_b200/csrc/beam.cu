// beam.cu -- batched beam search: many independent searches of one max_relator_length and one `cyclical`
// flag, each keeping at every level the `width` shortest new states, advance together through the same
// kernel launches on one GPU.
//
// Contract (tests/beam_oracle.py states it on the host).  The visited list V of a search starts as [root]
// and the level-0 beam is [root].  At level d the candidates c = 12*i + m (move m of beam node i) are
// walked in increasing c; the first that raises, has total length 2 or is in the goal set ends the search
// and nothing of the level is committed.  Otherwise the children whose state is not in V, each at its
// smallest c, are ordered by (total length, c); the first min(width, budget - |V|) of them become the next
// beam and are appended to V in that order.  The search stops after a level whose next beam is empty, that
// brought |V| to the budget, or that reached the depth limit.
//
// Design.  The engine is the batched BFS engine (mbfs.cu) with a different level: a chunk holds whole
// beams (a segment per search, one level each), and one chunk is
//
//   plan     (one warp) the active searches' beams, in search order, up to the parents cap
//   prep     reset the winner bitmap, the record cursor, the control minima, the length histograms and the
//            chunk's level table
//   expand   mb_expand_kernel: children to the record log, first solving / raising child and first child
//            of each new minimal length per segment
//   insert   a child whose (search, state) is in the visited table is dropped; the others claim a slot of
//            the level table, smallest candidate id wins (the winner bitmap as in mbfs.cu)
//   goal     mb_goal_kernel on the winners
//   hist     per segment, the winners' total lengths (at most 2*61 < 128): histogram and c -> record map
//   decide   one thread per segment: the event that ends the search, the minimal-length log, or the prefix
//            of the histogram -> the offset of each length in the next beam and its size
//   select   one block per segment walks its candidates in c order: a winner of total length L goes to
//            offset[L] + (winners of length L before it), ranked with match/popc per warp; winners below
//            the beam size become nodes and enter the visited table
//
// The visited table holds committed nodes only (mbfs.cu's slot format, no tombstones): the winners that
// miss the beam were only ever in the level table, which is cleared every chunk.  So the tables stay
// proportional to the budget, whatever the width.  The host enqueues chunks ahead of the device and reads
// only a lagging pinned copy of the run state, as mbfs.cu does.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "ac_core.cuh"
#include "ac_keys.cuh"
#include "acs_internal.h"
#include "bfs_common.cuh"
#include "goalset.cuh"
#include "mb_engine.cuh"

namespace acs {

constexpr int kBmLens = 128;                  // total lengths are at most 2 * 61
constexpr int64_t kBmMaxWidth = 1 << 24;      // widest beam: a chunk's candidate ids stay below 2^32

struct BmEngine {
    MbEngine E;          // E.table: the visited table of committed nodes
    uint64_t* ltab;      // level table: (fingerprint << 40 | record + 1) of this chunk's claims
    int64_t* lmask;      // [1] slots of this chunk's level table - 1
    uint32_t* rec_of;    // [rec_cap] record of the winner of candidate c
    uint8_t* wlen;       // [rec_cap] total length of the winner of candidate c
    uint32_t* hist;      // [n_search][kBmLens] winners per total length, then each length's first rank
    int64_t width;       // beam width
    int32_t max_depth;   // levels to run at most; 0: no limit
};

// ---- plan: the next chunk's whole beams (one warp) -------------------------------------------------------
__global__ void __launch_bounds__(32) bm_plan_kernel(const BmEngine B, int first) {
    const MbEngine& E = B.E;
    MbState* st = E.st;
    if (st->done) return;
    const int lane = threadIdx.x;
    const int n = st->n_search;
    const int64_t P = first ? (int64_t)n : st->chunk_cap;  // the first chunk expands every root
    const uint32_t lt = (1u << lane) - 1u;
    int64_t carryD = 0;
    int carryK = 0;
    for (int base = 0; base < n; base += 32) {
        const int s = base + lane;
        int64_t d = 0, head = 0;
        if (s < n && !E.srch[s].done) {
            head = E.srch[s].head;
            d = E.srch[s].level_end - head;  // a whole beam: at most the width, and the width fits a chunk
        }
        int64_t x = d;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xFFFFFFFFu, x, o);
            if (lane >= o) x += t;
        }
        const int64_t D = carryD + x - d;
        const bool on = d > 0 && carryD + x <= P;  // the running sum is monotone: the beams taken are a prefix
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, on);
        if (on) {
            const int k = carryK + __popc(b & lt);
            E.seg_search[k] = s;
            E.seg_head[k] = head;
            E.seg_off[k] = D;
            E.seg_of[s] = k;
        }
        carryK += __popc(b);
        const uint32_t fit = __ballot_sync(0xFFFFFFFFu, carryD + x <= P);
        carryD += __shfl_sync(0xFFFFFFFFu, x, 31);
        if (fit != 0xFFFFFFFFu) break;
    }
    if (lane == 0) {
        int64_t F = 0;
        if (carryK) {
            const int last = E.seg_search[carryK - 1];
            F = E.seg_off[carryK - 1] + (E.srch[last].level_end - E.srch[last].head);
        }
        E.seg_off[carryK] = F;
        st->n_seg = carryK;
        st->Ftot = F;
        uint64_t t = 1024;
        while (t < 24 * (uint64_t)F) t <<= 1;  // the level table stays at most half full
        *B.lmask = (int64_t)t - 1;
        if (carryK == 0) st->done = 1;
    }
}

// ---- prep ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bm_prep_kernel(const BmEngine B) {
    const MbEngine& E = B.E;
    const MbState* st = E.st;
    if (st->done) return;
    const int64_t nwords = (12 * st->Ftot + 31) / 32;
    const int64_t nctrl = st->n_seg * kMbCtrl, nhist = st->n_seg * kBmLens, nlt = *B.lmask + 1;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += stride) E.bitmap[i] = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nctrl; i += stride) E.ctrl[i] = ~0ull;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nhist; i += stride) B.hist[i] = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nlt; i += stride) B.ltab[i] = 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) *E.cursor = 0;
}

// ---- insert: drop visited children, smallest candidate id wins each new (search, state) ------------------
template <int W>
__device__ __forceinline__ bool bm_visited(const MbEngine& E, const Key<W>& key, uint32_t s, uint64_t h, uint64_t tmask) {
    const uint64_t fp23 = h >> 41;
    for (uint64_t t = (h & tmask) & ~3ull, n = 0; n <= tmask; t = (t + 4) & tmask, n += 4) {
        uint64_t vv[4];
        load_bucket(E.table + t, vv);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint64_t cur = vv[j];
            if (cur == 0) return false;  // committed nodes are never removed: the probe ends at a free slot
            if ((cur >> 40) != fp23) continue;
            Key<W> other;
            int64_t pl, s2;
            node_load<W>(E.nodes, (cur & kMbIdx) - 1, other, pl, s2);
            if ((uint32_t)s2 == s && key_eq<W>(other, key)) return true;
        }
    }
    return false;
}

template <int W>
__global__ void __launch_bounds__(256) bm_insert_kernel(const BmEngine B) {
    const MbEngine& E = B.E;
    MbState* st = E.st;
    if (st->done) return;
    const unsigned long long n = *E.cursor;
    const uint64_t tmask = st->tmask, lmask = (uint64_t)*B.lmask;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const Key<W> key = load_key_cg<W>(E.log_keys, i);
        const uint32_t c = __ldcg(E.log_c + i), s = __ldcg(E.log_s + i);
        const uint64_t h = mb_hash<W>(key, s);
        if (bm_visited<W>(E, key, s, h, tmask)) continue;
        const uint64_t fp23 = h >> 41;
        const uint64_t mine = (fp23 << 40) | (i + 1);
        bool finished = false;
        for (uint64_t t = (h & lmask) & ~3ull, probes = 0; !finished; t = (t + 4) & lmask, probes += 4) {
            if (probes > lmask) {  // cannot happen: the level table is sized for twice the chunk's records
                atomicOr(&st->ierr, MB_IERR_TABLE_FULL);
                break;
            }
            uint64_t vv[4];
            load_bucket(B.ltab + t, vv);
#pragma unroll
            for (int jj = 0; jj < 4 && !finished; ++jj) {
                uint64_t cur = vv[jj];
                unsigned long long* sp = (unsigned long long*)&B.ltab[t + jj];
                if (cur == 0) {
                    cur = atomicCAS(sp, 0ull, (unsigned long long)mine);
                    if (cur == 0) {  // first sighting of this (search, state) in the level: claim
                        atomicXor(&E.bitmap[c >> 5], 1u << (c & 31));
                        finished = true;
                        break;
                    }
                }
                if ((cur >> 40) != fp23) continue;
                uint64_t p2 = (cur & kMbIdx) - 1;
                if (__ldcg(E.log_s + p2) != s || !key_eq<W>(load_key_cg<W>(E.log_keys, p2), key)) continue;
                for (;;) {  // the same (search, state): the smaller candidate id keeps the slot
                    const uint32_t c2 = __ldcg(E.log_c + p2);
                    if (c2 < c) break;
                    const uint64_t old = atomicCAS(sp, (unsigned long long)cur, (unsigned long long)mine);
                    if (old == cur) {
                        atomicXor(&E.bitmap[c2 >> 5], 1u << (c2 & 31));
                        atomicXor(&E.bitmap[c >> 5], 1u << (c & 31));
                        break;
                    }
                    cur = old;
                    p2 = (cur & kMbIdx) - 1;
                }
                finished = true;
            }
        }
    }
}

// ---- hist: winners per (segment, total length), and the winner record of every candidate id --------------
template <int W>
__global__ void __launch_bounds__(256) bm_hist_kernel(const BmEngine B) {
    const MbEngine& E = B.E;
    const MbState* st = E.st;
    if (st->done) return;
    const unsigned long long n = *E.cursor;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t c = __ldcg(E.log_c + i);
        if (!((__ldcg(E.bitmap + (c >> 5)) >> (c & 31)) & 1u)) continue;
        const int L = key_total_len<W>(load_key_cg<W>(E.log_keys, i));
        B.rec_of[c] = (uint32_t)i;
        B.wlen[c] = (uint8_t)L;
        atomicAdd(&B.hist[(int64_t)E.seg_of[__ldcg(E.log_s + i)] * kBmLens + L], 1u);
    }
}

// ---- decide: one thread per segment --------------------------------------------------------------------
// seg_limit[k] = the size of the next beam (0 when the level ended the search), seg_base[k] = the slab index
// of its first node; hist[k] becomes the rank in the next beam of the first winner of each length.
__global__ void __launch_bounds__(128) bm_decide_kernel(const BmEngine B) {
    const MbEngine& E = B.E;
    MbState* st = E.st;
    if (st->done) return;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k == 0) st->chunks += 1;
    if (k >= st->n_seg) return;
    const int s = E.seg_search[k];
    MbSearch& M = E.srch[s];
    const unsigned long long* red = E.ctrl + (int64_t)k * kMbCtrl;
    const uint64_t off = (uint64_t)E.seg_off[k], F = (uint64_t)E.seg_off[k + 1] - off;
    const uint64_t c0 = 12 * off, head = (uint64_t)M.head;
    uint64_t limit = 12 * F;  // candidates evaluated: up to the event, or all
    const unsigned long long sol = red[kMbSol], err = red[kMbErr], goal = red[kMbGoal];
    bool sol_here = false, goal_here = false;
    int status = 0;
    uint64_t ev = 0;
    if (sol != ~0ull) {
        ev = sol - c0;
        limit = ev;
        sol_here = true;
    }
    if (goal != ~0ull && (goal >> 32) - c0 < limit) {  // on the solving child itself the solve wins
        ev = (goal >> 32) - c0;
        limit = ev;
        sol_here = goal_here = true;
    }
    if (err != ~0ull && (err >> 2) - c0 < limit) {
        ev = (err >> 2) - c0;
        limit = ev;
        status = (int)(err & 3);
        sol_here = goal_here = false;
    }
    const uint64_t c_limit = limit + (sol_here ? 1 : 0);
    int min_len = M.min_len;
    for (;;) {  // new minimal lengths in candidate order
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
    E.seg_limit[k] = 0;
    if (sol_here || status) {
        M.done = 1;
        M.n_expanded = (int64_t)((12 * head + ev) / 12 + 1);
        if (status) {
            M.status = status;
            M.err_code = (int64_t)(((12 * head + ev) << 2) | (uint64_t)status);
            return;
        }
        M.solved = 1;
        M.sol_gid = (int64_t)(12 * head + ev);
        M.sol_len = 2;
        if (goal_here) {
            const uint64_t e = goal & 0xFFFFFFFFull;
            const int W = key_words(st->mrl);
            const uint64_t* q = E.goals.nodes + e * node_words(W);
            M.sol_len = key_len(q, W, 0) + key_len(q, W, 1);
            E.goal_hit[s] = (int64_t)e;
        }
        return;
    }
    uint32_t* h = B.hist + (int64_t)k * kBmLens;
    uint64_t total = 0;
    for (int L = 0; L < kBmLens; ++L) {
        const uint32_t v = h[L];
        h[L] = (uint32_t)total;
        total += v;
    }
    const uint64_t room = (uint64_t)(M.budget - M.n_nodes);
    uint64_t take = (uint64_t)B.width < room ? (uint64_t)B.width : room;
    take = take < total ? take : total;
    E.seg_limit[k] = (int64_t)take;
    E.seg_base[k] = M.slab + M.n_nodes;
    M.n_expanded = (int64_t)(head + F);
    M.head = (int64_t)(head + F);
    M.n_nodes += (int64_t)take;
    M.level_end = M.n_nodes;
    M.levels += 1;
    if (M.n_nodes >= M.budget) M.budget_hit = 1;
    if (take == 0 || M.budget_hit || (B.max_depth > 0 && M.levels >= B.max_depth)) M.done = 1;
}

// ---- select: one block per segment, candidates in c order -------------------------------------------------
constexpr int kBmSelT = 256, kBmSelWarps = kBmSelT / 32;

template <int W>
__global__ void __launch_bounds__(kBmSelT) bm_select_kernel(const BmEngine B) {
    const MbEngine& E = B.E;
    const MbState* st = E.st;
    if (st->done) return;
    __shared__ uint32_t run[kBmLens];                 // winners of each length in earlier tiles, plus its offset
    __shared__ uint32_t cnt[kBmSelWarps][kBmLens];    // this tile: winners of each length per warp
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    for (int64_t k = blockIdx.x; k < st->n_seg; k += gridDim.x) {
        const int64_t take = E.seg_limit[k];
        if (take == 0) continue;  // block-uniform
        const int s = E.seg_search[k];
        const int64_t off = E.seg_off[k], c0 = 12 * off, c1 = 12 * E.seg_off[k + 1];
        const int64_t base = E.seg_base[k], head = E.seg_head[k];
        const uint64_t tmask = st->tmask;
        for (int L = threadIdx.x; L < kBmLens; L += kBmSelT) run[L] = B.hist[k * kBmLens + L];
        for (int64_t t0 = c0; t0 < c1; t0 += kBmSelT) {
            for (int i = threadIdx.x; i < kBmSelWarps * kBmLens; i += kBmSelT) (&cnt[0][0])[i] = 0;
            __syncthreads();
            const int64_t c = t0 + threadIdx.x;
            const bool win = c < c1 && ((__ldcg(E.bitmap + (c >> 5)) >> (c & 31)) & 1u);
            const int L = win ? B.wlen[c] : kBmLens;  // kBmLens: no winner
            const uint32_t peers = __match_any_sync(0xFFFFFFFFu, L);
            if (win && (peers & lt) == 0) cnt[wid][L] = __popc(peers);
            __syncthreads();
            if (win) {
                uint32_t pos = run[L] + __popc(peers & lt);
                for (int w = 0; w < wid; ++w) pos += cnt[w][L];
                if ((int64_t)pos < take) {  // a node of the next beam
                    const uint32_t i = B.rec_of[c];
                    const Key<W> key = load_key_cg<W>(E.log_keys, i);
                    const int64_t idx = base + pos;
                    const int64_t pgid = head + (c - c0) / 12;
                    node_store<W>(E.nodes, (uint64_t)idx, key, (pgid << 4) | (int64_t)(c % 12), (int64_t)s);
                    const uint64_t h = mb_hash<W>(key, (uint32_t)s);
                    const uint64_t v = ((h >> 41) << 40) | kMbNode | (uint64_t)(idx + 1);
                    bool placed = false;
                    for (uint64_t t = (h & tmask) & ~3ull, n = 0; n <= tmask && !placed; t = (t + 1) & tmask, ++n)
                        placed = atomicCAS((unsigned long long*)&E.table[t], 0ull, (unsigned long long)v) == 0ull;
                    if (!placed) atomicOr(&E.st->ierr, MB_IERR_TABLE_FULL);
                }
            }
            __syncthreads();
            for (int l = threadIdx.x; l < kBmLens; l += kBmSelT) {
                uint32_t a = 0;
#pragma unroll
                for (int w = 0; w < kBmSelWarps; ++w) a += cnt[w][l];
                run[l] += a;
            }
            __syncthreads();
        }
    }
}

}  // namespace acs

// ---------------------------------------------------------------------------------------------------------
using namespace acs;

namespace {
constexpr int kBmRing = 4, kBmLag = 2;

// sizes of an engine (shared by acs_beam_bytes and acs_beam_create)
struct BmPlan {
    int W;
    int64_t nodes, chunk, rec_cap, bitmap_words, ltab_slots;
    uint64_t tcap;
    int64_t bytes;
};

int bm_plan(int n_search, int mrl, int64_t width, const int64_t* max_nodes, int max_depth, BmPlan& P) {
    if (n_search < 1 || !max_nodes) return fail(ACS_ERR_INVALID, "beam: need at least one search");
    if (width < 1) return fail(ACS_ERR_INVALID, "beam: the beam width must be at least 1");
    if (width > kBmMaxWidth) return fail(ACS_ERR_UNSUPPORTED, "beam: the beam width must be at most 2^24");
    if (max_depth < 0) return fail(ACS_ERR_INVALID, "beam: the depth limit must be >= 1, or 0 for none");
    if (const int rc = check_key_mrl(mrl, "beam")) return rc;
    P.W = key_words(mrl);
    P.nodes = 0;
    int64_t beams = 0, widest = 1;
    for (int s = 0; s < n_search; ++s) {
        if (max_nodes[s] < 1) return fail(ACS_ERR_INVALID, "beam: every node budget must be at least 1");
        P.nodes += max_nodes[s];
        const int64_t b = std::min<int64_t>(width, max_nodes[s]);
        beams += b;
        widest = std::max<int64_t>(widest, b);
    }
    if (P.nodes >= (int64_t)kMbIdx) return fail(ACS_ERR_UNSUPPORTED, "beam: too many nodes for one engine");
    uint64_t t = 1024;  // the visited table holds committed nodes only and stays at most half full
    while (t < 2 * (uint64_t)P.nodes) t <<= 1;
    P.tcap = t;
    // parents per chunk: every search's beam up to ~4 Mi, and always one whole beam
    P.chunk = std::max<int64_t>(widest, std::min<int64_t>(beams, (int64_t)1 << 22));
    const int64_t most = std::max<int64_t>(P.chunk, n_search);  // the first chunk expands every root
    if (most > ((int64_t)1 << 32) / 12 - 1) return fail(ACS_ERR_UNSUPPORTED, "beam: too many searches");
    P.rec_cap = 12 * most;
    P.bitmap_words = (P.rec_cap + 31) / 32 + 8;
    uint64_t lt = 1024;
    while (lt < 2 * (uint64_t)P.rec_cap) lt <<= 1;
    P.ltab_slots = (int64_t)lt;
    const int64_t node_bytes = 8 * node_words(P.W);
    // per search: control minima, histogram, five segment arrays, the state and the root key
    const int64_t per_search = kMbCtrl * 8 + kBmLens * 4 + 4 + 8 + 8 + 8 + 8 + 4 + (int64_t)sizeof(MbSearch) + 16 * P.W;
    P.bytes = P.nodes * node_bytes + (int64_t)P.tcap * 8 + P.rec_cap * (16 * P.W + 4 + 4 + 4 + 1) + P.bitmap_words * 4 +
              P.ltab_slots * 8 + (int64_t)n_search * per_search + 8 + 8 + (int64_t)sizeof(MbState);
    return ACS_OK;
}
}  // namespace

struct acs_beam {
    int device = 0, n_search = 0, mrl = 0, W = 1, cyclical = 0;
    BmPlan plan{};
    BmEngine B{};
    uint64_t* d_roots = nullptr;
    int32_t* d_paths = nullptr;
    int32_t* d_plen = nullptr;
    int d_path_cap = 0;
    std::vector<int64_t> budgets;
    std::vector<MbSearch> h_final;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ring_ev[kBmRing] = {};
    MbState* h_ring = nullptr;  // pinned [kBmRing]
    int sms = 148;
    int expand_blocks = 148, expand_wpb = 8, insert_blocks = 148;
    size_t expand_smem = 0;
    bool ran = false;
    const acs_goalset* goals = nullptr;  // acs_beam_set_goals
};

extern "C" {

int acs_beam_bytes(int n_search, int mrl, int64_t beam_width, const int64_t* max_nodes, int max_depth,
                   int64_t* bytes_out) {
    if (!bytes_out) return ACS_ERR_INVALID;
    BmPlan P;
    const int rc = bm_plan(n_search, mrl, beam_width, max_nodes, max_depth, P);
    if (rc != ACS_OK) return rc;
    *bytes_out = P.bytes;
    return ACS_OK;
}

void acs_beam_destroy(acs_beam* b) {
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
    MbEngine& E = b->B.E;
    void* ptrs[] = {E.st, E.srch, E.nodes, E.table, E.log_keys, E.log_c, E.log_s, E.cursor, E.bitmap, E.ctrl,
                    E.seg_search, E.seg_head, E.seg_off, E.seg_limit, E.seg_base, E.seg_of, E.goal_hit, E.goal_hit_g,
                    b->B.ltab, b->B.lmask, b->B.rec_of, b->B.wlen, b->B.hist, b->d_roots, b->d_paths, b->d_plen};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (b->h_ring) cudaFreeHost(b->h_ring);
    cudaGetLastError();
    delete b;
}

int acs_beam_create(int device, int n_search, int mrl, int64_t beam_width, const int64_t* max_nodes, int max_depth,
                    int cyclical, acs_beam** out) {
    if (!out) return ACS_ERR_INVALID;
    *out = nullptr;
    BmPlan P;
    const int rc = bm_plan(n_search, mrl, beam_width, max_nodes, max_depth, P);
    if (rc != ACS_OK) return rc;
    if (const int rc2 = open_device(device, "beam")) return rc2;
    acs_beam* b = new acs_beam();
    b->device = device;
    b->n_search = n_search;
    b->mrl = mrl;
    b->W = P.W;
    b->cyclical = cyclical ? 1 : 0;
    b->plan = P;
    b->budgets.assign(max_nodes, max_nodes + n_search);
    BmEngine& B = b->B;
    B.width = beam_width;
    B.max_depth = max_depth;
    MbEngine& E = B.E;
    E.rec_cap = P.rec_cap;
    ACS_ALLOC(E.st, sizeof(MbState), acs_beam_destroy(b));
    ACS_ALLOC(E.srch, (size_t)n_search * sizeof(MbSearch), acs_beam_destroy(b));
    ACS_ALLOC(E.nodes, (size_t)P.nodes * 8 * node_words(P.W), acs_beam_destroy(b));
    ACS_ALLOC(E.table, (size_t)P.tcap * 8, acs_beam_destroy(b));
    ACS_ALLOC(E.log_keys, (size_t)P.rec_cap * 16 * P.W, acs_beam_destroy(b));
    ACS_ALLOC(E.log_c, (size_t)P.rec_cap * 4, acs_beam_destroy(b));
    ACS_ALLOC(E.log_s, (size_t)P.rec_cap * 4, acs_beam_destroy(b));
    ACS_ALLOC(E.cursor, 8, acs_beam_destroy(b));
    ACS_ALLOC(E.bitmap, (size_t)P.bitmap_words * 4, acs_beam_destroy(b));
    ACS_ALLOC(E.ctrl, (size_t)n_search * kMbCtrl * 8, acs_beam_destroy(b));
    ACS_ALLOC(E.seg_search, (size_t)n_search * 4, acs_beam_destroy(b));
    ACS_ALLOC(E.seg_head, (size_t)n_search * 8, acs_beam_destroy(b));
    ACS_ALLOC(E.seg_off, (size_t)(n_search + 1) * 8, acs_beam_destroy(b));
    ACS_ALLOC(E.seg_limit, (size_t)n_search * 8, acs_beam_destroy(b));
    ACS_ALLOC(E.seg_base, (size_t)n_search * 8, acs_beam_destroy(b));
    ACS_ALLOC(E.seg_of, (size_t)n_search * 4, acs_beam_destroy(b));
    ACS_ALLOC(B.ltab, (size_t)P.ltab_slots * 8, acs_beam_destroy(b));
    ACS_ALLOC(B.lmask, 8, acs_beam_destroy(b));
    ACS_ALLOC(B.rec_of, (size_t)P.rec_cap * 4, acs_beam_destroy(b));
    ACS_ALLOC(B.wlen, (size_t)P.rec_cap, acs_beam_destroy(b));
    ACS_ALLOC(B.hist, (size_t)n_search * kBmLens * 4, acs_beam_destroy(b));
    ACS_ALLOC(b->d_roots, (size_t)n_search * 16 * P.W, acs_beam_destroy(b));
    auto bail = [&](int code, const std::string& m) {
        acs_beam_destroy(b);
        return fail(code, m);
    };
    if (cudaMallocHost((void**)&b->h_ring, kBmRing * sizeof(MbState)) != cudaSuccess)
        return bail(ACS_ERR_NOMEM, "beam: cudaMallocHost");
    if (cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(ACS_ERR_CUDA, "beam: cudaStreamCreate");
    cudaEventCreate(&b->ev0);
    cudaEventCreate(&b->ev1);
    for (auto& e : b->ring_ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) b->sms = prop.multiProcessorCount;
    b->expand_smem = (size_t)b->expand_wpb * (P.W == 1 ? mb_stage_bytes_per_warp<1>() : mb_stage_bytes_per_warp<2>());
    int per_sm = 1, ib = 1;
    if (P.W == 1) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mb_expand_kernel<1, true, false, false>, 32 * b->expand_wpb,
                                                      b->expand_smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ib, bm_insert_kernel<1>, 256, 0);
    } else {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mb_expand_kernel<2, true, false, false>, 32 * b->expand_wpb,
                                                      b->expand_smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ib, bm_insert_kernel<2>, 256, 0);
    }
    cudaGetLastError();
    b->expand_blocks = b->sms * std::max(per_sm, 1);
    b->insert_blocks = b->sms * std::max(ib, 1);
    *out = b;
    return ACS_OK;
}

}  // extern "C"

namespace {

// Paths of the solved searches of the last run (see mb_paths in mbfs.cu)
template <int W>
int bm_paths(acs_beam* b, int32_t* h_paths, int path_cap, std::vector<int32_t>& plen) {
    const int n = b->n_search;
    cudaStream_t s = b->stream;
    ACS_CUDA(cudaSetDevice(b->device));
    const int cap = std::max(path_cap, 1);
    if (!b->d_paths || cap > b->d_path_cap) {
        if (b->d_paths) cudaFree(b->d_paths);
        b->d_paths = nullptr;
        b->d_path_cap = 0;
        ACS_CUDA(cudaMalloc((void**)&b->d_paths, (size_t)n * cap * 2 * sizeof(int32_t)));
        b->d_path_cap = cap;
    }
    if (!b->d_plen) ACS_CUDA(cudaMalloc((void**)&b->d_plen, (size_t)n * sizeof(int32_t)));
    mb_path_kernel<W, false><<<(n + 127) / 128, 128, 0, s>>>(b->B.E, b->d_paths, cap, b->d_plen);
    ACS_CUDA(cudaGetLastError());
    plen.resize((size_t)n);
    ACS_CUDA(cudaMemcpyAsync(plen.data(), b->d_plen, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < n; ++i)
        if (plen[i] > path_cap) return fail(ACS_ERR_INVALID, "beam: a solution path is longer than path_cap (see path_len)");
    if (h_paths && path_cap > 0) {
        ACS_CUDA(cudaMemcpyAsync(h_paths, b->d_paths, (size_t)n * path_cap * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        ACS_CUDA(cudaStreamSynchronize(s));
    }
    return ACS_OK;
}

template <int W>
int bm_run_impl(acs_beam* b, const int8_t* h_pres, int32_t* h_paths, int path_cap, acs_search_result* results) {
    const int n = b->n_search, mrl = b->mrl;
    BmEngine& B = b->B;
    MbEngine& E = B.E;
    std::vector<MbSearch> init((size_t)n);
    std::vector<uint64_t> roots((size_t)n * 2 * W, 0);
    int64_t slab = 0;
    // every row is checked before any device work
    for (int s = 0; s < n; ++s) {
        Key<W> root;
        int lens[2];
        if (pack_root<W>(h_pres + (size_t)s * 2 * mrl, mrl, root, lens) == RootCheck::bad_letter)
            return fail(ACS_ERR_UNSUPPORTED, "beam: letters outside {+-1,+-2} are not supported by the packed search");
    }
    for (int s = 0; s < n; ++s) {
        MbSearch& M = init[s];
        std::memset(&M, 0, sizeof(M));
        M.budget = b->budgets[s];
        M.cap = b->budgets[s];
        M.slab = slab;
        slab += M.cap;
        M.n_nodes = 1;
        M.level_end = 1;
        M.sol_gid = -1;
        Key<W> root;
        int lens[2];
        if (pack_root<W>(h_pres + (size_t)s * 2 * mrl, mrl, root, lens) != RootCheck::ok) {
            M.status = ACS_ROW_ASSERT;  // is_array_valid_presentation fails: nothing is searched
            M.done = 1;
            M.n_nodes = 0;
            continue;
        }
        M.min_len = lens[0] + lens[1];
        for (int i = 0; i < 2 * W; ++i) roots[(size_t)s * 2 * W + i] = root.k[i];
    }
    MbState st{};
    st.chunk_cap = b->plan.chunk;
    st.tmask = b->plan.tcap - 1;
    st.mrl = mrl;
    st.cyclical = b->cyclical;
    st.n_search = n;
    cudaStream_t s = b->stream;
    ACS_CUDA(cudaSetDevice(b->device));
    ACS_CUDA(cudaMemsetAsync(E.table, 0, b->plan.tcap * sizeof(uint64_t), s));
    if (E.goal_hit) ACS_CUDA(cudaMemsetAsync(E.goal_hit, 0xFF, (size_t)n * sizeof(int64_t), s));
    if (E.goal_hit_g) ACS_CUDA(cudaMemsetAsync(E.goal_hit_g, 0xFF, (size_t)n * sizeof(int32_t), s));
    b->h_ring[0] = st;  // pinned staging for the async upload
    ACS_CUDA(cudaMemcpyAsync(E.st, &b->h_ring[0], sizeof(MbState), cudaMemcpyHostToDevice, s));
    ACS_CUDA(cudaMemcpyAsync(E.srch, init.data(), init.size() * sizeof(MbSearch), cudaMemcpyHostToDevice, s));
    ACS_CUDA(cudaMemcpyAsync(b->d_roots, roots.data(), roots.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    E.root_g = nullptr;
    ACS_CUDA(cudaStreamSynchronize(s));  // the staging copies above read host memory that goes out of scope
    ACS_CUDA(cudaEventRecord(b->ev0, s));
    mb_init_kernel<W><<<(n + 127) / 128, 128, 0, s>>>(E, b->d_roots);
    if (b->goals) mb_goal_roots_kernel<W><<<(n + 127) / 128, 128, 0, s>>>(E);
    ACS_CUDA(cudaGetLastError());
    const int decide_blocks = (n + 127) / 128;
    const int select_blocks = std::min(n, b->sms * 8);
    for (int64_t chunk = 0;; ++chunk) {
        if (chunk >= kBmLag) {
            ACS_CUDA(cudaEventSynchronize(b->ring_ev[(chunk - kBmLag) % kBmRing]));
            if (b->h_ring[(chunk - kBmLag) % kBmRing].done) break;
        }
        bm_plan_kernel<<<1, 32, 0, s>>>(B, chunk == 0);
        bm_prep_kernel<<<b->sms * 2, 256, 0, s>>>(B);
        const dim3 eg(b->expand_blocks), et(32 * b->expand_wpb);
        // the roots are expanded without the normal-form shortcuts; no move-skip rule: beams are not FIFO
        if (chunk == 0) mb_expand_kernel<W, false, false, false><<<eg, et, b->expand_smem, s>>>(E);
        else mb_expand_kernel<W, true, false, false><<<eg, et, b->expand_smem, s>>>(E);
        bm_insert_kernel<W><<<b->insert_blocks, 256, 0, s>>>(B);
        if (b->goals) mb_goal_kernel<W><<<b->insert_blocks, 256, 0, s>>>(E);
        bm_hist_kernel<W><<<b->insert_blocks, 256, 0, s>>>(B);
        bm_decide_kernel<<<decide_blocks, 128, 0, s>>>(B);
        bm_select_kernel<W><<<select_blocks, kBmSelT, 0, s>>>(B);
        ACS_CUDA(cudaGetLastError());
        ACS_CUDA(cudaMemcpyAsync(&b->h_ring[chunk % kBmRing], E.st, sizeof(MbState), cudaMemcpyDeviceToHost, s));
        ACS_CUDA(cudaEventRecord(b->ring_ev[chunk % kBmRing], s));
    }
    ACS_CUDA(cudaEventRecord(b->ev1, s));
    MbState fin{};
    b->h_final.resize((size_t)n);
    ACS_CUDA(cudaMemcpyAsync(&fin, E.st, sizeof(MbState), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaMemcpyAsync(b->h_final.data(), E.srch, (size_t)n * sizeof(MbSearch), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaStreamSynchronize(s));
    if (fin.ierr) return fail(ACS_ERR_CUDA, "beam: internal error: a hash table is full");
    b->ran = true;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, b->ev0, b->ev1);
    std::vector<int32_t> plen((size_t)n);
    const int rc = bm_paths<W>(b, h_paths, path_cap, plen);
    for (int i = 0; i < n; ++i) {
        const MbSearch& f = b->h_final[i];
        acs_search_result* r = results + i;
        std::memset(r, 0, sizeof(*r));
        r->solved = f.solved;
        r->status = f.status;
        r->budget_hit = f.budget_hit;
        r->path_len = plen[i];
        r->seconds_device = ms * 1e-3;
        if (f.status == ACS_ROW_ASSERT && f.n_nodes == 0) continue;  // invalid root: nothing searched
        r->n_visited = f.n_nodes;
        r->n_expanded = f.n_expanded;
        r->n_moves = f.solved ? f.sol_gid + 1 : (f.status ? (int64_t)(((uint64_t)f.err_code >> 2) + 1) : f.n_expanded * 12);
        r->frontier_left = f.n_nodes - f.n_expanded;
        r->n_levels = f.levels;
        r->n_minlen = f.n_minlen;
        for (int j = 0; j < f.n_minlen && j < 128; ++j) r->minlen_log[j] = f.minlen_log[j];
    }
    return rc;
}

}  // namespace

extern "C" {

int acs_beam_run(acs_beam* b, const int8_t* h_presentations, int32_t* h_paths, int path_cap,
                 acs_search_result* results) {
    if (!b || !h_presentations || !results || path_cap < 0 || (!h_paths && path_cap > 0)) return ACS_ERR_INVALID;
    return b->W == 1 ? bm_run_impl<1>(b, h_presentations, h_paths, path_cap, results)
                     : bm_run_impl<2>(b, h_presentations, h_paths, path_cap, results);
}

int acs_beam_paths(acs_beam* b, int32_t* h_paths, int path_cap) {
    if (!b || path_cap < 0 || (!h_paths && path_cap > 0)) return ACS_ERR_INVALID;
    if (!b->ran) return fail(ACS_ERR_INVALID, "beam: no completed run");
    std::vector<int32_t> plen;
    return b->W == 1 ? bm_paths<1>(b, h_paths, path_cap, plen) : bm_paths<2>(b, h_paths, path_cap, plen);
}

int acs_beam_visited(acs_beam* b, int search, int8_t* h_out, int64_t cap_rows, int64_t* n_out) {
    if (!b || search < 0 || search >= b->n_search || (!h_out && cap_rows > 0)) return ACS_ERR_INVALID;
    if (!b->ran) return fail(ACS_ERR_INVALID, "beam: no completed run");
    ACS_CUDA(cudaSetDevice(b->device));
    const MbSearch& f = b->h_final[search];
    const int64_t n = std::min<int64_t>(f.n_nodes, std::max<int64_t>(cap_rows, 0));
    if (n_out) *n_out = n;
    const uint64_t* slab = b->B.E.nodes + (size_t)f.slab * node_words(b->W);
    return records_to_host(b->W, slab, node_words(b->W), n, b->mrl, h_out, nullptr, b->stream);
}

int acs_beam_set_goals(acs_beam* b, const acs_goalset* g) {
    if (!b) return ACS_ERR_INVALID;
    if (g) {
        if (g->mrl != b->mrl)
            return fail(ACS_ERR_INVALID, "beam_set_goals: the goal set's max_relator_length differs from the engine's");
        if (g->cyclical != b->cyclical)
            return fail(ACS_ERR_INVALID, "beam_set_goals: the goal set's cyclical flag differs from the engine's");
        if (g->device != b->device) return fail(ACS_ERR_INVALID, "beam_set_goals: the goal set lives on another device");
        if (g->n_entries >= (int64_t)0xFFFFFFFF)  // a hit packs the entry into 32 bits beside its candidate id
            return fail(ACS_ERR_UNSUPPORTED, "beam_set_goals: goal sets of 2^32 - 1 entries or more are not supported");
        MbEngine& E = b->B.E;
        if (!E.goal_hit) {
            ACS_CUDA(cudaSetDevice(b->device));
            ACS_CUDA(cudaMalloc((void**)&E.goal_hit, (size_t)b->n_search * sizeof(int64_t)));
            ACS_CUDA(cudaMemset(E.goal_hit, 0xFF, (size_t)b->n_search * sizeof(int64_t)));
            ACS_CUDA(cudaMalloc((void**)&E.goal_hit_g, (size_t)b->n_search * sizeof(int32_t)));
            ACS_CUDA(cudaMemset(E.goal_hit_g, 0xFF, (size_t)b->n_search * sizeof(int32_t)));
        }
        E.goals = g->view();
    } else {
        b->B.E.goals = GoalView{nullptr, nullptr, 0, 0};
    }
    b->goals = g;
    return ACS_OK;
}

int acs_beam_goal_hits(acs_beam* b, int64_t* h_entry) {
    if (!b || !h_entry) return ACS_ERR_INVALID;
    if (!b->ran) return fail(ACS_ERR_INVALID, "beam: no completed run");
    if (!b->B.E.goal_hit) {
        std::fill(h_entry, h_entry + b->n_search, (int64_t)-1);
        return ACS_OK;
    }
    ACS_CUDA(cudaSetDevice(b->device));
    ACS_CUDA(cudaMemcpyAsync(h_entry, b->B.E.goal_hit, (size_t)b->n_search * sizeof(int64_t), cudaMemcpyDeviceToHost,
                             b->stream));
    ACS_CUDA(cudaStreamSynchronize(b->stream));
    return ACS_OK;
}

int acs_beam_goal_hit_elements(acs_beam* b, int32_t* h_elem) {
    if (!b || !h_elem) return ACS_ERR_INVALID;
    if (!b->ran) return fail(ACS_ERR_INVALID, "beam: no completed run");
    if (!b->B.E.goal_hit_g) {
        std::fill(h_elem, h_elem + b->n_search, -1);
        return ACS_OK;
    }
    ACS_CUDA(cudaSetDevice(b->device));
    ACS_CUDA(cudaMemcpyAsync(h_elem, b->B.E.goal_hit_g, (size_t)b->n_search * sizeof(int32_t), cudaMemcpyDeviceToHost,
                             b->stream));
    ACS_CUDA(cudaStreamSynchronize(b->stream));
    return ACS_OK;
}

}  // extern "C"
