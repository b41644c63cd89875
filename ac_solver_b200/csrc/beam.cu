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
#include "mb_host.cuh"

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
    const MbEvent ev = mb_event(red, red[kMbSol], c0, limit);
    mb_minlen_log(M, red, c0, limit, ev.solved);
    E.seg_limit[k] = 0;
    if (ev.solved || ev.status) {
        M.done = 1;
        mb_end_at(E, M, s, red, ev, head);
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

struct acs_beam : MbHost {
    BmPlan plan{};
    BmEngine B{};
};

// launch sizes from the kernels' occupancy
template <int W>
static void bm_size_launches(acs_beam* b) {
    b->expand_smem = (size_t)b->expand_wpb * mb_stage_bytes_per_warp<W>();
    b->expand_blocks = mb_blocks(*b, mb_expand_kernel<W, true, false, false>, 32 * b->expand_wpb, b->expand_smem);
    b->insert_blocks = mb_blocks(*b, bm_insert_kernel<W>, 256, 0);
    cudaGetLastError();
}

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
    mb_close(*b, b->B.E);
    for (void* p : {(void*)b->B.ltab, (void*)b->B.lmask, (void*)b->B.rec_of, (void*)b->B.wlen, (void*)b->B.hist})
        if (p) cudaFree(p);
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
    mb_init(*b, device, n_search, mrl, P.W, cyclical, max_nodes);
    b->plan = P;
    BmEngine& B = b->B;
    B.width = beam_width;
    B.max_depth = max_depth;
    auto alloc = [&]() -> int {
        if (const int r = mb_alloc(b, B.E, P.nodes, P.tcap, P.rec_cap, P.bitmap_words)) return r;
        ACS_ALLOC(B.ltab, (size_t)P.ltab_slots * 8, (void)0);
        ACS_ALLOC(B.lmask, 8, (void)0);
        ACS_ALLOC(B.rec_of, (size_t)P.rec_cap * 4, (void)0);
        ACS_ALLOC(B.wlen, (size_t)P.rec_cap, (void)0);
        ACS_ALLOC(B.hist, (size_t)n_search * kBmLens * 4, (void)0);
        return mb_open(*b, "beam");
    };
    if (const int r = alloc()) {
        acs_beam_destroy(b);
        return r;
    }
    if (P.W == 1) bm_size_launches<1>(b);
    else bm_size_launches<2>(b);
    *out = b;
    return ACS_OK;
}

}  // extern "C"

namespace {

template <int W>
int bm_run_impl(acs_beam* b, const int8_t* h_pres, int32_t* h_paths, int path_cap, acs_search_result* results) {
    const int n = b->n_search;
    BmEngine& B = b->B;
    MbEngine& E = B.E;
    MbRoots R;  // slabs of exactly the budget: a level commits at most budget - |V| nodes
    if (const int rc = mb_pack_roots<W>(*b, h_pres, 0, false, "beam", R)) return rc;
    MbState st{};
    st.chunk_cap = b->plan.chunk;
    st.tmask = b->plan.tcap - 1;
    st.mrl = b->mrl;
    st.cyclical = b->cyclical;
    st.n_search = n;
    if (const int rc = mb_run_begin<W>(*b, E, st, R, nullptr)) return rc;
    cudaStream_t s = b->stream;
    const int decide_blocks = (n + 127) / 128;
    const int select_blocks = std::min(n, b->sms * 8);
    for (int64_t chunk = 0;; ++chunk) {
        if (const int done = mb_ring_done(*b, chunk)) {
            if (done < 0) return done;
            break;
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
        if (const int rc = mb_ring_publish(*b, E, chunk)) return rc;
    }
    int ierr = 0;
    const int rc = mb_run_end<W>(*b, E, false, "beam", h_paths, path_cap, results, ierr);
    if (ierr) return fail(ACS_ERR_CUDA, "beam: internal error: a hash table is full");
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
    return mb_paths_again(*b, b->B.E, false, "beam", h_paths, path_cap);
}

int acs_beam_visited(acs_beam* b, int search, int8_t* h_out, int64_t cap_rows, int64_t* n_out) {
    if (!b || search < 0 || search >= b->n_search || (!h_out && cap_rows > 0)) return ACS_ERR_INVALID;
    return mb_visited(*b, b->B.E, "beam", search, h_out, cap_rows, n_out);
}

int acs_beam_set_goals(acs_beam* b, const acs_goalset* g) {
    if (!b) return ACS_ERR_INVALID;
    if (g)
        if (const int rc = goalset_check(g, b->mrl, b->cyclical, b->device, false, "beam")) return rc;
    return mb_set_goals(*b, b->B.E, g);
}

int acs_beam_goal_hits(acs_beam* b, int64_t* h_entry) {
    if (!b || !h_entry) return ACS_ERR_INVALID;
    return mb_goal_hits<int64_t>(*b, b->B.E.goal_hit, h_entry, "beam");
}

int acs_beam_goal_hit_elements(acs_beam* b, int32_t* h_elem) {
    if (!b || !h_elem) return ACS_ERR_INVALID;
    return mb_goal_hits<int32_t>(*b, b->B.E.goal_hit_g, h_elem, "beam");
}

}  // extern "C"
