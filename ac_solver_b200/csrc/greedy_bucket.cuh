// greedy_bucket.cuh -- bucket-batched greedy search: one CTA per search, a whole (length, depth)
// bucket of the frontier expanded per round (SURVEY.md Appendix B), bit-exact with the reference's
// sequential greedy_search() (ac_solver/search/greedy.py:15-121, relative to /root/reference).
//
// The reference pops the minimum of (total_length, depth, state tuple) one node at a time.  All
// nodes of the minimal (length, depth) bucket are popped consecutively, in state order, until a
// child with a SMALLER total length is inserted (children have depth+1, so equal-length children
// land in a later bucket and never pre-empt).  Measured on the Miller-Schupp rows at budget 1e6:
// 120-160 k pops per unsolved search fall into only 240-2400 such runs.  So, per round:
//   pop      the minimal bucket from a small sorted directory in shared memory;
//   gather   its nodes (segments of an append-only frontier array) and SORT them by the
//            reference's tuple order (all-pairs ranking in shared memory for <= 256 nodes, a
//            bitonic network over (key, index) records otherwise);
//   tiles of <= 1024 sorted nodes:
//     expand   all 12 moves of every node in parallel, candidate id c = 12*position + action;
//     dedup    read-only probe of the exact visited table, then smallest-candidate-id-wins in a
//              per-round table -- duplicates keep the FIFO-earliest parent, like the reference;
//     decide   in candidate order: raising child, child of total length 2 (before the visited
//              test), budget reached after a node's 12 children, first node that produced a new
//              child with a smaller total length (the run ends after that node);
//     commit   winners below the limit are appended in candidate order (= the reference's
//              insertion order), entered into the visited table and into their buckets.
// Searches whose directory / segment pool / bucket size exceeds the fixed capacities are handed
// back (status kGbFallback) and re-run by the one-warp-per-search heap kernel in greedy.cu.
#pragma once
#include <cstdint>

#include "ac_core.cuh"
#include "ac_keys.cuh"
#include "goalset.cuh"

namespace acs {

// The capacities can be lowered at compile time (-DGB_TILE=64 ...), so that tests reach multi-tile
// buckets, the bitonic sort and every hand-back at budgets a CPU reference finishes quickly.
#ifndef GB_TILE
#define GB_TILE 1024
#endif
#ifndef GB_SMALL
#define GB_SMALL 256
#endif
#ifndef GB_BUCKETS1
#define GB_BUCKETS1 2048
#endif
#ifndef GB_BUCKETS2
#define GB_BUCKETS2 12288
#endif
#ifndef GB_MAX_SEG
#define GB_MAX_SEG 512
#endif
#ifndef GB_SEG_POOL
#define GB_SEG_POOL (1 << 16)
#endif
#ifndef GB_SORT_CAP
#define GB_SORT_CAP (1 << 16)
#endif
constexpr int kGbThreads = 256;
constexpr int kGbTile = GB_TILE;          // nodes per tile
constexpr int kGbCand = kGbTile * 12;     // candidates per tile
constexpr int kGbRoundSlots = 32768;      // per-round dedup table (power of two, > 2 * kGbCand)
constexpr int kGbBuckets1 = GB_BUCKETS1;  // open (length, depth) buckets per search: first pass ...
constexpr int kGbBuckets2 = GB_BUCKETS2;  // ... and for the searches that outgrow it (one CTA per SM)
constexpr int kGbMaxSeg = GB_MAX_SEG;     // segments gathered per bucket
constexpr int kGbSegPool = GB_SEG_POOL;   // segment records per search
constexpr int kGbSortCap = GB_SORT_CAP;   // nodes per bucket that can be sorted
constexpr int kGbSmall = GB_SMALL;        // buckets up to this size are ranked in shared memory
constexpr int kGbFallback = 99;           // internal status: re-run with the heap kernel
constexpr uint32_t kGbNone = 0xFFFFFFFFu;
// the dedup probe wraps with a mask and stays below half full
static_assert((kGbRoundSlots & (kGbRoundSlots - 1)) == 0 && kGbRoundSlots > 2 * kGbCand, "round table");
// the candidate bitmap has whole words, and its prefix scan takes at most 2 words per thread
static_assert(kGbTile > 0 && kGbCand % 32 == 0 && kGbCand / 32 <= 2 * kGbThreads, "tile size");
// the bitonic network pads a bucket to np2 <= kGbSortCap records
static_assert(kGbSortCap > 0 && (kGbSortCap & (kGbSortCap - 1)) == 0, "sort capacity");
// all-pairs ranking: thread t places record t
static_assert(kGbSmall >= 1 && kGbSmall <= kGbThreads, "all-pairs ranking");
static_assert(kGbMaxSeg >= 1 && kGbSegPool >= 1, "segments");

struct GbBucket {
    uint32_t key;       // length << 24 | depth
    uint32_t count;     // nodes
    uint32_t seg_head;  // segment record ids
    uint32_t seg_tail;
};
struct GbSeg {
    uint32_t start, count, next, pad;
};

// extra per-search pools of the bucket kernel (device pointers, strides per search)
struct GbArgs {
    uint32_t* frontier;   // [S][fcap]      append-only node indices, grouped by bucket segment
    GbSeg* segs;          // [S][kGbSegPool]
    uint64_t* sortbuf;    // [S][kGbSortCap][2W+2]  (key, index) records
    uint64_t* cand_key;   // [S][kGbCand][2W]
    uint32_t* cand_meta;  // [S][kGbCand]   length | status << 8 | emitted << 10 | visited << 11
    uint32_t* cand_slot;  // [S][kGbCand]
    uint64_t* round_tab;  // [S][kGbRoundSlots]
    uint64_t fcap;
    int max_buckets;      // capacity of the bucket directory in shared memory
    int retry_only;       // run only the searches a previous pass handed back
};

// (followed in shared memory by the bucket directory GbBucket B[max_buckets], sorted by key,
// DESCENDING: the minimum is the last entry)
struct GbShared {
    uint32_t bitmap[kGbCand / 32];
    uint32_t prefix[kGbCand / 32 + 1];
    uint32_t cntL[128], segstart[128], bucket_of[128];
    uint32_t first_len[128];
    uint32_t seg_start[kGbMaxSeg], seg_pref[kGbMaxSeg + 1];
    uint32_t scan_tmp[kGbThreads / 32];
    int nb;
    uint32_t n_seg, sol_c, err_c, tstar_c;
    uint32_t f_end, seg_used;
    uint32_t limit, n_commit, stop, processed;
    uint32_t cur_key, cur_n;
    int fallback;
};
enum : uint32_t { GB_CONT = 0, GB_INTERRUPT = 1, GB_BUDGET = 2, GB_SOLVED = 3, GB_ERROR = 4, GB_GOAL = 5 };

// words per sort record: the key, the node index and one spare word (a record of its own, not a node record)
__host__ __device__ constexpr int gb_rec_words(int W) { return 2 * W + 2; }
template <int W>
__device__ __forceinline__ uint64_t* gb_rec(uint64_t* sortbuf, uint32_t i) {
    return sortbuf + (size_t)i * gb_rec_words(W);
}
template <int W>
__device__ __forceinline__ Key<W> gb_rec_key(const uint64_t* sortbuf, uint32_t i) {
    Key<W> k;
    const uint64_t* p = sortbuf + (size_t)i * gb_rec_words(W);
#pragma unroll
    for (int t = 0; t < 2 * W; ++t) k.k[t] = p[t];
    return k;
}
// order of the sort records: padding records (index kGbNone) last, else the reference's tuple order
template <int W>
__device__ __forceinline__ bool gb_rec_less(const Key<W>& ka, uint32_t ia, const Key<W>& kb, uint32_t ib) {
    if (ia == kGbNone || ib == kGbNone) return ia != kGbNone && ib == kGbNone;
    return key_less<W>(ka, kb);
}

// block-wide exclusive scan of one value per thread (kGbThreads threads)
__device__ __forceinline__ uint32_t gb_block_scan(uint32_t v, uint32_t* tmp, uint32_t& total) {
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, x, off);
        if (lane >= off) x += t;
    }
    __syncthreads();
    if (lane == 31) tmp[wid] = x;
    __syncthreads();
    uint32_t before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kGbThreads / 32; ++w) {
        const uint32_t s = tmp[w];
        if (w < (int)wid) before += s;
        tot += s;
    }
    total = tot;
    return before + x - v;
}

__device__ __forceinline__ uint32_t gb_rank(const GbShared& sh, uint32_t c) {
    const uint32_t r = c & 31;
    return sh.prefix[c >> 5] + (r ? __popc(sh.bitmap[c >> 5] & ((1u << r) - 1u)) : 0u);
}

// position of `key` in the descending directory: first index whose key is <= `key`
__device__ __forceinline__ int gb_find(const GbBucket* B, int nb, uint32_t key) {
    int lo = 0, hi = nb;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (B[mid].key > key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// GOAL: the goal test of DESIGN.md §K9 against G.  A winner of the per-tile dedup that is in the set takes
// the minimum of (candidate << 32 | entry) in one more shared-memory word, placed after the bucket
// directory (the launch adds kGbGoalSmem bytes), and phase C resolves it like a solving child.  Only
// winners are looked up: a visited child was tested when it was first generated (the root at start), and a
// child that lost its slot follows a smaller candidate id of the same state.
constexpr int kGbGoalSmem = 16;
// both passes launch with the dynamic shared memory the host sets for kGbBuckets2 (greedy_run_impl), within the
// 227 KB a block may opt in to; the root's bucket needs one directory entry
static_assert(kGbBuckets1 >= 1 && kGbBuckets1 <= kGbBuckets2, "bucket directories");
static_assert(((sizeof(GbShared) + 15) / 16) * 16 + (size_t)kGbBuckets2 * sizeof(GbBucket) + kGbGoalSmem <= 227 * 1024,
              "the large bucket directory exceeds the shared memory of a block");
template <int W, bool GOAL>
#ifndef GB_MIN_BLOCKS
#define GB_MIN_BLOCKS 5  // resident CTAs per SM the register allocation must allow: 48 registers, 5 x 42 KB of shared memory
                         // -> 740 searches in flight on 148 SMs (the 657 unsolved rows of config 3 run as one wave)
#endif
__global__ void __launch_bounds__(kGbThreads, GB_MIN_BLOCKS)
    greedy_bucket_kernel(const GreedyArgs A, const GbArgs X, const GoalView G) {
    extern __shared__ __align__(16) unsigned char gb_smem_raw[];
    GbShared& sh = *reinterpret_cast<GbShared*>(gb_smem_raw);
    GbBucket* B = reinterpret_cast<GbBucket*>(gb_smem_raw + ((sizeof(GbShared) + 15) / 16) * 16);
    const int sidx = blockIdx.x;
    if (sidx >= A.n_search) return;
    if (X.retry_only && A.rec[sidx].status != kGbFallback) return;
    const int tid = threadIdx.x;
    constexpr int RS = gb_rec_words(W);
    uint64_t* keys = A.keys + (uint64_t)sidx * A.cap * 2 * W;
    uint64_t* parent = A.parent + (uint64_t)sidx * A.cap;
    uint64_t* table = A.table + (uint64_t)sidx * A.tcap;
    const uint64_t tmask = A.tcap - 1;
    GreedyRec* rec = A.rec + sidx;
    uint32_t* frontier = X.frontier + (uint64_t)sidx * X.fcap;
    GbSeg* segs = X.segs + (uint64_t)sidx * kGbSegPool;
    uint64_t* sortbuf = X.sortbuf + (uint64_t)sidx * kGbSortCap * RS;
    uint64_t* cand_key = X.cand_key + (uint64_t)sidx * kGbCand * 2 * W;
    uint32_t* cand_meta = X.cand_meta + (uint64_t)sidx * kGbCand;
    uint32_t* cand_slot = X.cand_slot + (uint64_t)sidx * kGbCand;
    uint64_t* round_tab = X.round_tab + (uint64_t)sidx * kGbRoundSlots;

    // ---- root ----
    Key<W> root;
#pragma unroll
    for (int i = 0; i < 2 * W; ++i) root.k[i] = A.roots[(uint64_t)sidx * 2 * W + i];
    const int L0 = key_total_len<W>(root);
    if (tid == 0) {
        store_key<W>(keys, 0, root);
        parent[0] = kNone;
        const uint64_t h = key_hash<W>(root);
        table[h & tmask] = ((h >> 40) << 40) | 1ull;
        frontier[0] = 0;
        segs[0] = GbSeg{0u, 1u, kGbNone, 0u};
        B[0] = GbBucket{(uint32_t)L0 << 24, 1u, 0u, 0u};
        sh.nb = 1;
        sh.f_end = 1;
        sh.seg_used = 1;
        sh.fallback = 0;
    }
    for (int i = tid; i < kGbRoundSlots; i += kGbThreads) round_tab[i] = 0;
    __syncthreads();
    // search state, replicated in every thread's registers (all decisions come from shared memory)
    uint64_t n_nodes = 1, n_expanded = 0, n_moves = 0;
    int min_len = L0, n_minlen = 0;
    int solved = 0, status = 0, budget_hit = 0;
    uint64_t cur = 0, cur_rest = 0;
    int final_action = 11, final_len = L0;
    bool finished = false;
    int rounds = 0;
    // with goals: the goal slot holds the winning (candidate << 32 | entry) of the current tile; after a hit
    // nothing resets it, and sh.stop says GB_GOAL (so no register carries the entry through the rounds)
    if constexpr (GOAL) {  // a root in the set: path [(-1, L0)], nothing expanded
        unsigned long long& goal_slot = *reinterpret_cast<unsigned long long*>(B + X.max_buckets);
        if (tid == 0) {
            const int64_t e = goal_find<W>(G, root);
            goal_slot = e < 0 ? ~0ull : (unsigned long long)e;
            sh.stop = e < 0 ? GB_CONT : GB_GOAL;
        }
        __syncthreads();
        if (goal_slot != ~0ull) {
            solved = 1;
            final_action = -1;
            finished = true;
        }
    }

    while (!finished) {
        if (sh.nb == 0 || sh.fallback) break;
        // ================= pop the minimal bucket =================
        __syncthreads();
        if (tid == 0) {
            const GbBucket b = B[sh.nb - 1];
            sh.nb -= 1;
            sh.cur_key = b.key;
            sh.cur_n = b.count;
            // walk its segment list
            uint32_t ns = 0, run = 0;
            for (uint32_t s = b.seg_head; s != kGbNone;) {
                if (ns >= kGbMaxSeg) {
                    sh.fallback = 1;  // reason 1: too many segments
                    break;
                }
                const GbSeg g = segs[s];
                sh.seg_start[ns] = g.start;
                sh.seg_pref[ns] = run;
                run += g.count;
                ++ns;
                s = g.next;
            }
            sh.seg_pref[ns] = run;
            sh.n_seg = ns;
            if (b.count > (uint32_t)kGbSortCap) sh.fallback = 2;  // bucket larger than the sort buffer
        }
        __syncthreads();
        if (sh.fallback) break;
        ++rounds;
        const uint32_t n = sh.cur_n;
        const int Lcur = (int)(sh.cur_key >> 24);
        const uint32_t dcur = sh.cur_key & 0xFFFFFFu;
        // ================= gather (key, index) records =================
        uint32_t np2 = 1;
        while (np2 < n) np2 <<= 1;
        for (uint32_t i = tid; i < np2; i += kGbThreads) {
            uint64_t* r = gb_rec<W>(sortbuf, i);
            if (i < n) {
                int lo = 0, hi = (int)sh.n_seg;  // segment containing position i
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (sh.seg_pref[mid] <= i) lo = mid;
                    else hi = mid;
                }
                const uint32_t idx = frontier[sh.seg_start[lo] + (i - sh.seg_pref[lo])];
                const Key<W> k = load_key<W>(keys, idx);
#pragma unroll
                for (int t = 0; t < 2 * W; ++t) r[t] = k.k[t];
                r[2 * W] = idx;
            } else {
                r[2 * W] = kGbNone;
            }
        }
        __syncthreads();
        // ================= sort by the reference's tuple order =================
        if (n > 1 && n <= (uint32_t)kGbSmall) {
            // all-pairs ranking (keys are distinct): thread t finds the position of record t
            Key<W> mine;
            uint32_t my_idx = kGbNone, rank = 0;
            if ((uint32_t)tid < n) {
                mine = gb_rec_key<W>(sortbuf, tid);
                my_idx = (uint32_t)sortbuf[(size_t)tid * RS + 2 * W];
                for (uint32_t j = 0; j < n; ++j) {
                    const Key<W> o = gb_rec_key<W>(sortbuf, j);
                    rank += (j != (uint32_t)tid && key_less<W>(o, mine)) ? 1u : 0u;
                }
            }
            __syncthreads();
            if ((uint32_t)tid < n) {
                uint64_t* r = gb_rec<W>(sortbuf, rank);
#pragma unroll
                for (int t = 0; t < 2 * W; ++t) r[t] = mine.k[t];
                r[2 * W] = my_idx;
            }
            __syncthreads();
        } else if (n > (uint32_t)kGbSmall) {
            for (uint32_t k2 = 2; k2 <= np2; k2 <<= 1) {
                for (uint32_t j = k2 >> 1; j > 0; j >>= 1) {
                    for (uint32_t i = tid; i < np2; i += kGbThreads) {
                        const uint32_t l = i ^ j;
                        if (l > i) {
                            const Key<W> ka = gb_rec_key<W>(sortbuf, i), kb = gb_rec_key<W>(sortbuf, l);
                            const uint32_t ia = (uint32_t)sortbuf[(size_t)i * RS + 2 * W];
                            const uint32_t ib = (uint32_t)sortbuf[(size_t)l * RS + 2 * W];
                            const bool asc = (i & k2) == 0;
                            const bool swap = asc ? gb_rec_less<W>(kb, ib, ka, ia) : gb_rec_less<W>(ka, ia, kb, ib);
                            if (swap) {
                                uint64_t* ra = gb_rec<W>(sortbuf, i);
                                uint64_t* rb = gb_rec<W>(sortbuf, l);
#pragma unroll
                                for (int t = 0; t < 2 * W; ++t) {
                                    ra[t] = kb.k[t];
                                    rb[t] = ka.k[t];
                                }
                                ra[2 * W] = ib;
                                rb[2 * W] = ia;
                            }
                        }
                    }
                    __syncthreads();
                }
            }
        }
        // ================= tiles of the sorted bucket =================
        uint32_t done_nodes = 0;  // nodes of this bucket already expanded
        uint32_t stop = GB_CONT;
        for (uint32_t tile0 = 0; tile0 < n && stop == GB_CONT; tile0 += kGbTile) {
            const uint32_t Tn = min((uint32_t)kGbTile, n - tile0);
            const uint32_t ncand = Tn * 12;
            // ---- reset the round state ----
            for (int i = tid; i < kGbCand / 32; i += kGbThreads) sh.bitmap[i] = 0;
            if (tid < 128) {
                sh.cntL[tid] = 0;
                sh.first_len[tid] = kGbNone;
            }
            if (tid == 0) {
                sh.sol_c = kGbNone;
                sh.err_c = kGbNone;
                sh.tstar_c = kGbNone;
                if constexpr (GOAL) *reinterpret_cast<unsigned long long*>(B + X.max_buckets) = ~0ull;
            }
            __syncthreads();
            // ---- A1: expand: candidate keys, lengths, events ----
            for (uint32_t c = tid; c < ncand; c += kGbThreads) {
                const uint32_t t = c / 12;
                const int a = (int)(c - t * 12);
                const Key<W> pk = gb_rec_key<W>(sortbuf, tile0 + t);
                const uint32_t pidx = (uint32_t)sortbuf[(size_t)(tile0 + t) * RS + 2 * W];
                Rel<2 * W> r0, r1;
                split_key<W>(pk, r0, r1);
                bool co;
                const int st = pidx ? apply_move<2 * W, true>(r0, r1, a, A.mrl, A.cyclical != 0, co)
                                    : apply_move<2 * W, false>(r0, r1, a, A.mrl, A.cyclical != 0, co);
                uint32_t meta = 0;
                if (st != ST_OK) {
                    atomicMin(&sh.err_c, (c << 2) | (uint32_t)st);
                    meta = (uint32_t)st << 8;
                } else {
                    const int L = r0.len + r1.len;
                    meta = (uint32_t)L;
                    if (L < min_len) atomicMin(&sh.first_len[L], c);
                    if (L == 2) atomicMin(&sh.sol_c, c);  // greedy.py:91-100, before the visited test
                    const Key<W> child = make_key<W>(r0, r1);
                    if (!key_eq<W>(child, pk)) {
                        meta |= 1u << 10;
                        store_key<W>(cand_key, c, child);
                    }
                }
                cand_meta[c] = meta;
            }
            __syncthreads();
            // ---- A2: dedup: read-only probe of the visited table, then smallest-candidate-id-wins
            // among the duplicates of this tile in the per-round table ----
            for (uint32_t c = tid; c < ncand; c += kGbThreads) {
                uint32_t slot = kGbNone;
                if ((cand_meta[c] >> 10) & 1u) {
                    const Key<W> child = load_key<W>(cand_key, c);
                    const uint64_t h = key_hash<W>(child);
                    const uint64_t fp = h >> 40;
                    bool visited = false;
                    for (uint64_t s = h & tmask;; s = (s + 1) & tmask) {  // the table holds committed nodes only
                        const uint64_t e = __ldcg(&table[s]);
                        if (e == 0) break;
                        if ((e >> 40) == fp && key_eq<W>(load_key<W>(keys, (e & kIdxMask) - 1), child)) {
                            visited = true;
                            break;
                        }
                    }
                    if (!visited) {
                        const uint64_t mine = ((h >> 32) << 32) | (uint64_t)(c + 1);
                        for (uint32_t s = (uint32_t)(h >> 7) & (kGbRoundSlots - 1);; s = (s + 1) & (kGbRoundSlots - 1)) {
                            uint64_t e = __ldcg(&round_tab[s]);
                            if (e == 0) {
                                e = atomicCAS((unsigned long long*)&round_tab[s], 0ull, (unsigned long long)mine);
                                if (e == 0) {
                                    slot = s;
                                    break;
                                }
                            }
                            if ((e >> 32) == (mine >> 32) && key_eq<W>(load_key<W>(cand_key, (uint32_t)e - 1), child)) {
                                atomicMin((unsigned long long*)&round_tab[s], (unsigned long long)mine);
                                slot = s;
                                break;
                            }
                        }
                    }
                }
                cand_slot[c] = slot;
            }
            __syncthreads();
            // ---- B: winners ----
            for (uint32_t c = tid; c < ncand; c += kGbThreads) {
                const uint32_t slot = cand_slot[c];
                if (slot == kGbNone) continue;
                if ((uint32_t)__ldcg(&round_tab[slot]) == c + 1) {
                    atomicOr(&sh.bitmap[c >> 5], 1u << (c & 31));
                    if ((int)(cand_meta[c] & 0xFF) < Lcur) atomicMin(&sh.tstar_c, c);
                    if constexpr (GOAL) {
                        const int64_t e = goal_find<W>(G, load_key<W>(cand_key, c));
                        if (e >= 0)
                            atomicMin(reinterpret_cast<unsigned long long*>(B + X.max_buckets),
                                      ((unsigned long long)c << 32) | (unsigned long long)e);
                    }
                }
            }
            __syncthreads();
            {
                // exclusive popcount prefix over the bitmap words (kGbCand/32 = 384 words, <= 2 per thread)
                constexpr int NWD = kGbCand / 32;
                uint32_t w0 = 0, w1 = 0;
                const int i0 = 2 * tid, i1 = 2 * tid + 1;
                if (i0 < NWD) w0 = __popc(sh.bitmap[i0]);
                if (i1 < NWD) w1 = __popc(sh.bitmap[i1]);
                uint32_t total;
                const uint32_t ex = gb_block_scan(w0 + w1, sh.scan_tmp, total);
                if (i0 < NWD) sh.prefix[i0] = ex;
                if (i1 < NWD) sh.prefix[i1] = ex + w0;
                if (tid == 0) sh.prefix[NWD] = total;
            }
            // the round table is cleared by the candidates that touched it
            for (uint32_t c = tid; c < ncand; c += kGbThreads) {
                const uint32_t slot = cand_slot[c];
                if (slot != kGbNone) round_tab[slot] = 0;
            }
            __syncthreads();
            // ---- C: decide (one thread; every thread then reads the outcome) ----
            if (tid == 0) {
                const uint32_t total = sh.prefix[kGbCand / 32];
                uint32_t limit = ncand, st2 = GB_CONT;
                if (n_nodes + total >= A.budget) {  // greedy.py:115-119: tested after a node's 12 children
                    uint32_t lo = 0, hi = Tn - 1;
                    bool hit = n_nodes + gb_rank(sh, ncand) >= A.budget;
                    if (hit) {
                        while (lo < hi) {
                            const uint32_t mid = (lo + hi) >> 1;
                            if (n_nodes + gb_rank(sh, (mid + 1) * 12) >= A.budget) hi = mid;
                            else lo = mid + 1;
                        }
                        limit = 12 * (lo + 1);
                        st2 = GB_BUDGET;
                    }
                }
                if (sh.tstar_c != kGbNone) {  // a new child with a smaller total length: the run ends after its parent
                    const uint32_t li = 12 * (sh.tstar_c / 12 + 1);
                    if (li < limit) {
                        limit = li;
                        st2 = GB_INTERRUPT;
                    }
                }
                const uint32_t ec = sh.err_c == kGbNone ? kGbNone : (sh.err_c >> 2);
                if (sh.sol_c != kGbNone && sh.sol_c < limit && sh.sol_c < ec) {
                    limit = sh.sol_c;
                    st2 = GB_SOLVED;
                } else if (ec != kGbNone && ec < limit) {
                    limit = ec;
                    st2 = GB_ERROR;
                }
                if constexpr (GOAL) {  // before every other event; on the solving child itself the solve wins
                    const uint32_t gc = (uint32_t)(*reinterpret_cast<unsigned long long*>(B + X.max_buckets) >> 32);
                    if (gc < limit) {  // kGbNone when no winner is a goal
                        limit = gc;
                        st2 = GB_GOAL;
                    }
                }
                sh.limit = limit;
                sh.stop = st2;
                sh.n_commit = gb_rank(sh, limit);
                sh.processed = (st2 == GB_SOLVED || st2 == GB_ERROR || (GOAL && st2 == GB_GOAL)) ? limit / 12 + 1 : limit / 12;
            }
            __syncthreads();
            const uint32_t limit = sh.limit;
            stop = sh.stop;
            const uint32_t processed = sh.processed;
            const bool goal_hit = GOAL && stop == GB_GOAL;
            // "New minimal length found" events in candidate order (greedy.py:82-85); replicated in every thread
            {
                const uint32_t gl = limit + (stop == GB_SOLVED || goal_hit ? 1u : 0u);
                for (;;) {
                    uint32_t best = kGbNone;
                    int bestL = -1;
                    for (int L = 0; L < min_len && L < 128; ++L) {
                        const uint32_t g = sh.first_len[L];
                        if (g < gl && g < best) {
                            best = g;
                            bestL = L;
                        }
                    }
                    if (bestL < 0) break;
                    min_len = bestL;
                    if (tid == 0 && n_minlen < 128) rec->minlen_log[n_minlen] = bestL;
                    ++n_minlen;
                }
            }
            // ---- D: commit the winners below the limit, in candidate order ----
            // (cand_slot is free again: it now receives each committed child's position inside its length group)
            for (uint32_t c = tid; c < ncand; c += kGbThreads) {
                uint32_t pos = kGbNone;
                if (c < limit && ((sh.bitmap[c >> 5] >> (c & 31)) & 1u)) {
                    const uint32_t L = cand_meta[c] & 0xFF;
                    const uint64_t idx = n_nodes + gb_rank(sh, c);
                    const Key<W> child = load_key<W>(cand_key, c);
                    store_key<W>(keys, idx, child);
                    const uint32_t pidx = (uint32_t)sortbuf[(size_t)(tile0 + c / 12) * RS + 2 * W];
                    parent[idx] = ((uint64_t)pidx << 4) | (uint64_t)(c % 12);
                    const uint64_t h = key_hash<W>(child);
                    const uint64_t v = ((h >> 40) << 40) | (idx + 1);
                    for (uint64_t s = h & tmask;; s = (s + 1) & tmask) {  // the key is absent: take the first free slot
                        if (__ldcg(&table[s]) == 0 &&
                            atomicCAS((unsigned long long*)&table[s], 0ull, (unsigned long long)v) == 0)
                            break;
                    }
                    pos = atomicAdd(&sh.cntL[L], 1u);
                }
                cand_slot[c] = pos;
            }
            __syncthreads();
            // ---- directory update: one segment per child length, appended to bucket (length, depth+1) ----
            if (tid == 0) {
                const uint32_t dnext = dcur + 1;
                for (int L = 0; L < 128; ++L) {
                    const uint32_t cnt = sh.cntL[L];
                    if (!cnt) continue;
                    if (sh.seg_used >= (uint32_t)kGbSegPool || (uint64_t)sh.f_end + cnt > X.fcap || dnext >= (1u << 24)) {
                        sh.fallback = sh.seg_used >= (uint32_t)kGbSegPool ? 3 : ((uint64_t)sh.f_end + cnt > X.fcap ? 4 : 6);
                        break;
                    }
                    const uint32_t sid = sh.seg_used++;
                    sh.segstart[L] = sh.f_end;
                    segs[sid] = GbSeg{sh.f_end, cnt, kGbNone, 0u};
                    sh.f_end += cnt;
                    const uint32_t key = ((uint32_t)L << 24) | dnext;
                    const int p = gb_find(B, sh.nb, key);
                    if (p < sh.nb && B[p].key == key) {
                        segs[B[p].seg_tail].next = sid;
                        B[p].seg_tail = sid;
                        B[p].count += cnt;
                    } else {
                        if (sh.nb >= X.max_buckets) {
                            sh.fallback = 5;  // directory full
                            break;
                        }
                        for (int i = sh.nb; i > p; --i) B[i] = B[i - 1];
                        B[p] = GbBucket{key, cnt, sid, sid};
                        sh.nb += 1;
                    }
                }
            }
            __syncthreads();
            if (sh.fallback) break;
            for (uint32_t c = tid; c < ncand; c += kGbThreads) {
                const uint32_t pos = cand_slot[c];
                if (pos == kGbNone) continue;
                const uint32_t L = cand_meta[c] & 0xFF;
                frontier[sh.segstart[L] + pos] = (uint32_t)(n_nodes + gb_rank(sh, c));
            }
            // ---- counters (replicated) ----
            n_nodes += sh.n_commit;
            n_expanded += processed;
            n_moves += (stop == GB_SOLVED || stop == GB_ERROR || goal_hit) ? (uint64_t)limit + 1 : (uint64_t)limit;
            if (processed > 0) {
                cur = (uint32_t)sortbuf[(size_t)(tile0 + processed - 1) * RS + 2 * W];
                if (stop != GB_SOLVED && stop != GB_ERROR && !goal_hit)
                    final_len = (int)(cand_meta[(processed - 1) * 12 + 11] & 0xFF);
            }
            done_nodes = tile0 + processed;
            if (stop == GB_SOLVED) {
                solved = 1;
                final_action = (int)(limit % 12);
                final_len = 2;
            } else if (goal_hit) {
                solved = 1;
                final_action = (int)(limit % 12);
                final_len = (int)(cand_meta[limit] & 0xFF);
            } else if (stop == GB_ERROR) {
                status = (int)(sh.err_c & 3);
            } else if (stop == GB_BUDGET) {
                budget_hit = 1;
            }
            __syncthreads();
        }
        if (sh.fallback) break;
        if (stop == GB_SOLVED || stop == GB_ERROR || stop == GB_BUDGET || (GOAL && stop == GB_GOAL)) {
            cur_rest = n - done_nodes;  // still in the reference's heap
            finished = true;
            break;
        }
        // ================= interrupted: the unexpanded rest goes back into its bucket =================
        if (done_nodes < n) {
            const uint32_t rest = n - done_nodes;
            __syncthreads();
            if (tid == 0) {
                if (sh.seg_used >= (uint32_t)kGbSegPool || (uint64_t)sh.f_end + rest > X.fcap || sh.nb >= X.max_buckets) {
                    sh.fallback = sh.seg_used >= (uint32_t)kGbSegPool ? 3 : ((uint64_t)sh.f_end + rest > X.fcap ? 4 : 5);
                } else {
                    const uint32_t sid = sh.seg_used++;
                    segs[sid] = GbSeg{sh.f_end, rest, kGbNone, 0u};
                    sh.segstart[0] = sh.f_end;
                    sh.f_end += rest;
                    const int p = gb_find(B, sh.nb, sh.cur_key);  // the bucket was removed when it was popped
                    for (int i = sh.nb; i > p; --i) B[i] = B[i - 1];
                    B[p] = GbBucket{sh.cur_key, rest, sid, sid};
                    sh.nb += 1;
                }
            }
            __syncthreads();
            if (sh.fallback) break;
            for (uint32_t i = tid; i < rest; i += kGbThreads)
                frontier[sh.segstart[0] + i] = (uint32_t)sortbuf[(size_t)(done_nodes + i) * RS + 2 * W];
            __syncthreads();
        }
    }
    __syncthreads();
    if (tid == 0) {
        uint64_t left = cur_rest;
        for (int i = 0; i < sh.nb; ++i) left += B[i].count;
        rec->solved = solved;
        rec->status = sh.fallback ? kGbFallback : status;
        rec->budget_hit = budget_hit;
        rec->n_minlen = min(n_minlen, 128);
        rec->n_nodes = n_nodes;
        rec->n_expanded = n_expanded;
        rec->n_moves = n_moves;
        rec->heap_left = left;
        rec->final_node = cur;
        rec->final_action = solved ? final_action : 11;
        rec->final_len = final_len;
        rec->rounds = sh.fallback ? -sh.fallback : rounds;
        rec->engine = 1;
        if constexpr (GOAL)  // -1 for a search handed back: it had not stopped
            rec->goal = solved && sh.stop == GB_GOAL
                            ? (int64_t)(*reinterpret_cast<unsigned long long*>(B + X.max_buckets) & 0xFFFFFFFFull)
                            : -1;
    }
}

}  // namespace acs
