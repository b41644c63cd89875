// pbfs.cu -- hash-partitioned breadth-first search of the AC graph, native driver.
//
// Contract (reference, paths relative to /root/reference): ac_solver/search/breadth_first.py:15-97
// -- FIFO order, children in action order, "solved" test before the visited test, budget test
// after each node's 12 children.  Result, visited ARRAY (order included), "New minimal length"
// sequence and counters are identical to the sequential reference for every world size.
//
// Design (B200-first; nothing here is host Python, and nothing in the chunk loop syncs with the
// host).  The visited set and the node store are partitioned by owner(state) = hash(key) -> rank.
// Nodes carry GLOBAL ids equal to their FIFO position.  The search advances in chunks of
// consecutive global ids [head, head+F); one chunk is this stream-ordered pipeline on every rank:
//
//   prep     local parent range [l0,l1) of the chunk, reset of cursors / control block / bitmap
//   expand   one thread per owned parent, a warp = 32 parents stepping through the 12 moves
//            together (uniform control flow).  Children are labelled with the chunk-local
//            candidate id c = 12*(gid-head)+action and appended to per-warp, per-destination
//            shared-memory queues; a full queue (32 records) is flushed with ONE coalesced
//            512-byte burst of peer stores straight into the owner rank's inbox over NVLink
//            (the compute step and the all-to-all are one kernel; there is no pack, no count
//            exchange and no send buffer).  Each (source, destination) pair owns a fixed inbox
//            region, so the write cursors are local atomics.
//   signal/wait   every rank stores its control block (minima for solved / raising child /
//            first occurrence of each total length, record counts) into every peer's control
//            inbox and publishes an epoch flag with st.release.sys; a one-block kernel spins on
//            the G flags with ld.acquire.sys (bounded by a timeout).  No NCCL, no host.
//   insert   owner side: one thread per received record; exact open-addressing table of 8-byte
//            slots probed a 32-byte sector (4 slots) at a time; "smallest candidate id wins" by
//            atomicMin on tentative slots.  A claim flips bit c of the winner bitmap, a displaced
//            claim flips it back (XOR is order independent), so no second pass over the table.
//   signal/wait
//   scan     OR of all ranks' winner bitmaps by peer loads, popcount prefix sums (global and
//            local) -> every winner's global id and local index
//   decide   one block, identical on every rank (replicated data => identical decisions): budget
//            cut by binary search in the prefix sums, solved / raising child, minimal-length
//            log, counters, next chunk.  Writes the device-resident state read by all kernels.
//   commit   winners below the limit are appended (key, parent link, global id) and their table
//            slots re-pointed at the node.
// Inboxes, control inboxes and bitmaps are double buffered by chunk parity, so a rank may run
// one pipeline stage ahead of its peers without overwriting what they still read.  The host
// enqueues chunk pipelines ahead of the device and only looks at a lagging copy of the state.
//
// One process per GPU: the exchange arena is shared with cudaIpc handles (acs_pbfs_export /
// acs_pbfs_connect); for tests all shards may also live in one process (acs_pbfs_connect_local),
// on one device (kernels of the shards are then serialised on one stream) or on several.
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
#include "bfs_common.cuh"

namespace acs {

constexpr int kPbMaxWorld = 16;
constexpr int kCtrlWords = 136;        // sol, err, first_len[128], log end, ierr, log start, pad
constexpr int kCtrlSol = 0, kCtrlErr = 1, kCtrlLen0 = 2, kCtrlCount = 130, kCtrlIerr = 131, kCtrlStart = 132;
// table slot: 23-bit fingerprint << 40 | (record-log position + 1); 0 = empty
constexpr uint64_t kPosMask = (1ull << 40) - 1;
// the per-destination log cursors are hot atomics: one per 256 bytes, so that they sit in different L2 lines / slices
constexpr int kCurStride = 32;

enum : int { IERR_LOG_FULL = 1, IERR_TABLE_FULL = 2, IERR_SHARD_FULL = 4, IERR_TIMEOUT = 8 };

// Device-resident run state of one rank.  Every scalar decision is replicated on all ranks.
struct PbState {
    // constants of the run
    int64_t budget, cap_local, chunk_cap, log_cap;
    uint64_t tmask;
    int32_t mrl, cyclical, world, rank;
    // current chunk
    int64_t head, F, n_nodes, n_local, l0, l1, level_end;
    uint64_t epoch;        // chunk counter, monotone across runs (flags carry it)
    int32_t buf, min_len, levels, done;
    // decided for the commit of the current chunk
    int64_t limit, n_nodes0, n_local0, head0;
    int32_t commit_pending, pad1;
    // results
    int64_t n_expanded, sol_gid, err_code, chunks;
    int32_t solved, budget_hit, status, ierr, n_minlen, pad0;
    int32_t minlen_log[128];
    unsigned long long records_sent, records_recv;  // statistics
};

// Pointers of one rank.  The "arena" part is visible to the peers (IPC or same process).
struct PbShard {
    PbState* st;
    uint64_t* nodes;     // [cap][2W+2]  owned nodes in FIFO order: key words, parent link, global id
    uint64_t* table;     // [tmask+1]
    uint4* rt;           // [words+1] rank table: {global prefix, global bits, local prefix, local bits}
    unsigned long long* cursors;     // [world * kCurStride] append positions in the peers' record logs (persist over a run)
    unsigned long long* cstart;      // [world] their values at the start of the current chunk
    unsigned long long* ctrl_local;  // [kCtrlWords]
    // arena (same layout on every rank)
    char* arena;                     // own
    char* peer[kPbMaxWorld];         // peer arenas as seen from this process
    int64_t off_flags;               // [3 kinds][world] u64
    int64_t off_ctrl;                // [2 buf][world][kCtrlWords] u64
    int64_t off_bitmap;              // [2 buf][bitmap_words] u32   this rank's winner bits
    int64_t off_bmg;                 // [bitmap_words] u32          all ranks' winner bits (filled slice-wise by the peers)
    int64_t off_bsums;               // [2][nblk] u32               popcounts per scan block (global, local)
    int64_t off_keys;                // [world src][log_cap][2W] u64   record log: state keys ...
    int64_t off_c;                   // [world src][log_cap] u32        ... and candidate ids
    int64_t bitmap_words, nblk;
    int32_t W, world, rank, pad;
};

__device__ __forceinline__ int64_t node_gid_rt(const uint64_t* nodes, int W, int64_t idx) {
    return (int64_t)nodes[idx * node_words(W) + 2 * W + 1];
}

__device__ __forceinline__ void st_release_sys(uint64_t* p, uint64_t v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_acquire_sys(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t global_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Owner rank of a state: a cheap 32-bit multiply-xor hash of the key words, a different function
// from pb_hash so that the owner is independent of the table slot and fingerprint bits.
template <int W>
__host__ __device__ __forceinline__ int pb_owner(const Key<W>& q, int world) {
    uint32_t x = 0x9E3779B9u;
#pragma unroll
    for (int i = 0; i < 2 * W; ++i) {
        x = (x ^ (uint32_t)q.k[i]) * 0x85EBCA6Bu;
        x = (x ^ (x >> 15) ^ (uint32_t)(q.k[i] >> 32)) * 0xC2B2AE35u;
    }
    x ^= x >> 16;
    x *= 0x7FEB352Du;
    x ^= x >> 15;
    return (int)(((uint64_t)x * (uint32_t)world) >> 32);
}


__device__ __forceinline__ uint64_t* sh_flags(const PbShard& S, char* base, int kind) {
    return reinterpret_cast<uint64_t*>(base + S.off_flags) + kind * S.world;
}
__device__ __forceinline__ unsigned long long* sh_ctrl(const PbShard& S, char* base, int buf, int src) {
    return reinterpret_cast<unsigned long long*>(base + S.off_ctrl) + ((int64_t)buf * S.world + src) * kCtrlWords;
}
__device__ __forceinline__ uint32_t* sh_bitmap(const PbShard& S, char* base, int buf) {
    return reinterpret_cast<uint32_t*>(base + S.off_bitmap) + (int64_t)buf * S.bitmap_words;
}
__device__ __forceinline__ uint32_t* sh_bmg(const PbShard& S, char* base) {
    return reinterpret_cast<uint32_t*>(base + S.off_bmg);
}
__device__ __forceinline__ uint32_t* sh_bsums(const PbShard& S, char* base) {
    return reinterpret_cast<uint32_t*>(base + S.off_bsums);
}
__device__ __forceinline__ uint64_t* sh_keys(const PbShard& S, char* base) {
    return reinterpret_cast<uint64_t*>(base + S.off_keys);
}
__device__ __forceinline__ uint32_t* sh_c(const PbShard& S, char* base) {
    return reinterpret_cast<uint32_t*>(base + S.off_c);
}

// ---- prep ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pb_prep_kernel(const PbShard S) {
    PbState* st = S.st;
    if (blockIdx.x == 0 && threadIdx.x == 0) st->commit_pending = 0;  // set again by this chunk's decide
    if (st->done) return;
    const int64_t nwords = (12 * st->F + 31) / 32;
    uint32_t* bm = sh_bitmap(S, S.arena, st->buf);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += (int64_t)gridDim.x * blockDim.x)
        bm[i] = 0;
    if (blockIdx.x != 0) return;
    if (threadIdx.x < S.world) S.cstart[threadIdx.x] = S.cursors[threadIdx.x * kCurStride];
    if (threadIdx.x < kCtrlWords)
        S.ctrl_local[threadIdx.x] = (threadIdx.x == kCtrlCount || threadIdx.x == kCtrlIerr) ? 0ull : ~0ull;
    if (threadIdx.x == 0) {
        // owned parents of [head, head+F): gid[] is increasing, the range starts where the last ended
        const int64_t l0 = st->l1, want = st->head + st->F;
        int64_t lo = l0, hi = st->n_local;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (node_gid_rt(S.nodes, S.W, mid) < want) lo = mid + 1;
            else hi = mid;
        }
        st->l0 = l0;
        st->l1 = lo;
    }
}

// ---- expand ----------------------------------------------------------------------------------
// Per-warp staging in shared memory: kStage records (key, candidate id, destination rank) in
// generation order, a second buffer of the same size for the destination-sorted copy, and the
// per-destination counters of the flush.  The size does not depend on the world size.
constexpr int kStage = 128;
#ifndef PB_UNROLL
#define PB_UNROLL 4
#endif
constexpr int kPbUnroll = PB_UNROLL;  // of the 12-move loop in the expansion kernel
template <int W>
__host__ __device__ constexpr int stage_bytes_per_warp() {
    return 2 * kStage * (16 * W + 4 + 4) + kPbMaxWorld * (4 + 4 + 8);
}
extern __shared__ __align__(16) unsigned char pb_smem[];
template <int W>
struct Stage {
    ulonglong2* keys;  // [kStage][W]
    uint32_t* c;       // [kStage]
    uint32_t* dest;    // [kStage]
    ulonglong2* keys2;
    uint32_t* c2;
    uint32_t* dest2;
    uint32_t* cnt;     // [kPbMaxWorld]
    uint32_t* off;     // [kPbMaxWorld]
    unsigned long long* gpos;  // [kPbMaxWorld]
    __device__ __forceinline__ explicit Stage(int wib) {
        unsigned char* p = pb_smem + wib * stage_bytes_per_warp<W>();
        keys = reinterpret_cast<ulonglong2*>(p);
        keys2 = reinterpret_cast<ulonglong2*>(p + kStage * 16 * W);
        gpos = reinterpret_cast<unsigned long long*>(p + 2 * kStage * 16 * W);
        uint32_t* q = reinterpret_cast<uint32_t*>(p + 2 * kStage * 16 * W + kPbMaxWorld * 8);
        c = q;
        dest = q + kStage;
        c2 = q + 2 * kStage;
        dest2 = q + 3 * kStage;
        cnt = q + 4 * kStage;
        off = cnt + kPbMaxWorld;
    }
};
// block-wide: where this rank's records go in every destination's log
struct DestBase {
    ulonglong2* keys[kPbMaxWorld];
    uint32_t* c[kPbMaxWorld];
};

// Flush the n staged records of this warp: a counting sort by destination rank in shared memory,
// ONE atomic instruction reserving space in all destination logs (local atomics: every (source,
// destination) pair has its own log), then runs of coalesced stores straight into the
// destinations' memory -- peer stores over NVLink when the destination is another GPU.  This is
// the all-to-all of the search, fused into the expansion kernel.
template <int W>
__device__ __noinline__ void pb_flush(const PbShard& S, const DestBase* DB, int wib, uint32_t n, int lane,
                                      int64_t log_cap, int world) {
    Stage<W> Q(wib);
    if (world == 1) {
        unsigned long long pos = 0;
        if (lane == 0) pos = atomicAdd(&S.cursors[0], (unsigned long long)n);
        pos = __shfl_sync(0xFFFFFFFFu, pos, 0);
        if (pos + n > (unsigned long long)log_cap) {
            if (lane == 0) atomicOr(&S.ctrl_local[kCtrlIerr], (unsigned long long)IERR_LOG_FULL);
        } else {
            ulonglong2* dk = DB->keys[0] + pos * W;
            uint32_t* dc = DB->c[0] + pos;
#pragma unroll
            for (int r = 0; r < kStage / 32; ++r) {
                const uint32_t idx = r * 32 + lane;
                if (idx < n) {
#pragma unroll
                    for (int i = 0; i < W; ++i) dk[(size_t)idx * W + i] = Q.keys[idx * W + i];
                    dc[idx] = Q.c[idx];
                }
            }
        }
        __syncwarp();
        return;
    }
    if (lane < kPbMaxWorld) Q.cnt[lane] = 0;
    __syncwarp();
    uint32_t d[kStage / 32], rk[kStage / 32];
#pragma unroll
    for (int r = 0; r < kStage / 32; ++r) {
        const uint32_t idx = r * 32 + lane;
        d[r] = 0;
        rk[r] = 0;
        if (idx < n) {
            d[r] = Q.dest[idx];
            rk[r] = atomicAdd(&Q.cnt[d[r]], 1u);
        }
    }
    __syncwarp();
    {
        // lanes < world: exclusive prefix of the counts (position in the sorted buffer) and the log reservation
        const uint32_t cnt = lane < world ? Q.cnt[lane] : 0u;
        uint32_t x = cnt;
#pragma unroll
        for (int o = 1; o < kPbMaxWorld; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, x, o);
            if (lane >= o) x += t;
        }
        if (lane < world) {
            Q.off[lane] = x - cnt;
            unsigned long long pos = ~0ull;
            if (cnt) {
                pos = atomicAdd(&S.cursors[lane * kCurStride], (unsigned long long)cnt);
                if (pos + cnt > (unsigned long long)log_cap) {
                    atomicOr(&S.ctrl_local[kCtrlIerr], (unsigned long long)IERR_LOG_FULL);
                    pos = ~0ull;
                }
            }
            Q.gpos[lane] = pos;
        }
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < kStage / 32; ++r) {
        const uint32_t idx = r * 32 + lane;
        if (idx < n) {
            const uint32_t t = Q.off[d[r]] + rk[r];
#pragma unroll
            for (int i = 0; i < W; ++i) Q.keys2[t * W + i] = Q.keys[idx * W + i];
            Q.c2[t] = Q.c[idx];
            Q.dest2[t] = d[r];
        }
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < kStage / 32; ++r) {
        const uint32_t t = r * 32 + lane;
        if (t < n) {
            const uint32_t dd = Q.dest2[t];
            const unsigned long long pos = Q.gpos[dd];
            if (pos != ~0ull) {
                const unsigned long long o = pos + (t - Q.off[dd]);
                ulonglong2* dk = DB->keys[dd] + o * W;
#pragma unroll
                for (int i = 0; i < W; ++i) dk[i] = Q.keys2[t * W + i];
                DB->c[dd][o] = Q.c2[t];
            }
        }
    }
    __syncwarp();
}

template <int W, bool TRUSTED>
__global__ void __launch_bounds__(256) pb_expand_kernel(const PbShard S, int warps_per_block) {
    const PbState* st = S.st;
    if (st->done) return;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int world = S.world;
    __shared__ DestBase DB;
    const int64_t l1 = st->l1, log_cap = st->log_cap;
    if (threadIdx.x < world) {
        char* base = S.peer[threadIdx.x];
        DB.keys[threadIdx.x] = reinterpret_cast<ulonglong2*>(sh_keys(S, base)) + (int64_t)S.rank * log_cap * W;
        DB.c[threadIdx.x] = sh_c(S, base) + (int64_t)S.rank * log_cap;
    }
    __syncthreads();
    Stage<W> Q(wib);
    ulonglong2* sk = Q.keys;
    uint32_t* sc = Q.c;
    uint32_t* sd = Q.dest;
    const uint64_t head = (uint64_t)st->head;
    const int mrl = st->mrl;
    const bool cyc = st->cyclical != 0;
    const int min_len = st->min_len;
    const int64_t gw = (int64_t)blockIdx.x * warps_per_block + wib, nw = (int64_t)gridDim.x * warps_per_block;
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t staged = 0;  // warp-uniform
    unsigned long long sent = 0;
    for (int64_t base = st->l0 + 32 * gw; base < l1; base += 32 * nw) {
        const int64_t j = base + lane;
        const bool valid = j < l1;
        Key<W> pk;
#pragma unroll
        for (int i = 0; i < 2 * W; ++i) pk.k[i] = 0;
        uint64_t pg = 0;
        uint32_t skip = 0;  // moves of this node whose child is certainly a duplicate of an EARLIER candidate
        if (valid) {
            int64_t pl, gj;
            node_load<W>(S.nodes, (uint64_t)j, pk, pl, gj);
            pg = (uint64_t)gj;
            skip = skip_moves<TRUSTED>(pl, cyc);
        }
        Rel<2 * W> p0, p1;
        split_key<W>(pk, p0, p1);
        const uint32_t cbase = (uint32_t)((pg - head) * 12);
        const uint64_t gbase = pg * 12;
#pragma unroll kPbUnroll
        for (int a = 0; a < 12; ++a) {
            Rel<2 * W> r0 = p0, r1 = p1;
            bool emit = false;
            Key<W> child;
#pragma unroll
            for (int i = 0; i < 2 * W; ++i) child.k[i] = 0;
            if (valid && !((skip >> a) & 1u)) {
                bool co;
                const int stt = apply_move<2 * W, TRUSTED>(r0, r1, a, mrl, cyc, co);
                if (stt != ST_OK) {
                    atomicMin(&S.ctrl_local[kCtrlErr], (unsigned long long)(((gbase + a) << 2) | (unsigned)stt));
                } else {
                    const int L = r0.len + r1.len;
                    if (L < min_len) atomicMin(&S.ctrl_local[kCtrlLen0 + L], (unsigned long long)(gbase + a));
                    if (L == 2) atomicMin(&S.ctrl_local[kCtrlSol], (unsigned long long)(gbase + a));  // before the visited test
                    child = make_key<W>(r0, r1);
                    emit = !key_eq<W>(child, pk);
                }
            }
            const uint32_t act = __ballot_sync(0xFFFFFFFFu, emit);
            if (emit) {
                const uint32_t q = staged + __popc(act & lt);
#pragma unroll
                for (int i = 0; i < W; ++i) sk[q * W + i] = make_ulonglong2(child.k[2 * i], child.k[2 * i + 1]);
                sc[q] = cbase + a;
                if (world > 1) sd[q] = (uint32_t)pb_owner<W>(child, world);
            }
            staged += __popc(act);
            if (staged > kStage - 32) {
                __syncwarp();
                pb_flush<W>(S, &DB, wib, staged, lane, log_cap, world);
                sent += staged;
                staged = 0;
            }
        }
    }
    if (staged) {
        __syncwarp();
        pb_flush<W>(S, &DB, wib, staged, lane, log_cap, world);
        sent += staged;
    }
    // the peer stores of this thread are performed before anything a later kernel publishes
    __threadfence_system();
    if (lane == 0 && sent) atomicAdd(&S.st->records_sent, sent);
}

// ---- expand, block-level staging (world > 1) -------------------------------------------------
// The per-warp flush above sends ~16 records per destination at a time: 256-byte key runs and
// 64-byte id runs at arbitrary alignment, i.e. NVLink write packets of ~60 bytes with byte enables.
// Here the whole block stages the children of kCtaMoves moves of its 32*warps parents (up to
// 32*warps*kCtaMoves records), sorts them by destination rank with a counting sort over all
// threads and sends one run per destination: ~1 KB of keys per run on the AC(3) workload, mostly
// whole 128-byte lines.  Same records, same logs, same cursors as the per-warp path.
constexpr int kCtaMoves = 4;  // moves per flush (the 12-move loop is unrolled by the same factor)
template <int W>
__host__ __device__ constexpr int cta_stage_bytes(int warps) {
    // keys | candidate ids | sorted order (u16) | destination (u8) | counters
    return warps * 32 * kCtaMoves * (16 * W + 4 + 2 + 1) + kPbMaxWorld * (4 + 4 + 8) + 16;
}
template <int W>
struct CtaStage {
    ulonglong2* keys;
    uint32_t* c;
    uint16_t* perm;
    uint8_t* dest;
    unsigned long long* gpos;
    uint32_t* cnt;
    uint32_t* off;
    uint32_t* total;
    __device__ __forceinline__ explicit CtaStage(int warps) {
        const int cap = warps * 32 * kCtaMoves;
        unsigned char* p = pb_smem;
        keys = reinterpret_cast<ulonglong2*>(p);
        p += (size_t)cap * 16 * W;
        gpos = reinterpret_cast<unsigned long long*>(p);
        p += kPbMaxWorld * 8;
        c = reinterpret_cast<uint32_t*>(p);
        p += (size_t)cap * 4;
        cnt = reinterpret_cast<uint32_t*>(p);
        p += kPbMaxWorld * 4;
        off = reinterpret_cast<uint32_t*>(p);
        p += kPbMaxWorld * 4;
        total = reinterpret_cast<uint32_t*>(p);
        p += 16;
        perm = reinterpret_cast<uint16_t*>(p);
        p += (size_t)cap * 2;
        dest = p;
    }
};

// all threads of the block; *Q.total records are staged.  Leaves *Q.total == 0 and cnt[] == 0.
template <int W>
__device__ __forceinline__ void pb_flush_cta(const PbShard& S, const DestBase* DB, const CtaStage<W>& Q, int64_t log_cap,
                                             int world) {
    constexpr int kMaxPer = kCtaMoves;  // records per thread: cap / threads = 32*warps*kCtaMoves / (32*warps)
    __syncthreads();  // every warp's records of this batch are staged
    const uint32_t n = *Q.total;
    const int tid = threadIdx.x, nt = blockDim.x;
    uint32_t d[kMaxPer], rk[kMaxPer];
#pragma unroll
    for (int r = 0; r < kMaxPer; ++r) {
        const uint32_t idx = r * nt + tid;
        d[r] = 0;
        rk[r] = 0;
        if (idx < n) {
            d[r] = Q.dest[idx];
            rk[r] = atomicAdd(&Q.cnt[d[r]], 1u);
        }
    }
    __syncthreads();
    if (tid < 32) {
        const uint32_t cnt = tid < world ? Q.cnt[tid] : 0u;
        uint32_t x = cnt;
#pragma unroll
        for (int o = 1; o < kPbMaxWorld; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, x, o);
            if (tid >= o) x += t;
        }
        if (tid < world) {
            Q.off[tid] = x - cnt;
            unsigned long long pos = ~0ull;
            if (cnt) {
                pos = atomicAdd(&S.cursors[tid * kCurStride], (unsigned long long)cnt);
                if (pos + cnt > (unsigned long long)log_cap) {
                    atomicOr(&S.ctrl_local[kCtrlIerr], (unsigned long long)IERR_LOG_FULL);
                    pos = ~0ull;
                }
            }
            Q.gpos[tid] = pos;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kMaxPer; ++r) {
        const uint32_t idx = r * nt + tid;
        if (idx < n) Q.perm[Q.off[d[r]] + rk[r]] = (uint16_t)idx;
    }
    __syncthreads();
    if (tid < kPbMaxWorld) Q.cnt[tid] = 0;  // for the next flush (read again only after its first barrier)
    if (tid == 0) *Q.total = 0;
    for (uint32_t t = tid; t < n; t += nt) {
        const uint32_t idx = Q.perm[t];
        const uint32_t dd = Q.dest[idx];
        const unsigned long long pos = Q.gpos[dd];
        if (pos != ~0ull) {
            const unsigned long long o = pos + (t - Q.off[dd]);
            ulonglong2* dk = DB->keys[dd] + o * W;
#pragma unroll
            for (int i = 0; i < W; ++i) dk[i] = Q.keys[idx * W + i];
            DB->c[dd][o] = Q.c[idx];
        }
    }
    __syncthreads();  // the staging area is free again
}

template <int W, bool TRUSTED>
__global__ void __launch_bounds__(512) pb_expand_cta_kernel(const PbShard S) {
    const PbState* st = S.st;
    if (st->done) return;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const int world = S.world;
    __shared__ DestBase DB;
    const int64_t l1 = st->l1, log_cap = st->log_cap;
    CtaStage<W> Q(warps);
    if (threadIdx.x < world) {
        char* base = S.peer[threadIdx.x];
        DB.keys[threadIdx.x] = reinterpret_cast<ulonglong2*>(sh_keys(S, base)) + (int64_t)S.rank * log_cap * W;
        DB.c[threadIdx.x] = sh_c(S, base) + (int64_t)S.rank * log_cap;
    }
    if (threadIdx.x < kPbMaxWorld) Q.cnt[threadIdx.x] = 0;
    if (threadIdx.x == 0) *Q.total = 0;
    __syncthreads();
    const uint64_t head = (uint64_t)st->head;
    const int mrl = st->mrl;
    const bool cyc = st->cyclical != 0;
    const int min_len = st->min_len;
    const uint32_t lt = (1u << lane) - 1u;
    unsigned long long sent = 0;
    // block-uniform trip count: the block's 32*warps consecutive parents per round
    for (int64_t bbase = st->l0 + (int64_t)blockIdx.x * 32 * warps; bbase < l1; bbase += (int64_t)gridDim.x * 32 * warps) {
        const int64_t j = bbase + 32 * wib + lane;
        const bool valid = j < l1;
        Key<W> pk;
#pragma unroll
        for (int i = 0; i < 2 * W; ++i) pk.k[i] = 0;
        uint64_t pg = 0;
        uint32_t skip = 0;  // see skip_moves
        if (valid) {
            int64_t pl, gj;
            node_load<W>(S.nodes, (uint64_t)j, pk, pl, gj);
            pg = (uint64_t)gj;
            skip = skip_moves<TRUSTED>(pl, cyc);
        }
        Rel<2 * W> p0, p1;
        split_key<W>(pk, p0, p1);
        const uint32_t cbase = (uint32_t)((pg - head) * 12);
        const uint64_t gbase = pg * 12;
#pragma unroll 1
        for (int a0 = 0; a0 < 12; a0 += kCtaMoves) {
#pragma unroll
            for (int aa = 0; aa < kCtaMoves; ++aa) {
                const int a = a0 + aa;
                Rel<2 * W> r0 = p0, r1 = p1;
                bool emit = false;
                Key<W> child;
#pragma unroll
                for (int i = 0; i < 2 * W; ++i) child.k[i] = 0;
                if (valid && !((skip >> a) & 1u)) {
                    bool co;
                    const int stt = apply_move<2 * W, TRUSTED>(r0, r1, a, mrl, cyc, co);
                    if (stt != ST_OK) {
                        atomicMin(&S.ctrl_local[kCtrlErr], (unsigned long long)(((gbase + a) << 2) | (unsigned)stt));
                    } else {
                        const int L = r0.len + r1.len;
                        if (L < min_len) atomicMin(&S.ctrl_local[kCtrlLen0 + L], (unsigned long long)(gbase + a));
                        if (L == 2) atomicMin(&S.ctrl_local[kCtrlSol], (unsigned long long)(gbase + a));  // before the visited test
                        child = make_key<W>(r0, r1);
                        emit = !key_eq<W>(child, pk);
                    }
                }
                const uint32_t act = __ballot_sync(0xFFFFFFFFu, emit);
                uint32_t wbase = 0;
                if (lane == 0 && act) wbase = atomicAdd(Q.total, (uint32_t)__popc(act));
                wbase = __shfl_sync(0xFFFFFFFFu, wbase, 0);
                if (emit) {
                    const uint32_t q = wbase + __popc(act & lt);
#pragma unroll
                    for (int i = 0; i < W; ++i) Q.keys[q * W + i] = make_ulonglong2(child.k[2 * i], child.k[2 * i + 1]);
                    Q.c[q] = cbase + a;
                    Q.dest[q] = (uint8_t)pb_owner<W>(child, world);
                }
                sent += __popc(act);
            }
            pb_flush_cta<W>(S, &DB, Q, log_cap, world);
        }
    }
    __threadfence_system();
    if (lane == 0 && sent) atomicAdd(&S.st->records_sent, sent);
}

// ---- signal / wait ---------------------------------------------------------------------------
// kind 0: "my records and control block for this chunk are in your inbox"
// kind 1: "my winner bitmap for this chunk is final"
__global__ void __launch_bounds__(256) pb_signal_kernel(const PbShard S, int kind) {
    const PbState* st = S.st;
    if (st->done) return;
    const int world = S.world;
    if (kind == 0) {
        for (int i = threadIdx.x; i < world * kCtrlWords; i += blockDim.x) {
            const int d = i / kCtrlWords, w = i % kCtrlWords;
            unsigned long long v = S.ctrl_local[w];
            if (w == kCtrlCount) v = S.cursors[d * kCurStride];
            if (w == kCtrlStart) v = S.cstart[d];
            if (w == kCtrlIerr) v |= (unsigned long long)st->ierr;
            sh_ctrl(S, S.peer[d], st->buf, S.rank)[w] = v;
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < world) st_release_sys(sh_flags(S, S.peer[threadIdx.x], kind) + S.rank, st->epoch + 1);
}

__global__ void __launch_bounds__(32) pb_wait_kernel(const PbShard S, int kind, unsigned long long timeout_ns) {
    PbState* st = S.st;
    if (st->done) return;
    if (threadIdx.x < S.world) {
        const uint64_t* f = sh_flags(S, S.arena, kind) + threadIdx.x;
        const uint64_t want = st->epoch + 1;
        const uint64_t t0 = global_ns();
        while (ld_acquire_sys(f) < want) {
            if (global_ns() - t0 > timeout_ns) {
                atomicOr(&st->ierr, IERR_TIMEOUT);
                break;
            }
            __nanosleep(200);
        }
    }
}

// ---- insert ----------------------------------------------------------------------------------
// The records of a chunk are the tails [start, end) of the per-source record logs.
struct RegionMap {
    unsigned long long vstart[kPbMaxWorld + 1];  // prefix of the per-source record counts of this chunk
    unsigned long long cstart[kPbMaxWorld];      // log offset of each source's first record of this chunk
};
__device__ __forceinline__ void load_regions(const PbShard& S, const PbState* st, int buf, RegionMap* R) {
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int s = 0; s < S.world; ++s) {
            const unsigned long long* ctrl = sh_ctrl(S, S.arena, buf, s);
            unsigned long long lo = __ldcg(&ctrl[kCtrlStart]), hi = __ldcg(&ctrl[kCtrlCount]);
            if (hi > (unsigned long long)st->log_cap) hi = (unsigned long long)st->log_cap;  // overflow is flagged by the sender
            if (lo > hi) lo = hi;
            R->vstart[s] = run;
            R->cstart[s] = lo;
            run += hi - lo;
        }
        for (int s = S.world; s <= kPbMaxWorld; ++s) R->vstart[s] = run;
    }
    __syncthreads();
}
// does log position p belong to the current chunk (a tentative entry)?
__device__ __forceinline__ bool is_tentative(const RegionMap* R, int world, int64_t log_cap, uint64_t p) {
    int s = 0;
#pragma unroll 1
    for (int k = 1; k < world; ++k) s += (p >= (uint64_t)k * (uint64_t)log_cap) ? 1 : 0;
    return p - (uint64_t)s * (uint64_t)log_cap >= R->cstart[s];
}

// The insert is bound by the number of divergent memory requests (see above), so it is written
// for few of them: per record one bucket load, one log-key load per fingerprint match, one CAS
// per claim; the winner-bitmap atomics of a warp fall into a few sectors (candidate ids of
// consecutive log records are close), the record itself is read coalesced.
template <int W>
__global__ void __launch_bounds__(256) pb_insert_kernel(const PbShard S) {
    PbState* st = S.st;
    if (st->done) return;
    __shared__ RegionMap R;
    load_regions(S, st, st->buf, &R);
    const unsigned long long total = R.vstart[S.world];
    const int64_t log_cap = st->log_cap;
    const int world = S.world;
    const uint64_t* in_keys = sh_keys(S, S.arena);
    const uint32_t* in_c = sh_c(S, S.arena);
    uint32_t* bm = sh_bitmap(S, S.arena, st->buf);
    const uint64_t tmask = st->tmask;
    if (blockIdx.x == 0 && threadIdx.x == 0) st->records_recv += total;
    // Every block works on ONE source log (block b on source b mod G), so all G logs are walked at the same
    // time and at the same pace: candidate ids grow along every log, hence the G walks touch the same moving
    // window of the winner bitmap (here) and of the rank table (commit) -- it is read from HBM once per chunk,
    // not once per source.  No per-record search for the source region either.
    {
    const int src = (int)(blockIdx.x % (unsigned)world);
    const unsigned long long bsrc = blockIdx.x / (unsigned)world;
    const unsigned long long nbsrc = (gridDim.x - (unsigned)src + (unsigned)world - 1u) / (unsigned)world;
    const unsigned long long n_src = R.vstart[src + 1] - R.vstart[src];
    const int64_t base_src = (int64_t)src * log_cap + (int64_t)R.cstart[src];
    for (unsigned long long v = bsrc * blockDim.x + threadIdx.x; v < n_src; v += nbsrc * blockDim.x) {
        const int64_t i = base_src + (int64_t)v;
        const Key<W> key = load_key_cg<W>(in_keys, (uint64_t)i);
        const uint32_t c = __ldcg(in_c + i);
        const uint64_t h = pb_hash<W>(key);
        const uint64_t fp23 = h >> 41;
        const uint64_t mine = (fp23 << 40) | ((uint64_t)i + 1);
        uint64_t s = (h & tmask) & ~3ull;
        uint64_t probes = 0;
        bool finished = false;
        while (!finished) {
            uint64_t vv[4];
            load_bucket(S.table + s, vv);
#pragma unroll
            for (int jj = 0; jj < 4 && !finished; ++jj) {
                uint64_t cur = vv[jj];
                unsigned long long* slot = (unsigned long long*)&S.table[s + jj];
                if (cur == 0) {
                    cur = atomicCAS(slot, 0ull, (unsigned long long)mine);
                    if (cur == 0) {  // first sighting of this state: claim
                        atomicXor(&bm[c >> 5], 1u << (c & 31));
                        finished = true;
                        break;
                    }
                }
                if ((cur >> 40) != fp23) continue;
                uint64_t p2 = (cur & kPosMask) - 1;
                const Key<W> other = load_key_cg<W>(in_keys, p2);
                if (!key_eq<W>(other, key)) continue;
                // the same state: an older chunk's record (visited), or a record of this chunk --
                // then the smaller candidate id keeps the slot (FIFO order of the reference)
                if (is_tentative(&R, world, log_cap, p2)) {
                    for (;;) {
                        const uint32_t c2 = __ldcg(in_c + p2);
                        if (c2 < c) break;
                        const uint64_t old = atomicCAS(slot, (unsigned long long)cur, (unsigned long long)mine);
                        if (old == cur) {  // displaced the holder: its claim bit flips back, mine flips on
                            atomicXor(&bm[c2 >> 5], 1u << (c2 & 31));
                            atomicXor(&bm[c >> 5], 1u << (c & 31));
                            break;
                        }
                        cur = old;  // someone else replaced it meanwhile (same state): look again
                        p2 = (cur & kPosMask) - 1;
                    }
                }
                finished = true;
            }
            if (!finished) {
                s = (s + 4) & tmask;
                probes += 4;
                if (probes > tmask) {  // cannot happen with the chunk sizing (table <= 3/4 full)
                    atomicOr(&st->ierr, IERR_TABLE_FULL);
                    finished = true;
                }
            }
        }
    }
    }
}

// ---- scan ------------------------------------------------------------------------------------
__device__ __forceinline__ void block_sum2(uint32_t& a, uint32_t& b) {
    __shared__ uint32_t wa[kScanT / 32], wb[kScanT / 32];
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        a += __shfl_xor_sync(0xFFFFFFFFu, a, off);
        b += __shfl_xor_sync(0xFFFFFFFFu, b, off);
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) {
        wa[wid] = a;
        wb[wid] = b;
    }
    __syncthreads();
    a = b = 0;
#pragma unroll
    for (int w = 0; w < kScanT / 32; ++w) {
        a += wa[w];
        b += wb[w];
    }
}
// Winner bits of all ranks, reduce-scatter / all-gather over peer memory: scan block b is combined
// by rank b % world (OR of the G local bitmaps, peer loads) and the result stored into EVERY
// rank's global bitmap together with its popcount, so a rank moves 2*(G-1)/G of a bitmap over
// NVLink per chunk instead of reading G-1 whole bitmaps.  The local popcounts need no exchange.
__global__ void __launch_bounds__(kScanT) pb_scan_sums_kernel(const PbShard S) {
    const PbState* st = S.st;
    if (st->done) return;
    const int64_t nwords = (12 * st->F + 31) / 32;
    const int64_t nblk = (nwords + kScanBlock - 1) / kScanBlock;
    const uint32_t* mine = sh_bitmap(S, S.arena, st->buf);
    uint32_t* my_sums = sh_bsums(S, S.arena);
    for (int64_t b = blockIdx.x; b < nblk; b += gridDim.x) {
        const bool combine = (int)(b % S.world) == S.rank;
        uint32_t sg = 0, sl = 0;
        uint32_t g[kScanPer];
#pragma unroll
        for (int k = 0; k < kScanPer; ++k) {
            const int64_t i = b * kScanBlock + (int64_t)k * kScanT + threadIdx.x;
            g[k] = i < nwords ? __ldcg(mine + i) : 0u;
            sl += __popc(g[k]);
        }
        if (combine) {
            // peer loads in batches of four ranks: 32 independent NVLink loads per thread are in flight
            // before the first one is consumed (one round trip per batch instead of one per peer)
            for (int r0 = 0; r0 < S.world; r0 += 4) {
                uint32_t t[4][kScanPer];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int r = r0 + q;
                    const bool on = r < S.world && r != S.rank;
                    const uint32_t* pb = sh_bitmap(S, S.peer[on ? r : S.rank], st->buf);
#pragma unroll
                    for (int k = 0; k < kScanPer; ++k) {
                        const int64_t i = b * kScanBlock + (int64_t)k * kScanT + threadIdx.x;
                        t[q][k] = (on && i < nwords) ? __ldcv(pb + i) : 0u;
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int k = 0; k < kScanPer; ++k) g[k] |= t[q][k];
            }
            for (int r = 0; r < S.world; ++r) {
                uint32_t* pg = sh_bmg(S, S.peer[r]);
#pragma unroll
                for (int k = 0; k < kScanPer; ++k) {
                    const int64_t i = b * kScanBlock + (int64_t)k * kScanT + threadIdx.x;
                    if (i < nwords) pg[i] = g[k];
                }
            }
#pragma unroll
            for (int k = 0; k < kScanPer; ++k) sg += __popc(g[k]);
        }
        block_sum2(sg, sl);
        if (threadIdx.x == 0) {
            my_sums[S.nblk + b] = sl;
            if (combine)
                for (int r = 0; r < S.world; ++r) sh_bsums(S, S.peer[r])[b] = sg;
        }
        __syncthreads();
    }
    __threadfence_system();
}
// single block: exclusive scans of both block-sum arrays in place; totals to the last rank-table entry
__global__ void __launch_bounds__(kScanT) pb_scan_top_kernel(const PbShard S) {
    const PbState* st = S.st;
    if (st->done) return;
    const int64_t nwords = (12 * st->F + 31) / 32;
    const int64_t nblk = (nwords + kScanBlock - 1) / kScanBlock;
    uint32_t tot[2] = {0, 0};
    for (int which = 0; which < 2; ++which) {
        uint32_t* sums = sh_bsums(S, S.arena) + which * S.nblk;
        uint32_t carry = 0;
        for (int64_t base = 0; base < nblk; base += kScanT) {
            const int64_t i = base + threadIdx.x;
            const uint32_t v = i < nblk ? __ldcg(sums + i) : 0u;
            uint32_t total;
            const uint32_t ex = block_excl_scan(v, total);
            if (i < nblk) sums[i] = carry + ex;
            carry += total;
            __syncthreads();
        }
        tot[which] = carry;
    }
    if (threadIdx.x == 0) S.rt[nwords] = make_uint4(tot[0], 0u, tot[1], 0u);
}
// rank table: per bitmap word {winners before it (all ranks), its bits (all ranks), same for this rank}
__global__ void __launch_bounds__(kScanT) pb_scan_final_kernel(const PbShard S) {
    const PbState* st = S.st;
    if (st->done) return;
    const int64_t nwords = (12 * st->F + 31) / 32;
    const int64_t nblk = (nwords + kScanBlock - 1) / kScanBlock;
    const uint32_t* loc = sh_bitmap(S, S.arena, st->buf);
    const uint32_t* glob = sh_bmg(S, S.arena);
    const uint32_t* sums = sh_bsums(S, S.arena);
    for (int64_t b = blockIdx.x; b < nblk; b += gridDim.x) {
        const int64_t first = b * kScanBlock + (int64_t)threadIdx.x * kScanPer;
        uint32_t wg[kScanPer], wl[kScanPer];
        uint32_t sg = 0, sl = 0;
#pragma unroll
        for (int k = 0; k < kScanPer; ++k) {
            const bool in = first + k < nwords;
            wg[k] = in ? __ldcg(glob + first + k) : 0u;
            wl[k] = in ? __ldcg(loc + first + k) : 0u;
            sg += __popc(wg[k]);
            sl += __popc(wl[k]);
        }
        uint32_t tg, tl;
        uint32_t rg = sums[b] + block_excl_scan(sg, tg);
        __syncthreads();
        uint32_t rl = sums[S.nblk + b] + block_excl_scan(sl, tl);
#pragma unroll
        for (int k = 0; k < kScanPer; ++k) {
            if (first + k < nwords) S.rt[first + k] = make_uint4(rg, wg[k], rl, wl[k]);
            rg += __popc(wg[k]);
            rl += __popc(wl[k]);
        }
        __syncthreads();
    }
}

// winners with candidate id < c: .x over all ranks, .y on this rank (one 16-byte load)
__device__ __forceinline__ uint2 rt_rank(const uint4* rt, uint64_t c) {
    const uint4 e = rt[c >> 5];
    const uint32_t m = (1u << (c & 31)) - 1u;
    return make_uint2(e.x + __popc(e.y & m), e.z + __popc(e.w & m));
}

// ---- decide ----------------------------------------------------------------------------------
// Same arithmetic on every rank (all inputs are replicated): see the sequential rules in
// SURVEY.md Appendix B, generalised from levels to chunks.
__global__ void __launch_bounds__(kCtrlWords) pb_decide_kernel(const PbShard S) {
    PbState* st = S.st;
    if (st->done) return;
    __shared__ unsigned long long red[kCtrlWords];
    {
        const int w = threadIdx.x;
        unsigned long long v = (w == kCtrlIerr || w == kCtrlCount) ? 0ull : ~0ull;
        for (int s = 0; s < S.world; ++s) {
            const unsigned long long x = __ldcg(&sh_ctrl(S, S.arena, st->buf, s)[w]);
            if (w == kCtrlIerr) v |= x;
            else if (w == kCtrlCount) v += x;
            else v = x < v ? x : v;
        }
        red[w] = v;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const uint64_t F = (uint64_t)st->F, head = (uint64_t)st->head, n_nodes = (uint64_t)st->n_nodes;
    const uint64_t budget = (uint64_t)st->budget;
    const int64_t nwords = (12 * (int64_t)F + 31) / 32;
    const uint64_t total = S.rt[nwords].x;
    uint64_t limit = 12 * F;
    bool cut = false;
    uint64_t cut_p = 0;
    if (n_nodes + total >= budget) {
        // first chunk-local parent p with n_nodes + #winners(parents <= p) >= budget (monotone in p)
        uint64_t lo = 0, hi = F - 1;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (n_nodes + rt_rank(S.rt, (mid + 1) * 12).x >= budget) hi = mid;
            else lo = mid + 1;
        }
        cut = true;
        cut_p = lo;
        if (12 * (cut_p + 1) < limit) limit = 12 * (cut_p + 1);
    }
    const unsigned long long sol = red[kCtrlSol], err = red[kCtrlErr];
    const int ierr = (int)red[kCtrlIerr];  // replicated: what every rank reported with this chunk's exchange
    bool sol_here = false;
    int status = 0;
    if (sol != ~0ull && sol - 12 * head < limit) {  // solved at or before the cut parent
        limit = sol - 12 * head;
        sol_here = true;
        cut = false;
    }
    if (err != ~0ull && (err >> 2) - 12 * head < limit) {  // the reference raises here, before anything later
        limit = (err >> 2) - 12 * head;
        status = (int)(err & 3);
        sol_here = false;
        cut = false;
    }
    // "New minimal length found" events in reference order
    const uint64_t gid_limit = 12 * head + limit + (sol_here ? 1 : 0);
    int min_len = st->min_len;
    for (;;) {
        unsigned long long best = ~0ull;
        int bestL = -1;
        for (int L = 0; L < min_len && L < 128; ++L) {
            const unsigned long long g = red[kCtrlLen0 + L];
            if (g < gid_limit && g < best) {
                best = g;
                bestL = L;
            }
        }
        if (bestL < 0) break;
        min_len = bestL;
        if (st->n_minlen < 128) st->minlen_log[st->n_minlen++] = bestL;
    }
    st->min_len = min_len;
    const uint2 at_limit = rt_rank(S.rt, limit);
    const uint64_t cg = at_limit.x, cl = at_limit.y;
    st->limit = (int64_t)limit;
    st->head0 = st->head;
    st->commit_pending = 1;
    st->n_nodes0 = st->n_nodes;
    st->n_local0 = st->n_local;
    int my_ierr = ierr | st->ierr;
    if ((uint64_t)st->n_local + cl > (uint64_t)st->cap_local) my_ierr |= IERR_SHARD_FULL;  // commit drops the excess
    st->n_nodes += (int64_t)cg;
    {
        const uint64_t room_local = (uint64_t)st->cap_local - (uint64_t)st->n_local;
        st->n_local += (int64_t)(cl < room_local ? cl : room_local);
    }
    if (sol_here) {
        st->solved = 1;
        st->sol_gid = (int64_t)sol;
        st->n_expanded = (int64_t)(sol / 12 + 1);
    } else if (status) {
        st->status = status;
        st->err_code = (int64_t)err;
        st->n_expanded = (int64_t)((err >> 2) / 12 + 1);
    } else if (cut) {
        st->budget_hit = 1;
        st->n_expanded = (int64_t)(head + cut_p + 1);
    } else {
        st->n_expanded = (int64_t)(head + F);
    }
    st->head += (int64_t)F;
    st->chunks += 1;
    st->epoch += 1;
    st->buf ^= 1;
    st->ierr = my_ierr;
    // a rank-local error found after the exchange travels with the NEXT chunk's control block, so
    // that every rank stops in the same chunk; errors seen by everyone stop the search now
    const bool stop = st->solved || st->budget_hit || st->status || ierr || st->head >= st->n_nodes;
    if (stop) {
        st->done = 1;
        return;
    }
    if (st->head == st->level_end) {
        st->level_end = st->n_nodes;
        st->levels += 1;
    }
    // chunk size: within the level, within the exchange buffers, and small enough that every
    // rank's table stays <= 3/4 full even if all 12*F candidates were new (shares assumed <= 1.1/G + slack)
    const int64_t G = st->world;
    const int64_t est_local = G == 1 ? st->n_nodes : (int64_t)((double)st->n_nodes / (double)G * 1.1) + 100000;
    const int64_t free_slots = (int64_t)(3 * ((st->tmask + 1) / 4)) - est_local;
    int64_t room = G == 1 ? free_slots / 12 : (int64_t)((double)free_slots * (double)G / (12.0 * 1.15));
    if (room < 1) room = 1;
    int64_t Fn = st->level_end - st->head;
    if (Fn > st->chunk_cap) Fn = st->chunk_cap;
    if (Fn > room) Fn = room;
    st->F = Fn;
}

// ---- commit ----------------------------------------------------------------------------------
template <int W>
__global__ void __launch_bounds__(256) pb_commit_kernel(const PbShard S) {
    PbState* st = S.st;
    // runs after decide of the same chunk: buf was flipped there, this chunk's buffers are buf^1.
    // decide sets `done` for the LAST chunk too, whose winners must still be appended, so the
    // commit is gated on the flag decide raises (prep of a later no-op chunk clears it).
    if (!st->commit_pending) return;
    const int buf = st->buf ^ 1;
    __shared__ RegionMap R;
    load_regions(S, st, buf, &R);
    const unsigned long long total = R.vstart[S.world];
    const int64_t log_cap = st->log_cap;
    const uint64_t* in_keys = sh_keys(S, S.arena);
    const uint32_t* in_c = sh_c(S, S.arena);
    const uint64_t limit = (uint64_t)st->limit;
    const uint64_t n_nodes0 = (uint64_t)st->n_nodes0, n_local0 = (uint64_t)st->n_local0;
    const uint64_t head0 = (uint64_t)st->head0;
    (void)total;
    {  // block b walks source log b mod G (see pb_insert_kernel): the rank table is streamed once per chunk
    const int src = (int)(blockIdx.x % (unsigned)S.world);
    const unsigned long long bsrc = blockIdx.x / (unsigned)S.world;
    const unsigned long long nbsrc = (gridDim.x - (unsigned)src + (unsigned)S.world - 1u) / (unsigned)S.world;
    const unsigned long long n_src = R.vstart[src + 1] - R.vstart[src];
    const int64_t base_src = (int64_t)src * log_cap + (int64_t)R.cstart[src];
    for (unsigned long long v = bsrc * blockDim.x + threadIdx.x; v < n_src; v += nbsrc * blockDim.x) {
        const int64_t i = base_src + (int64_t)v;
        const uint64_t c = __ldcg(in_c + i);
        if (c >= limit) continue;
        const uint4 e = S.rt[c >> 5];
        if (!((e.w >> (c & 31)) & 1u)) continue;  // an already visited state, or lost to an earlier candidate
        const uint32_t m = (1u << (c & 31)) - 1u;
        const uint64_t g = n_nodes0 + e.x + __popc(e.y & m);
        const uint64_t idx = n_local0 + e.z + __popc(e.w & m);
        if (idx >= (uint64_t)st->cap_local) continue;  // IERR_SHARD_FULL was raised by decide
        node_store<W>(S.nodes, idx, load_key_cg<W>(in_keys, (uint64_t)i), (int64_t)(((head0 + c / 12) << 4) | (c % 12)),
                      (int64_t)g);
    }
    }
}

}  // namespace acs

namespace acs {

// one thread: smallest local index with gid >= value
__device__ __forceinline__ int64_t pb_lower_bound(const uint64_t* nodes, int W, int64_t n, int64_t value) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (node_gid_rt(nodes, W, mid) < value) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// out = {found, parent gid, action, total length} of the node with global id `value`
template <int W>
__global__ void pb_lookup_kernel(const PbShard S, int64_t value, long long* out) {
    const int64_t n = S.st->n_local;
    const int64_t lo = pb_lower_bound(S.nodes, W, n, value);
    out[0] = out[1] = out[2] = out[3] = 0;
    Key<W> k;
    int64_t par = 0, g = -1;
    if (lo < n) node_load<W>(S.nodes, (uint64_t)lo, k, par, g);
    if (lo < n && g == value) {
        out[0] = 1;
        out[1] = par < 0 ? -1 : (par >> 4);
        out[2] = par < 0 ? -1 : (par & 15);
        out[3] = key_total_len<W>(k);
    }
}

// all shards in this process: path of node `node` from the root, then (extra_action, extra_len)
template <int W>
__global__ void pb_path_kernel(const PbShard* shards, int n_shards, int64_t node, int extra_action, int extra_len,
                               int32_t* path, int path_cap, int32_t* path_len) {
    // pass 1: depth; pass 2: fill back to front
    for (int pass = 0, depth = 0; pass < 2; ++pass) {
        int pos = depth - 1, d = 0;
        for (int64_t g = node; g >= 0;) {
            int64_t par = -1;
            int act = -1, L = 0;
            for (int s = 0; s < n_shards; ++s) {
                const PbShard& S = shards[s];
                const int64_t n = S.st->n_local;
                const int64_t lo = pb_lower_bound(S.nodes, W, n, g);
                Key<W> k;
                int64_t pl = 0, gg = -1;
                if (lo < n) node_load<W>(S.nodes, (uint64_t)lo, k, pl, gg);
                if (lo < n && gg == g) {
                    L = key_total_len<W>(k);
                    par = pl < 0 ? -1 : (pl >> 4);
                    act = pl < 0 ? -1 : (int)(pl & 15);
                    break;
                }
            }
            if (pass == 1 && pos >= 0 && pos < path_cap) {
                path[2 * pos] = act;
                path[2 * pos + 1] = L;
            }
            --pos;
            ++d;
            g = par;
        }
        if (pass == 0) {
            depth = d;
            *path_len = depth + 1;
            if (depth < path_cap) {
                path[2 * depth] = extra_action;
                path[2 * depth + 1] = extra_len;
            }
        }
    }
}

}  // namespace acs

// ---------------------------------------------------------------------------------------------
using namespace acs;

namespace {
inline int64_t align256(int64_t x) { return (x + 255) / 256 * 256; }
constexpr int kRing = 4, kLag = 2;
}  // namespace

struct acs_pbfs {
    int device = 0, rank = 0, world = 1, mrl = 0, W = 1, cyclical = 0;
    int64_t budget = 0, cap_local = 0, chunk_cap = 0, log_cap = 0;
    uint64_t tcap = 0;
    int64_t arena_bytes = 0;
    PbShard S{};              // host copy of the pointer block (passed by value to the kernels)
    PbShard* d_shards = nullptr;  // device array of all local shards (path kernel), owned by shard 0 of a local group
    int n_group = 0;
    void* ipc_opened[kPbMaxWorld] = {};
    bool connected = false;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ring_ev[kRing] = {};
    PbState* h_ring = nullptr;  // pinned [kRing]
    PbState h_final{};
    uint64_t epoch = 0;
    int sms = 148;
    int expand_wpb = 8, expand_blocks = 148, insert_blocks = 148, commit_blocks = 148;
    size_t expand_smem = 0;
    bool cta_stage = false;  // block-level staging of the expansion (world > 1; ACS_PBFS_CTA_STAGE=0 disables)
    int cta_blocks = 148, cta_threads = 256;
    size_t cta_smem = 0;
    int32_t* d_path = nullptr;
    int path_cap = 1 << 16;
    long long* d_small = nullptr;
    unsigned long long timeout_ns = 20ull * 1000 * 1000 * 1000;
};

extern "C" {

int acs_pbfs_create(int device, int rank, int world, int mrl, int64_t max_nodes, int cyclical, int64_t chunk_parents,
                    acs_pbfs** out) {
    if (!out) return ACS_ERR_INVALID;
    *out = nullptr;
    if (const int rc = check_key_mrl(mrl, "bfs")) return rc;
    if (world < 1 || world > kPbMaxWorld || rank < 0 || rank >= world || max_nodes < 0)
        return fail(ACS_ERR_INVALID, "pbfs: bad rank / world / budget");
    if (const int rc = open_device(device, "pbfs")) return rc;
    acs_pbfs* b = new acs_pbfs();
    b->device = device;
    b->rank = rank;
    b->world = world;
    b->mrl = mrl;
    b->W = key_words(mrl);
    b->cyclical = cyclical ? 1 : 0;
    b->budget = max_nodes;
    // hash partitioning is balanced to a few sigma of sqrt(n/world); the budget test overshoots by <= 11
    b->cap_local = world == 1 ? max_nodes + 16 : (int64_t)((double)(max_nodes + 16) / world * 1.1) + 200000;
    uint64_t t = 1024;
    while (t < 2 * (uint64_t)b->cap_local) t <<= 1;
    b->tcap = t;
    auto bail = [&](int code, const std::string& m) {
        acs_pbfs_destroy(b);
        return fail(code, m);
    };
    if (t > (1ull << 31)) return bail(ACS_ERR_UNSUPPORTED, "pbfs: more than 2^30 nodes per rank: use more GPUs");
    // chunk size: per-rank work of ~4 Mi parents; candidate ids are 32-bit
    int64_t chunk = chunk_parents > 0 ? chunk_parents : (int64_t)world << 22;
    chunk = std::min<int64_t>(chunk, std::max<int64_t>(max_nodes + 16, 1024));
    chunk = std::min<int64_t>(chunk, ((int64_t)1 << 32) / 12 - 1);
    b->chunk_cap = chunk;
    // Record logs: every generated child that is not a self loop is appended to the (source ->
    // owner) log and stays there (table slots point at log positions, so nothing is rewritten
    // when a node is committed).  At most 12 records per expanded node; AC graphs produce ~2.2
    // per visited node, the default budgets 3 (ACS_PBFS_LOG_FACTOR overrides) plus the last
    // chunk's overshoot past the budget cut.
    double factor = 3.0;
    if (const char* f = std::getenv("ACS_PBFS_LOG_FACTOR")) factor = std::max(0.1, std::atof(f));
    const double worst = 12.0 * (double)(max_nodes + 16 + chunk);
    const double total = std::min(worst, factor * (double)max_nodes + 12.0 * (double)chunk + 1048576.0);
    b->log_cap = world == 1 ? (int64_t)total + 64 : (int64_t)(total / ((double)world * world) * 1.15) + 65536;
    if ((double)b->log_cap * world >= (double)(1ull << 40)) return bail(ACS_ERR_UNSUPPORTED, "pbfs: record log too large");
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) b->sms = prop.multiProcessorCount;
    if (const char* g = std::getenv("ACS_L2_FETCH")) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)std::atoi(g));

    PbShard& S = b->S;
    S.W = b->W;
    S.world = world;
    S.rank = rank;
    S.bitmap_words = (12 * chunk + 31) / 32 + 8;
    S.nblk = (S.bitmap_words + kScanBlock - 1) / kScanBlock + 1;
    int64_t off = 0;
    S.off_flags = off;
    off = align256(off + 3 * (int64_t)world * 8);
    S.off_ctrl = off;
    off = align256(off + 2 * (int64_t)world * kCtrlWords * 8);
    const int64_t zero_bytes = off;  // flags / control inboxes start at zero (epochs start at 1)
    S.off_bitmap = off;
    off = align256(off + 2 * S.bitmap_words * 4);
    S.off_bmg = off;
    off = align256(off + S.bitmap_words * 4);
    S.off_bsums = off;
    off = align256(off + 2 * S.nblk * 4);
    S.off_keys = off;
    off = align256(off + (int64_t)world * b->log_cap * 16 * b->W);
    S.off_c = off;
    off = align256(off + (int64_t)world * b->log_cap * 4);
    b->arena_bytes = off;
    ACS_ALLOC(S.arena, b->arena_bytes, acs_pbfs_destroy(b));
    ACS_ALLOC(S.st, sizeof(PbState), acs_pbfs_destroy(b));
    ACS_ALLOC(S.nodes, (size_t)b->cap_local * 8 * node_words(b->W), acs_pbfs_destroy(b));
    ACS_ALLOC(S.table, (size_t)b->tcap * 8, acs_pbfs_destroy(b));
    ACS_ALLOC(S.rt, (size_t)(S.bitmap_words + 1) * sizeof(uint4), acs_pbfs_destroy(b));
    ACS_ALLOC(S.cursors, kPbMaxWorld * kCurStride * 8, acs_pbfs_destroy(b));
    ACS_ALLOC(S.cstart, kPbMaxWorld * 8, acs_pbfs_destroy(b));
    ACS_ALLOC(S.ctrl_local, kCtrlWords * 8, acs_pbfs_destroy(b));
    ACS_ALLOC(b->d_path, (size_t)b->path_cap * 2 * sizeof(int32_t) + 16, acs_pbfs_destroy(b));
    ACS_ALLOC(b->d_small, 8 * sizeof(long long), acs_pbfs_destroy(b));
    // flags / control inboxes start at zero (epochs start at 1)
    if (cudaMemset(S.arena, 0, (size_t)zero_bytes) != cudaSuccess) return bail(ACS_ERR_CUDA, "pbfs: memset(arena)");
    if (cudaMallocHost((void**)&b->h_ring, kRing * sizeof(PbState)) != cudaSuccess)
        return bail(ACS_ERR_NOMEM, "pbfs: cudaMallocHost");
    if (cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(ACS_ERR_CUDA, "pbfs: cudaStreamCreate");
    cudaEventCreate(&b->ev0);
    cudaEventCreate(&b->ev1);
    for (auto& e : b->ring_ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    // expand launch shape: as many warps per block as ~100 KB of staging allows
    const size_t per_warp = b->W == 1 ? stage_bytes_per_warp<1>() : stage_bytes_per_warp<2>();
    int wpb = 8;
    while (wpb > 1 && per_warp * wpb > 100 * 1024) wpb /= 2;
    b->expand_wpb = wpb;
    b->expand_smem = per_warp * wpb;
    cudaError_t e = cudaSuccess;
    if (b->W == 1) {
        e = cudaFuncSetAttribute(pb_expand_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->expand_smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(pb_expand_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->expand_smem);
    } else {
        e = cudaFuncSetAttribute(pb_expand_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->expand_smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(pb_expand_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->expand_smem);
    }
    if (e != cudaSuccess) return bail(ACS_ERR_CUDA, std::string("pbfs: expand smem attribute: ") + cudaGetErrorString(e));
    int per_sm = 1;
    if (b->W == 1) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pb_expand_kernel<1, true>, 32 * wpb, b->expand_smem);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pb_expand_kernel<2, true>, 32 * wpb, b->expand_smem);
    b->expand_blocks = b->sms * std::max(per_sm, 1);
    {
        const char* e2 = std::getenv("ACS_PBFS_CTA_STAGE");
        b->cta_stage = world > 1 && !(e2 && e2[0] == '0');
        b->cta_threads = 512;  // 16 warps stage together: ~120 records (1.9 KB of keys) per destination and flush at G = 8
        if (const char* e3 = std::getenv("ACS_PBFS_CTA_THREADS")) {
            const int v = std::atoi(e3);
            if (v == 128 || v == 256 || v == 512) b->cta_threads = v;
        }
        b->cta_smem = b->W == 1 ? cta_stage_bytes<1>(b->cta_threads / 32) : cta_stage_bytes<2>(b->cta_threads / 32);
        int cps = 1;
        if (b->W == 1) {
            cudaFuncSetAttribute(pb_expand_cta_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->cta_smem);
            cudaFuncSetAttribute(pb_expand_cta_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->cta_smem);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cps, pb_expand_cta_kernel<1, true>, b->cta_threads, b->cta_smem);
        } else {
            cudaFuncSetAttribute(pb_expand_cta_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->cta_smem);
            cudaFuncSetAttribute(pb_expand_cta_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->cta_smem);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cps, pb_expand_cta_kernel<2, true>, b->cta_threads, b->cta_smem);
        }
        b->cta_blocks = b->sms * std::max(cps, 1);
    }
    // persistent grid-stride kernels: exactly one wave of resident blocks
    int ib = 1, cb = 1;
    if (b->W == 1) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ib, pb_insert_kernel<1>, 256, 0);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cb, pb_commit_kernel<1>, 256, 0);
    } else {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ib, pb_insert_kernel<2>, 256, 0);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cb, pb_commit_kernel<2>, 256, 0);
    }
    // (at least one block per source log: block b works on source b mod world)
    b->insert_blocks = std::max(b->sms * std::max(ib, 1), world);
    b->commit_blocks = std::max(b->sms * std::max(cb, 1), world);
    for (int r = 0; r < kPbMaxWorld; ++r) S.peer[r] = nullptr;
    S.peer[rank] = S.arena;
    b->connected = world == 1;
    *out = b;
    return ACS_OK;
}

void acs_pbfs_destroy(acs_pbfs* b) {
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->stream) {
        cudaStreamSynchronize(b->stream);
        cudaStreamDestroy(b->stream);
    }
    for (auto p : b->ipc_opened)
        if (p) cudaIpcCloseMemHandle(p);
    if (b->ev0) cudaEventDestroy(b->ev0);
    if (b->ev1) cudaEventDestroy(b->ev1);
    for (auto e : b->ring_ev)
        if (e) cudaEventDestroy(e);
    PbShard& S = b->S;
    cudaFree(S.arena);
    cudaFree(S.st);
    cudaFree(S.nodes);
    cudaFree(S.table);
    cudaFree(S.rt);
    cudaFree(S.cursors);
    cudaFree(S.cstart);
    cudaFree(S.ctrl_local);
    cudaFree(b->d_path);
    cudaFree(b->d_small);
    cudaFree(b->d_shards);
    if (b->h_ring) cudaFreeHost(b->h_ring);
    cudaGetLastError();
    delete b;
}

/* 64-byte cudaIpcMemHandle_t of this rank's exchange arena (inboxes, control inboxes, flags, bitmaps) */
int acs_pbfs_export(acs_pbfs* b, void* handle64) {
    if (!b || !handle64) return ACS_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    ACS_CUDA(cudaSetDevice(b->device));
    cudaIpcMemHandle_t h;
    ACS_CUDA(cudaIpcGetMemHandle(&h, b->S.arena));
    std::memcpy(handle64, &h, 64);
    return ACS_OK;
}

/* handles: world x 64 bytes in rank order (as gathered from acs_pbfs_export on every rank) */
int acs_pbfs_connect(acs_pbfs* b, const void* handles) {
    if (!b || !handles) return ACS_ERR_INVALID;
    ACS_CUDA(cudaSetDevice(b->device));
    for (int r = 0; r < b->world; ++r) {
        if (r == b->rank) continue;
        cudaIpcMemHandle_t h;
        std::memcpy(&h, static_cast<const char*>(handles) + 64 * r, 64);
        void* p = nullptr;
        ACS_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        b->ipc_opened[r] = p;
        b->S.peer[r] = static_cast<char*>(p);
    }
    b->connected = true;
    return ACS_OK;
}

/* every rank of the world lives in this process (tests; single-process multi-GPU) */
int acs_pbfs_connect_local(acs_pbfs** shards, int n) {
    if (!shards || n < 1) return ACS_ERR_INVALID;
    for (int i = 0; i < n; ++i)
        if (!shards[i] || shards[i]->world != n || shards[i]->rank != i) return fail(ACS_ERR_INVALID, "pbfs: shards must be ranks 0..n-1 of a world of n");
    for (int i = 0; i < n; ++i) {
        for (int j = 0; j < n; ++j) {
            shards[i]->S.peer[j] = shards[j]->S.arena;
            if (shards[i]->device != shards[j]->device) {
                ACS_CUDA(cudaSetDevice(shards[i]->device));
                int can = 0;
                ACS_CUDA(cudaDeviceCanAccessPeer(&can, shards[i]->device, shards[j]->device));
                if (!can) return fail(ACS_ERR_UNSUPPORTED, "pbfs: no peer access between the devices");
                cudaError_t e = cudaDeviceEnablePeerAccess(shards[j]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) ACS_CUDA(e);
                cudaGetLastError();
            }
        }
        shards[i]->connected = true;
    }
    // device array of the pointer blocks for the path kernel
    acs_pbfs* b0 = shards[0];
    ACS_CUDA(cudaSetDevice(b0->device));
    if (b0->d_shards) cudaFree(b0->d_shards);
    b0->d_shards = nullptr;
    ACS_CUDA(cudaMalloc((void**)&b0->d_shards, n * sizeof(PbShard)));
    for (int i = 0; i < n; ++i)
        ACS_CUDA(cudaMemcpy(b0->d_shards + i, &shards[i]->S, sizeof(PbShard), cudaMemcpyHostToDevice));
    b0->n_group = n;
    return ACS_OK;
}

}  // extern "C"

namespace {

template <int W>
int pb_run_impl(acs_pbfs** sh, int n_local, const int8_t* h_presentation, int32_t* h_path, int path_cap,
                acs_search_result* res) {
    std::memset(res, 0, sizeof(*res));
    acs_pbfs* b0 = sh[0];
    const int world = b0->world;
    Key<W> root;
    int lens[2];
    const RootCheck rc0 = pack_root<W>(h_presentation, b0->mrl, root, lens);
    if (rc0 == RootCheck::bad_letter)
        return fail(ACS_ERR_UNSUPPORTED, "bfs: letters outside {+-1,+-2} are not supported by the packed search");
    if (rc0 != RootCheck::ok) {  // breadth_first.py:36-38 asserts is_array_valid_presentation
        res->status = ACS_ROW_ASSERT;
        return ACS_OK;
    }
    const uint64_t h = pb_hash<W>(root);
    const int owner = world > 1 ? pb_owner<W>(root, world) : 0;
    bool same_device = true;
    for (int i = 0; i < n_local; ++i) same_device = same_device && sh[i]->device == b0->device;
    auto stream_of = [&](acs_pbfs* b) { return same_device ? b0->stream : b->stream; };

    for (int i = 0; i < n_local; ++i) {
        acs_pbfs* b = sh[i];
        if (!b->connected) return fail(ACS_ERR_INVALID, "pbfs: shard is not connected to its peers");
        ACS_CUDA(cudaSetDevice(b->device));
        cudaStream_t s = stream_of(b);
        ACS_CUDA(cudaMemsetAsync(b->S.table, 0, b->tcap * sizeof(uint64_t), s));
        ACS_CUDA(cudaMemsetAsync(b->S.cursors, 0, kPbMaxWorld * kCurStride * 8, s));
        PbState st{};
        st.budget = b->budget;
        st.cap_local = b->cap_local;
        st.chunk_cap = b->chunk_cap;
        st.log_cap = b->log_cap;
        st.tmask = b->tcap - 1;
        st.mrl = b->mrl;
        st.cyclical = b->cyclical;
        st.world = world;
        st.rank = b->rank;
        st.head = 0;
        st.F = 1;
        st.n_nodes = 1;
        st.n_local = b->rank == owner ? 1 : 0;
        st.level_end = 1;
        st.epoch = b->epoch;
        st.buf = (int)(b->epoch & 1);
        st.min_len = lens[0] + lens[1];
        st.sol_gid = -1;
        b->h_ring[0] = st;  // pinned staging for the async upload
        ACS_CUDA(cudaMemcpyAsync(b->S.st, &b->h_ring[0], sizeof(PbState), cudaMemcpyHostToDevice, s));
        if (b->rank == owner) {
            // the root is record 0 of the owner's own (owner -> owner) log, node 0 of its shard, and
            // sits in the first slot of its 4-slot bucket (where the insert kernel's probe starts)
            const uint64_t log_pos = (uint64_t)owner * (uint64_t)b->log_cap;
            const uint64_t slot_val = ((h >> 41) << 40) | (log_pos + 1);
            const unsigned long long one = 1;
            const uint32_t c0 = 0;
            char* arena = b->S.arena;
            uint64_t node0[node_words(W)];
            node_pack<W>(root, -1, 0, node0);
            ACS_CUDA(cudaMemcpyAsync(b->S.nodes, node0, sizeof(node0), cudaMemcpyHostToDevice, s));
            ACS_CUDA(cudaMemcpyAsync(arena + b->S.off_keys + log_pos * sizeof(root), &root, sizeof(root), cudaMemcpyHostToDevice, s));
            ACS_CUDA(cudaMemcpyAsync(arena + b->S.off_c + log_pos * 4, &c0, 4, cudaMemcpyHostToDevice, s));
            ACS_CUDA(cudaMemcpyAsync(b->S.cursors + owner * kCurStride, &one, 8, cudaMemcpyHostToDevice, s));
            ACS_CUDA(cudaMemcpyAsync(b->S.table + ((h & (b->tcap - 1)) & ~3ull), &slot_val, 8, cudaMemcpyHostToDevice, s));
        }
        ACS_CUDA(cudaStreamSynchronize(s));  // the staging copies above read host stack memory
    }
    ACS_CUDA(cudaSetDevice(b0->device));
    ACS_CUDA(cudaEventRecord(b0->ev0, stream_of(b0)));

    auto each = [&](auto&& fn) -> int {
        for (int i = 0; i < n_local; ++i) {
            acs_pbfs* b = sh[i];
            if (!same_device) {
                cudaError_t e = cudaSetDevice(b->device);
                if (e != cudaSuccess) return fail(ACS_ERR_CUDA, cudaGetErrorString(e));
            }
            fn(b, stream_of(b));
        }
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(ACS_ERR_CUDA, std::string("pbfs launch: ") + cudaGetErrorString(e));
        return ACS_OK;
    };
    int rc = ACS_OK;
    // ACS_PBFS_PROFILE=1: CUDA events after every phase of rank sh[0] -> per-phase totals on stderr
    const bool profile = std::getenv("ACS_PBFS_PROFILE") != nullptr;
    static const char* kPhaseNames[14] = {"prep", "expand", "signal0", "wait0", "insert", "signal1", "wait1",
                                          "scan_sums", "signal2", "wait2", "scan_top", "scan_final", "decide", "commit"};
    std::vector<cudaEvent_t> pev;
    int phase_idx = 0;
    auto mark = [&]() {
        if (!profile) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, stream_of(b0));
        pev.push_back(e);
    };
    (void)phase_idx;
    mark();
    for (int64_t chunk = 0;; ++chunk) {
        if (chunk >= kLag) {
            ACS_CUDA(cudaEventSynchronize(b0->ring_ev[(chunk - kLag) % kRing]));
            if (b0->h_ring[(chunk - kLag) % kRing].done) break;
        }
#define PB_PHASE(expr)                                       \
    rc = each([&](acs_pbfs* b, cudaStream_t s) { expr; });   \
    if (rc != ACS_OK) return rc;                             \
    mark();
        PB_PHASE((pb_prep_kernel<<<b->sms * 2, 256, 0, s>>>(b->S)));
        if (b0->cta_stage) {
            if (chunk == 0) {
                PB_PHASE((pb_expand_cta_kernel<W, false><<<b->cta_blocks, b->cta_threads, b->cta_smem, s>>>(b->S)));
            } else {
                PB_PHASE((pb_expand_cta_kernel<W, true><<<b->cta_blocks, b->cta_threads, b->cta_smem, s>>>(b->S)));
            }
        } else if (chunk == 0) {
            PB_PHASE((pb_expand_kernel<W, false><<<b->expand_blocks, 32 * b->expand_wpb, b->expand_smem, s>>>(b->S, b->expand_wpb)));
        } else {
            PB_PHASE((pb_expand_kernel<W, true><<<b->expand_blocks, 32 * b->expand_wpb, b->expand_smem, s>>>(b->S, b->expand_wpb)));
        }
        PB_PHASE((pb_signal_kernel<<<1, 256, 0, s>>>(b->S, 0)));
        if (world > 1) { PB_PHASE((pb_wait_kernel<<<1, 32, 0, s>>>(b->S, 0, b->timeout_ns))); } else mark();
        PB_PHASE((pb_insert_kernel<W><<<b->insert_blocks, 256, 0, s>>>(b->S)));
        if (world > 1) {
            PB_PHASE((pb_signal_kernel<<<1, 256, 0, s>>>(b->S, 1)));
            PB_PHASE((pb_wait_kernel<<<1, 32, 0, s>>>(b->S, 1, b->timeout_ns)));
        } else {
            mark();
            mark();
        }
        PB_PHASE((pb_scan_sums_kernel<<<b->sms * 4, kScanT, 0, s>>>(b->S)));
        if (world > 1) {
            PB_PHASE((pb_signal_kernel<<<1, 256, 0, s>>>(b->S, 2)));
            PB_PHASE((pb_wait_kernel<<<1, 32, 0, s>>>(b->S, 2, b->timeout_ns)));
        } else {
            mark();
            mark();
        }
        PB_PHASE((pb_scan_top_kernel<<<1, kScanT, 0, s>>>(b->S)));
        PB_PHASE((pb_scan_final_kernel<<<b->sms * 4, kScanT, 0, s>>>(b->S)));
        PB_PHASE((pb_decide_kernel<<<1, kCtrlWords, 0, s>>>(b->S)));
        PB_PHASE((pb_commit_kernel<W><<<b->commit_blocks, 256, 0, s>>>(b->S)));
#undef PB_PHASE
        if (!same_device) ACS_CUDA(cudaSetDevice(b0->device));
        ACS_CUDA(cudaMemcpyAsync(&b0->h_ring[chunk % kRing], b0->S.st, sizeof(PbState), cudaMemcpyDeviceToHost, stream_of(b0)));
        ACS_CUDA(cudaEventRecord(b0->ring_ev[chunk % kRing], stream_of(b0)));
    }
    ACS_CUDA(cudaEventRecord(b0->ev1, stream_of(b0)));
    int ierr = 0;
    for (int i = 0; i < n_local; ++i) {
        acs_pbfs* b = sh[i];
        ACS_CUDA(cudaSetDevice(b->device));
        ACS_CUDA(cudaStreamSynchronize(stream_of(b)));
        ACS_CUDA(cudaMemcpy(&b->h_final, b->S.st, sizeof(PbState), cudaMemcpyDeviceToHost));
        b->epoch = b->h_final.epoch;
        ierr |= b->h_final.ierr;
    }
    ACS_CUDA(cudaSetDevice(b0->device));
    const PbState& f = b0->h_final;
    if (ierr) {
        std::string m = "pbfs: internal error:";
        if (ierr & IERR_LOG_FULL) m += " record log full (raise ACS_PBFS_LOG_FACTOR: this graph generates more than 3 children per visited state)";
        if (ierr & IERR_TABLE_FULL) m += " visited table full";
        if (ierr & IERR_SHARD_FULL) m += " shard capacity exceeded (skewed partition)";
        if (ierr & IERR_TIMEOUT) m += " timed out waiting for a peer rank";
        return fail(ACS_ERR_CUDA, m);
    }
    res->solved = f.solved;
    res->status = f.status;
    res->budget_hit = f.budget_hit;
    res->n_visited = f.n_nodes;
    res->n_expanded = f.n_expanded;
    res->n_moves = f.solved ? f.sol_gid + 1 : (f.status ? (int64_t)(((uint64_t)f.err_code >> 2) + 1) : f.n_expanded * 12);
    res->frontier_left = f.n_nodes - f.n_expanded;
    res->n_levels = f.levels;
    res->n_minlen = f.n_minlen;
    for (int i = 0; i < f.n_minlen && i < 128; ++i) res->minlen_log[i] = f.minlen_log[i];
    float ms = 0.f;
    cudaEventElapsedTime(&ms, b0->ev0, b0->ev1);
    res->seconds_device = ms * 1e-3;
    if (profile && pev.size() > 1) {
        double tot[14] = {};
        for (size_t k = 1; k < pev.size(); ++k) {
            float t = 0.f;
            cudaEventElapsedTime(&t, pev[k - 1], pev[k]);
            tot[(k - 1) % 14] += t;
        }
        std::string line = "{\"pbfs_profile_ms\": {";
        for (int k = 0; k < 14; ++k) {
            char buf[64];
            std::snprintf(buf, sizeof buf, "%s\"%s\": %.3f", k ? ", " : "", kPhaseNames[k], tot[k]);
            line += buf;
        }
        char tail[160];
        std::snprintf(tail, sizeof tail, "}, \"rank\": %d, \"world\": %d, \"chunks\": %lld, \"total_ms\": %.3f}\n", b0->rank, world,
                      (long long)f.chunks, ms);
        line += tail;
        std::fputs(line.c_str(), stderr);
        for (auto e : pev) cudaEventDestroy(e);
    }
    if (f.solved && n_local == world && b0->d_shards && b0->n_group == world) {
        const int cap = std::min(path_cap, b0->path_cap);
        int32_t* d_len = b0->d_path + 2 * (size_t)b0->path_cap;
        cudaStream_t s = stream_of(b0);
        pb_path_kernel<W><<<1, 1, 0, s>>>(b0->d_shards, world, f.sol_gid / 12, (int)(f.sol_gid % 12), 2, b0->d_path, cap, d_len);
        ACS_CUDA(cudaGetLastError());
        int32_t plen = 0;
        ACS_CUDA(cudaMemcpyAsync(&plen, d_len, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        ACS_CUDA(cudaStreamSynchronize(s));
        res->path_len = plen;
        if (h_path && cap > 0)
            ACS_CUDA(cudaMemcpy(h_path, b0->d_path, (size_t)std::min(plen, cap) * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    }
    return ACS_OK;
}

}  // namespace

extern "C" {

/* Runs the search on the local shards (all `world` ranks of a single-process world, or this
 * process's one rank of a multi-process world: every process calls it with the same arguments).
 * The path is produced here only when all ranks are local; otherwise walk it with
 * acs_pbfs_lookup (see ac_solver_b200/search/partitioned.py). */
int acs_pbfs_run(acs_pbfs** shards, int n_local, const int8_t* h_presentation, int32_t* h_path, int path_cap,
                 acs_search_result* res) {
    if (!shards || n_local < 1 || !shards[0] || !h_presentation || !res) return ACS_ERR_INVALID;
    for (int i = 0; i < n_local; ++i)
        if (!shards[i] || shards[i]->W != shards[0]->W || shards[i]->world != shards[0]->world) return ACS_ERR_INVALID;
    if (n_local != 1 && n_local != shards[0]->world) return fail(ACS_ERR_INVALID, "pbfs: pass one shard or all of them");
    return shards[0]->W == 1 ? pb_run_impl<1>(shards, n_local, h_presentation, h_path, path_cap, res)
                             : pb_run_impl<2>(shards, n_local, h_presentation, h_path, path_cap, res);
}

/* out4 = {found on this rank, parent global id (-1 root), action (-1 root), total length} */
int acs_pbfs_lookup(acs_pbfs* b, int64_t gid, int64_t* out4) {
    if (!b || !out4) return ACS_ERR_INVALID;
    ACS_CUDA(cudaSetDevice(b->device));
    if (b->W == 1) pb_lookup_kernel<1><<<1, 1, 0, b->stream>>>(b->S, gid, b->d_small);
    else pb_lookup_kernel<2><<<1, 1, 0, b->stream>>>(b->S, gid, b->d_small);
    ACS_CUDA(cudaGetLastError());
    ACS_CUDA(cudaMemcpyAsync(out4, b->d_small, 4 * sizeof(long long), cudaMemcpyDeviceToHost, b->stream));
    ACS_CUDA(cudaStreamSynchronize(b->stream));
    return ACS_OK;
}

/* this rank's visited states (int8 rows) and their global ids (= FIFO positions), local order */
int acs_pbfs_visited(acs_pbfs* b, int64_t* h_gid, int8_t* h_rows, int64_t cap_rows, int64_t* n_out) {
    if (!b || (cap_rows > 0 && (!h_gid || !h_rows))) return ACS_ERR_INVALID;
    ACS_CUDA(cudaSetDevice(b->device));
    const int64_t n = std::min<int64_t>(b->h_final.n_local, std::max<int64_t>(cap_rows, 0));
    if (n_out) *n_out = n;
    return records_to_host(b->W, b->S.nodes, node_words(b->W), n, b->mrl, h_rows, h_gid, b->stream);
}

/* counters of the last run on this rank: {n_local, chunks, records sent, records received, chunk_cap, log_cap (records per source),
 * arena bytes, table slots} */
int acs_pbfs_stats(acs_pbfs* b, int64_t* out8) {
    if (!b || !out8) return ACS_ERR_INVALID;
    out8[0] = b->h_final.n_local;
    out8[1] = b->h_final.chunks;
    out8[2] = (int64_t)b->h_final.records_sent;
    out8[3] = (int64_t)b->h_final.records_recv;
    out8[4] = b->chunk_cap;
    out8[5] = b->log_cap;
    out8[6] = b->arena_bytes;
    out8[7] = (int64_t)b->tcap;
    return ACS_OK;
}

int acs_pbfs_set_timeout(acs_pbfs* b, double seconds) {
    if (!b || seconds <= 0) return ACS_ERR_INVALID;
    b->timeout_ns = (unsigned long long)(seconds * 1e9);
    return ACS_OK;
}

}  // extern "C"

// ---- single-GPU search API (acs_bfs_*): the partitioned engine with a world of one ----------------
struct acs_bfs {
    acs_pbfs* shard = nullptr;
};

extern "C" {

int acs_bfs_create(acs_ctx* /*ctx*/, int device, int mrl, int64_t max_nodes, int cyclical, acs_bfs** out) {
    if (!out) return ACS_ERR_INVALID;
    *out = nullptr;
    acs_pbfs* p = nullptr;
    const int rc = acs_pbfs_create(device, 0, 1, mrl, max_nodes, cyclical, 0, &p);
    if (rc != ACS_OK) return rc;
    acs_pbfs* arr[1] = {p};
    const int rc2 = acs_pbfs_connect_local(arr, 1);
    if (rc2 != ACS_OK) {
        acs_pbfs_destroy(p);
        return rc2;
    }
    acs_bfs* b = new acs_bfs();
    b->shard = p;
    *out = b;
    return ACS_OK;
}

int acs_bfs_run(acs_bfs* b, const int8_t* h_presentation, int32_t* h_path, int path_cap, acs_search_result* res) {
    if (!b || !b->shard || !h_presentation || !res) return ACS_ERR_INVALID;
    acs_pbfs* arr[1] = {b->shard};
    return acs_pbfs_run(arr, 1, h_presentation, h_path, path_cap, res);
}

int acs_bfs_visited(acs_bfs* b, int8_t* h_out, int64_t cap_rows, int64_t* n_out) {
    if (!b || !b->shard || (!h_out && cap_rows > 0)) return ACS_ERR_INVALID;
    // with one rank the local order IS the global (FIFO) order
    std::vector<int64_t> gid((size_t)std::max<int64_t>(std::min<int64_t>(cap_rows, b->shard->h_final.n_local), 1));
    return acs_pbfs_visited(b->shard, gid.data(), h_out, cap_rows, n_out);
}

void acs_bfs_destroy(acs_bfs* b) {
    if (!b) return;
    acs_pbfs_destroy(b->shard);
    delete b;
}

}  // extern "C"
