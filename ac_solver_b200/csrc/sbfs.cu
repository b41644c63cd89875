// sbfs.cu -- device kernels of the hash-partitioned (multi-GPU) breadth-first search.
//
// Same sequential contract as bfs.cu (reference: ac_solver/search/breadth_first.py:15-97), with
// the visited set and the node store partitioned by owner(state) = hash(key) mod world.  The
// host loop (ac_solver_b200/search/sharded.py) processes chunks of consecutive GLOBAL node ids
// in lockstep on all ranks; per chunk, on each rank:
//   expand  every owned parent of the chunk generates its 12 children (packed moves of
//           ac_core.cuh), labelled with the chunk-local candidate id c = 12*(gid-head)+action,
//           and bins them by owner rank (block-level shared-memory histogram, one global
//           atomic per block and destination);
//   [NCCL all-to-all of (key, c) records -- the only data-path collective]
//   insert  the owner inserts received records into its exact open-addressing table with
//           "smallest candidate id wins" (one atomicMin: committed entries have bit 63 clear,
//           tentative ones carry c in the top bits);
//   mark    winners set bit c of a chunk bitmap;
//   [all-reduce(sum) of the bitmap: bits are disjoint, so every rank sees all winners]
//   scan    prefix popcounts give every winner its GLOBAL rank (= FIFO position) and the
//           budget cut, identically on every rank;
//   commit  owners append their winners below the limit, in c order, with global ids.
// Results (path, visited array in global-id order, stdout) are bit-identical to the
// single-GPU search and therefore to the reference, for every world size.
#include <algorithm>
#include <cstdint>
#include <cstring>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "ac_core.cuh"
#include "ac_keys.cuh"
#include "acs_internal.h"

namespace acs {

constexpr int kSbThreads = 384;  // 32 parents x 12 actions
constexpr uint32_t kNoSlot32 = 0xFFFFFFFFu;
constexpr uint64_t kTentBit = 1ull << 63;
constexpr uint64_t kMask26 = (1ull << 26) - 1;
constexpr int kMaxWorld = 16;

// The owner must be statistically independent of the table slot (low bits of h) and of the
// fingerprints (high bits): taking it from a bit range of h itself pins those bits for every key
// a rank owns, which clusters its table into 1/world of the slots once the table is larger than
// that bit position (found at 8 GPUs: probe chains exploded for tables >= 2^25 slots).
__host__ __device__ __forceinline__ int owner_of(uint64_t h, int world) {
    return (int)((uint32_t)(mix64(h ^ 0x9e3779b97f4a7c15ull) >> 40) % (uint32_t)world);
}

template <int W>
__device__ __forceinline__ int sb_child(const acs_sbfs_args& A, int64_t j, int action, Key<W>& child, Key<W>& pk, int& L) {
    pk = load_key<W>(A.keys, (uint64_t)j);
    Rel<2 * W> r0, r1;
    split_key<W>(pk, r0, r1);
    bool co;
    const int st = A.trusted ? apply_move<2 * W, true>(r0, r1, action, A.mrl, A.cyclical != 0, co)
                             : apply_move<2 * W, false>(r0, r1, action, A.mrl, A.cyclical != 0, co);
    child = make_key<W>(r0, r1);
    L = r0.len + r1.len;
    return st;
}

// phase 0: count records per destination and resolve sol / err / first_len minima
// phase 1: write the records to the send buffers at the reserved offsets
template <int W, int PHASE>
__global__ void __launch_bounds__(kSbThreads) sb_expand_kernel(const acs_sbfs_args A) {
    __shared__ unsigned s_cnt[kMaxWorld];
    __shared__ unsigned long long s_base[kMaxWorld];
    if (threadIdx.x < kMaxWorld) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int64_t t = (int64_t)blockIdx.x * kSbThreads + threadIdx.x;
    const int64_t nloc = A.l1 - A.l0;
    int dest = -1;
    unsigned local_off = 0;
    Key<W> child, pk;
    uint32_t c = 0;
    if (t < nloc * 12) {
        const int64_t j = A.l0 + t / 12;
        const int a = (int)(t % 12);
        const uint64_t pg = (uint64_t)A.gid[j];
        const uint64_t gidc = pg * 12 + a;
        c = (uint32_t)((pg - (uint64_t)A.head) * 12 + a);
        int L;
        const int st = sb_child<W>(A, j, a, child, pk, L);
        if (st != ST_OK) {
            if (PHASE == 0) atomicMin(&A.ctrl[1], (gidc << 2) | (unsigned)st);
        } else {
            if (PHASE == 0) {
                if (L < A.min_len) atomicMin(&A.ctrl[2 + L], gidc);
                if (L == 2) atomicMin(&A.ctrl[0], gidc);
            }
            if (!key_eq<W>(child, pk)) {
                dest = owner_of(key_hash<W>(child), A.world);
                local_off = atomicAdd(&s_cnt[dest], 1u);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < A.world && s_cnt[threadIdx.x]) {
        if (PHASE == 0) atomicAdd(&A.dest_count[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
        else s_base[threadIdx.x] = atomicAdd(&A.dest_cursor[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
    }
    if (PHASE == 1) {
        __syncthreads();
        if (dest >= 0) {
            const uint64_t pos = s_base[dest] + local_off;
            store_key<W>(A.send_keys, pos, child);
            A.send_c[pos] = c;
        }
    }
}

template <int W>
__global__ void __launch_bounds__(256) sb_insert_kernel(const acs_sbfs_args A) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n_recv) return;
    const Key<W> key = load_key<W>(A.recv_keys, (uint64_t)i);
    const uint64_t c = A.recv_c[i];
    const uint64_t h = key_hash<W>(key);
    const uint64_t mine = kTentBit | (c << 37) | ((uint64_t)i << 11) | (h >> 53);
    uint64_t s = h & A.tmask;
    uint32_t my_slot = kNoSlot32;
    uint64_t probes = 0;
    for (;;) {
        uint64_t cur = __ldcg(&A.table[s]);
        if (cur == 0) {
            cur = atomicCAS((unsigned long long*)&A.table[s], 0ull, (unsigned long long)mine);
            if (cur == 0) {
                my_slot = (uint32_t)s;
                break;
            }
        }
        if (!(cur & kTentBit)) {  // committed node
            if (((cur >> 40) & 0x7FFFFFull) == (h >> 41)) {
                const Key<W> other = load_key<W>(A.keys, (cur & kIdxMask) - 1);
                if (key_eq<W>(other, key)) break;  // already visited
            }
        } else if ((cur & 0x7FFull) == (h >> 53)) {  // tentative record of this chunk
            const Key<W> other = load_key<W>(A.recv_keys, (cur >> 11) & kMask26);
            if (key_eq<W>(other, key)) {
                atomicMin((unsigned long long*)&A.table[s], (unsigned long long)mine);
                my_slot = (uint32_t)s;
                break;
            }
        }
        s = (s + 1) & A.tmask;
        if (++probes > A.tmask) {  // cannot happen with the host's chunk sizing
            atomicMin(&A.ctrl[1], 3ull);
            break;
        }
    }
    A.rec_slot[i] = my_slot;
}

__global__ void __launch_bounds__(256) sb_mark_kernel(const acs_sbfs_args A) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n_recv) return;
    const uint32_t s = A.rec_slot[i];
    if (s == kNoSlot32) return;
    const uint64_t cur = A.table[s];
    if ((cur & kTentBit) && ((cur >> 11) & kMask26) == (uint64_t)i) {
        const uint32_t c = A.recv_c[i];
        atomicOr(&A.bitmap_local[c >> 5], 1u << (c & 31));
    } else {
        A.rec_slot[i] = kNoSlot32;  // lost to an earlier candidate
    }
}

// Exclusive prefix of popcounts over nwords 32-bit words; prefix[nwords] = total.  Three passes
// (block sums -> scan of the block sums -> per-block prefixes), 2048 words per 256-thread block.
// (The first version scanned with ONE block: 60 % of the whole sharded search at budget 1e9.)
constexpr int kScanThreads = 256;
constexpr int kScanPerThread = 8;
constexpr int kScanBlockWords = kScanThreads * kScanPerThread;

__device__ __forceinline__ uint32_t scan_block_exclusive(uint32_t v, uint32_t& total) {
    __shared__ uint32_t wsum[kScanThreads / 32];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, x, off);
        if (lane >= off) x += t;
    }
    if (lane == 31) wsum[wid] = x;
    __syncthreads();
    uint32_t before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kScanThreads / 32; ++w) {
        const uint32_t s = wsum[w];
        if (w < (int)wid) before += s;
        tot += s;
    }
    __syncthreads();
    total = tot;
    return before + x - v;
}

__global__ void __launch_bounds__(kScanThreads) sb_scan_sums_kernel(const uint32_t* bitmap, uint32_t* block_sums,
                                                                    int64_t nwords) {
    const int64_t base = (int64_t)blockIdx.x * kScanBlockWords;
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < kScanPerThread; ++k) {
        const int64_t i = base + (int64_t)k * kScanThreads + threadIdx.x;  // coalesced
        if (i < nwords) s += __popc(bitmap[i]);
    }
    uint32_t total;
    scan_block_exclusive(s, total);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single block: exclusive scan of block_sums[0..nblocks) in place, grand total to *total_out
__global__ void __launch_bounds__(kScanThreads) sb_scan_top_kernel(uint32_t* block_sums, int64_t nblocks,
                                                                   uint32_t* total_out) {
    uint32_t carry = 0;
    for (int64_t base = 0; base < nblocks; base += kScanThreads) {
        const int64_t i = base + threadIdx.x;
        const uint32_t v = i < nblocks ? block_sums[i] : 0u;
        uint32_t total;
        const uint32_t ex = scan_block_exclusive(v, total);
        if (i < nblocks) block_sums[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(kScanThreads) sb_scan_final_kernel(const uint32_t* bitmap, const uint32_t* block_sums,
                                                                     uint32_t* prefix, int64_t nwords) {
    const int64_t first = (int64_t)blockIdx.x * kScanBlockWords + (int64_t)threadIdx.x * kScanPerThread;
    uint32_t c[kScanPerThread];
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < kScanPerThread; ++k) {
        c[k] = (first + k < nwords) ? __popc(bitmap[first + k]) : 0u;
        s += c[k];
    }
    uint32_t total;
    uint32_t run = block_sums[blockIdx.x] + scan_block_exclusive(s, total);
#pragma unroll
    for (int k = 0; k < kScanPerThread; ++k) {
        if (first + k < nwords) prefix[first + k] = run;
        run += c[k];
    }
}

__device__ __forceinline__ uint32_t bitmap_rank(const uint32_t* bitmap, const uint32_t* prefix, uint64_t c) {
    const uint32_t r = (uint32_t)(c & 31);
    // c may equal the bit count (one past the end): prefix has nwords+1 entries
    return prefix[c >> 5] + (r ? __popc(bitmap[c >> 5] & ((1u << r) - 1u)) : 0u);
}

// first chunk-local parent p with n_nodes + #winners(parents <= p) >= budget
__global__ void __launch_bounds__(256) sb_cut_kernel(const acs_sbfs_args A) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= A.nparents) return;
    const uint64_t incl = bitmap_rank(A.bitmap_global, A.prefix_global, (uint64_t)(p + 1) * 12);
    if ((uint64_t)A.n_nodes + incl >= (uint64_t)A.budget) atomicMin(A.cut, (unsigned long long)p);
}

// out[0] = global winners below limit, out[1] = local winners below limit
__global__ void sb_rank_at_kernel(const acs_sbfs_args A, unsigned long long* out) {
    out[0] = bitmap_rank(A.bitmap_global, A.prefix_global, (uint64_t)A.limit);
    out[1] = bitmap_rank(A.bitmap_local, A.prefix_local, (uint64_t)A.limit);
}

template <int W>
__global__ void __launch_bounds__(256) sb_commit_kernel(const acs_sbfs_args A) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n_recv) return;
    const uint32_t s = A.rec_slot[i];
    if (s == kNoSlot32) return;
    const uint64_t c = A.recv_c[i];
    if (c >= (uint64_t)A.limit) return;
    const uint64_t g = (uint64_t)A.n_nodes + bitmap_rank(A.bitmap_global, A.prefix_global, c);
    const uint64_t idx = (uint64_t)A.n_local + bitmap_rank(A.bitmap_local, A.prefix_local, c);
    const Key<W> key = load_key<W>(A.recv_keys, (uint64_t)i);
    store_key<W>(A.keys, idx, key);
    A.parent[idx] = (int64_t)((((uint64_t)A.head + c / 12) << 4) | (c % 12));
    A.gid[idx] = (int64_t)g;
    const uint64_t h = key_hash<W>(key);
    A.table[s] = ((h >> 41) << 40) | (idx + 1);
}

// smallest local index whose gid >= value (gid is increasing); one thread
__global__ void sb_lower_bound_kernel(const int64_t* gid, int64_t n, int64_t value, long long* out) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (gid[mid] < value) lo = mid + 1;
        else hi = mid;
    }
    *out = lo;
}

// out = {found, parent gid, action, total length} of the node with global id `value`
template <int W>
__global__ void sb_lookup_kernel(const acs_sbfs_args A, int64_t value, long long* out) {
    int64_t lo = 0, hi = A.n_local;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (A.gid[mid] < value) lo = mid + 1;
        else hi = mid;
    }
    out[0] = out[1] = out[2] = out[3] = 0;
    if (lo < A.n_local && A.gid[lo] == value) {
        const Key<W> k = load_key<W>(A.keys, (uint64_t)lo);
        out[0] = 1;
        out[1] = A.parent[lo] < 0 ? -1 : (A.parent[lo] >> 4);
        out[2] = A.parent[lo] < 0 ? -1 : (A.parent[lo] & 15);
        out[3] = key_total_len<W>(k);
    }
}

}  // namespace acs

using namespace acs;

#define SB_CHECK(A)                                                                  \
    if (!(A) || (A)->world < 1 || (A)->world > kMaxWorld || ((A)->W != 1 && (A)->W != 2)) { \
        acs::set_last_error("sbfs: bad argument block");                             \
        return ACS_ERR_INVALID;                                                      \
    }
// the error of the launches just made, if any
static int launched() {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? ACS_OK : cuda_fail(e, "sbfs launch");
}

extern "C" {

int acs_sbfs_pack_root(const int8_t* h_presentation, int mrl, uint64_t* key_out /*[4]*/, uint64_t* hash_out,
                       int* total_len, int* valid) {
    if (!h_presentation || !key_out || !hash_out || !total_len || !valid || mrl < 1 || mrl > kMaxKeyMrl)
        return ACS_ERR_INVALID;
    int lens[2];
    bool v;
    std::memset(key_out, 0, 4 * sizeof(uint64_t));
    if (key_words(mrl) == 1) {
        Key<1> k;
        if (!pack_root<1>(h_presentation, mrl, k, lens, v)) return ACS_ERR_UNSUPPORTED;
        std::memcpy(key_out, k.k, sizeof(k.k));
        *hash_out = key_hash<1>(k);
    } else {
        Key<2> k;
        if (!pack_root<2>(h_presentation, mrl, k, lens, v)) return ACS_ERR_UNSUPPORTED;
        std::memcpy(key_out, k.k, sizeof(k.k));
        *hash_out = key_hash<2>(k);
    }
    *total_len = lens[0] + lens[1];
    *valid = v ? 1 : 0;
    return ACS_OK;
}

int acs_sbfs_owner(uint64_t hash, int world) { return owner_of(hash, world); }

int acs_sbfs_expand(const acs_sbfs_args* A, int phase, void* stream) {
    SB_CHECK(A);
    const int64_t n = (A->l1 - A->l0) * 12;
    if (n <= 0) return ACS_OK;
    const unsigned blocks = (unsigned)((n + kSbThreads - 1) / kSbThreads);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (A->W == 1) {
        if (phase == 0) sb_expand_kernel<1, 0><<<blocks, kSbThreads, 0, s>>>(*A);
        else sb_expand_kernel<1, 1><<<blocks, kSbThreads, 0, s>>>(*A);
    } else {
        if (phase == 0) sb_expand_kernel<2, 0><<<blocks, kSbThreads, 0, s>>>(*A);
        else sb_expand_kernel<2, 1><<<blocks, kSbThreads, 0, s>>>(*A);
    }
    return launched();
}

int acs_sbfs_insert_mark(const acs_sbfs_args* A, void* stream) {
    SB_CHECK(A);
    if (A->n_recv <= 0) return ACS_OK;
    if (A->n_recv > (int64_t)kMask26) {
        acs::set_last_error("sbfs: more than 2^26 records in one chunk");
        return ACS_ERR_INVALID;
    }
    const unsigned blocks = (unsigned)((A->n_recv + 255) / 256);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (A->W == 1) sb_insert_kernel<1><<<blocks, 256, 0, s>>>(*A);
    else sb_insert_kernel<2><<<blocks, 256, 0, s>>>(*A);
    sb_mark_kernel<<<blocks, 256, 0, s>>>(*A);
    return launched();
}

int acs_sbfs_scan(const uint32_t* d_bitmap, uint32_t* d_prefix, int64_t nwords, void* stream) {
    if (!d_bitmap || !d_prefix || nwords < 0) return ACS_ERR_INVALID;
    // d_prefix holds nwords+1 prefixes followed by scratch for the block sums (see the header)
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t nblocks = (nwords + kScanBlockWords - 1) / kScanBlockWords;
    uint32_t* block_sums = d_prefix + nwords + 1;
    if (nblocks > 0) sb_scan_sums_kernel<<<(unsigned)nblocks, kScanThreads, 0, s>>>(d_bitmap, block_sums, nwords);
    sb_scan_top_kernel<<<1, kScanThreads, 0, s>>>(block_sums, nblocks, d_prefix + nwords);
    if (nblocks > 0)
        sb_scan_final_kernel<<<(unsigned)nblocks, kScanThreads, 0, s>>>(d_bitmap, block_sums, d_prefix, nwords);
    return launched();
}

int acs_sbfs_cut(const acs_sbfs_args* A, void* stream) {
    SB_CHECK(A);
    if (A->nparents <= 0) return ACS_OK;
    sb_cut_kernel<<<(unsigned)((A->nparents + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(*A);
    return launched();
}

int acs_sbfs_rank_at(const acs_sbfs_args* A, uint64_t* d_out2, void* stream) {
    SB_CHECK(A);
    sb_rank_at_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(*A, (unsigned long long*)d_out2);
    return launched();
}

int acs_sbfs_commit(const acs_sbfs_args* A, void* stream) {
    SB_CHECK(A);
    if (A->n_recv <= 0) return ACS_OK;
    const unsigned blocks = (unsigned)((A->n_recv + 255) / 256);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (A->W == 1) sb_commit_kernel<1><<<blocks, 256, 0, s>>>(*A);
    else sb_commit_kernel<2><<<blocks, 256, 0, s>>>(*A);
    return launched();
}

int acs_sbfs_lower_bound(const int64_t* d_gid, int64_t n, int64_t value, int64_t* d_out, void* stream) {
    if (!d_gid || !d_out || n < 0) return ACS_ERR_INVALID;
    sb_lower_bound_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(d_gid, n, value, (long long*)d_out);
    return launched();
}

int acs_sbfs_lookup(const acs_sbfs_args* A, int64_t gid, int64_t* d_out4, void* stream) {
    SB_CHECK(A);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (A->W == 1) sb_lookup_kernel<1><<<1, 1, 0, s>>>(*A, gid, (long long*)d_out4);
    else sb_lookup_kernel<2><<<1, 1, 0, s>>>(*A, gid, (long long*)d_out4);
    return launched();
}

int acs_sbfs_unpack(const uint64_t* d_keys, int8_t* d_out, int64_t n, int mrl, void* stream) {
    if (n <= 0) return ACS_OK;
    if (!d_keys || !d_out || mrl < 1 || mrl > kMaxKeyMrl) return ACS_ERR_INVALID;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (key_words(mrl) == 1) records_unpack_kernel<1><<<blocks, 256, 0, s>>>(d_keys, 2, nullptr, d_out, (uint64_t)n, mrl);
    else records_unpack_kernel<2><<<blocks, 256, 0, s>>>(d_keys, 4, nullptr, d_out, (uint64_t)n, mrl);
    return launched();
}

}  // extern "C"
