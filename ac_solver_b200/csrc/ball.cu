// ball.cu -- breadth-first exploration of the AC graph in the state model of the reference's
// `barcode_analysis` C++ tools (SURVEY 8f-3), on the GPU:
//   barcode_analysis/5_steps_neibourhoods/neibourhoods.cpp:18-54     size of the radius-r ball
//   barcode_analysis/simplex_data_generation/*/ac_bfs.cpp:36-91      0/1-simplices + filtrations
//   .../AC_UTILS_no_hash.cpp, .../AC_UTILS_as_sets.h                  the moves and the state order
// (paths relative to /root/reference).  That model differs from the Python path: a state is an
// UNORDERED pair of relators (kept sorted: shorter first, then lexicographic on the integers
// -2 < -1 < 1 < 2), relators have no length cap, every move is followed by FULL free reduction,
// there is no cyclic reduction; 12 "prime" moves or 14 "classic" moves.
//
// Same search substrate as the other searches here: chunks of consecutive BFS nodes, one thread
// per candidate (node, move) with candidate id c = K*position + move, children written to a
// candidate buffer, exact open-addressing table with smallest-candidate-id-wins (so the node
// numbering is the reference's FIFO discovery order, which the simplex dump needs), ballot/popc
// ranking, ordered commit.  Relators are variable-length byte strings (a ball of radius 5 around
// a Miller-Schupp presentation holds words of a few hundred letters), so this engine works in
// the byte domain with a fixed per-run stride instead of the 2-bit packed registers.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "acs_internal.h"

namespace acs {

constexpr int kBallThreads = 128;
constexpr uint64_t kBallIdxMask = (1ull << 40) - 1;

struct BallArgs {
    int8_t* nodes;      // [cap][stride]  rel1 letters [0,L), rel2 letters [L,2L)
    uint16_t* lens;     // [cap][2]
    uint8_t* level;     // [cap]
    uint32_t* root_of;  // [cap]  index of the start presentation this node was reached from (multi-root runs)
    uint64_t* table;    // [tmask+1]  fp24 << 40 | index+1 ; index >= n_nodes: tentative candidate n_nodes + c
    uint64_t tmask;
    int8_t* cand;       // [ccap][stride]
    uint16_t* cand_lens;  // [ccap][2]   0xFFFF,0xFFFF = filtered out (size cap) / not generated
    uint32_t* cand_slot;  // [ccap]
    uint32_t* cand_node;  // [ccap]  node index of the candidate's state (visited, or newly numbered)
    uint32_t* rank;     // [ccap+1] exclusive winner prefix
    uint8_t* win;       // [ccap]
    unsigned long long* ctrl;  // [0] overflow flag (relator longer than L), [1] winners, [2] edges
    uint32_t* edges;    // [ecap][3]  (cn, cc, filtration) in candidate order
    uint64_t lo;        // first parent of the chunk
    uint64_t nparents, n_nodes;
    int L, K, classic, size_cap, want_edges;
    int literal;        // some start word is not freely reduced: restate the reference's reduce_ pass by pass (see ball_move)
};

__device__ __forceinline__ bool rel_less(const int8_t* x, int lx, const int8_t* y, int ly) {
    if (lx != ly) return lx < ly;
    for (int i = 0; i < lx; ++i)
        if (x[i] != y[i]) return x[i] < y[i];
    return false;
}
__host__ __device__ __forceinline__ uint64_t ball_hash(const int8_t* r1, int l1, const int8_t* r2, int l2, uint32_t root) {
    uint64_t h = (0xcbf29ce484222325ull ^ ((uint64_t)l1 << 32 | (uint64_t)l2)) + 0x9E3779B97F4A7C15ull * root;
    for (int i = 0; i < l1; ++i) h = (h ^ (uint8_t)r1[i]) * 0x100000001b3ull;
    h = (h ^ 0xFF) * 0x100000001b3ull;
    for (int i = 0; i < l2; ++i) h = (h ^ (uint8_t)r2[i]) * 0x100000001b3ull;
    h ^= h >> 29;
    h *= 0xbf58476d1ce4e5b9ull;
    h ^= h >> 32;
    return h;
}
// append letter v to the freely reduced word out[0..n): returns the new length
__device__ __forceinline__ int push_reduced(int8_t* out, int n, int8_t v) {
    if (n > 0 && out[n - 1] == -v) return n - 1;
    out[n] = v;
    return n + 1;
}
// The reference's reduce0_ (AC_UTILS_no_hash.cpp:58-79), literally: one left-to-right pass that drops adjacent
// inverse pairs, and keeps the last letter iff it does not cancel against its LEFT NEIGHBOUR IN THE INPUT -- also
// when that neighbour was already consumed by a pair (so [.., X, x, X] loses its last letter although free
// reduction keeps it).  reduce_ (:81-88) repeats the pass until nothing changes.  On a concatenation / conjugation
// of freely reduced words the fixpoint IS the free reduction (the odd case needs x X x at the end of the input),
// so the fast path below uses a stack; only runs that start from a non-reduced word take this literal path.
__device__ int reduce_literal(int8_t* w, int n, int8_t* tmp) {
    int8_t* cur = w;
    int8_t* nxt = tmp;
    for (;;) {
        int m = 0;
        if (n < 2) {
            m = n;
            if (n == 1) nxt[0] = cur[0];
        } else {
            int j = 0;
            while (j < n - 1) {
                if (cur[j] + cur[j + 1] == 0) j += 2;
                else nxt[m++] = cur[j++];
            }
            if (cur[n - 1] + cur[n - 2] != 0) nxt[m++] = cur[n - 1];
        }
        int8_t* t = cur;
        cur = nxt;
        nxt = t;
        if (m == n) break;  // a pass that removes nothing returns its input
        n = m;
    }
    if (cur != w)
        for (int i = 0; i < n; ++i) w[i] = cur[i];
    return n;
}

// child of (r1, r2) under move t (AC_UTILS_no_hash.cpp:153-211, AC_UTILS_as_sets.h:337-362); the
// changed relator is built fully reduced in `nw` (capacity 2L+2); returns its length, `which` = 0/1.
// literal: build the raw word and reduce it with the reference's own pass structure (tmp: second buffer).
__device__ int ball_move(const int8_t* r1, int l1, const int8_t* r2, int l2, int t, bool classic, int8_t* nw, int& which,
                         bool literal, int8_t* tmp) {
    // decode: op 0 = concat(x, y), 1 = concat(x, inv y), 2 = conj(x, g), 3 = inv(x)
    int op, tgt, g = 0;
    bool other_first = false;  // concat(other, target) instead of concat(target, other)
    if (classic) {
        // 0: (r1 r2, r2) 1: (r2 r1, r2) 2: (r1, r1 r2) 3: (r1, r2 r1) 4-7: conj r2 by a,b,A,B 8-11: conj r1 12: inv r1 13: inv r2
        if (t < 4) {
            op = 0;
            tgt = t >> 1;
            other_first = (t == 1) || (t == 2);
        } else if (t < 12) {
            op = 2;
            tgt = t < 8 ? 1 : 0;
            const int gs[4] = {1, 2, -1, -2};
            g = gs[t & 3];
        } else {
            op = 3;
            tgt = t - 12;
        }
    } else {
        // 0: (r1 r2, r2) 1: (r1, r2 r1) 2: (r1 r2^-1, r2) 3: (r1, r2 r1^-1) 4-7: conj r1 by B,A,a,b 8-11: conj r2
        if (t < 4) {
            op = t < 2 ? 0 : 1;
            tgt = t & 1;
        } else {
            op = 2;
            tgt = t < 8 ? 0 : 1;
            const int gs[4] = {-2, -1, 1, 2};
            g = gs[t & 3];
        }
    }
    which = tgt;
    const int8_t* x = tgt ? r2 : r1;
    const int lx = tgt ? l2 : l1;
    const int8_t* y = tgt ? r1 : r2;
    const int ly = tgt ? l1 : l2;
    int n = 0;
    if (literal) {
        // raw words exactly as concat_ / conj0_ / inv0_ assemble them; inv0_ alone does not reduce (:104-110)
        if (op == 0) {
            const int8_t* p = other_first ? y : x;
            const int lp = other_first ? ly : lx;
            const int8_t* q = other_first ? x : y;
            const int lq = other_first ? lx : ly;
            for (int i = 0; i < lp; ++i) nw[n++] = p[i];
            for (int i = 0; i < lq; ++i) nw[n++] = q[i];
        } else if (op == 1) {
            for (int i = 0; i < lx; ++i) nw[n++] = x[i];
            for (int i = ly - 1; i >= 0; --i) nw[n++] = (int8_t)-y[i];
        } else if (op == 2) {
            nw[n++] = (int8_t)-g;
            for (int i = 0; i < lx; ++i) nw[n++] = x[i];
            nw[n++] = (int8_t)g;
        } else {
            for (int i = lx - 1; i >= 0; --i) nw[n++] = (int8_t)-x[i];
            return n;
        }
        return reduce_literal(nw, n, tmp);
    }
    if (op == 0) {
        if (other_first) {
            for (int i = 0; i < ly; ++i) n = push_reduced(nw, n, y[i]);
            for (int i = 0; i < lx; ++i) n = push_reduced(nw, n, x[i]);
        } else {
            for (int i = 0; i < lx; ++i) n = push_reduced(nw, n, x[i]);
            for (int i = 0; i < ly; ++i) n = push_reduced(nw, n, y[i]);
        }
    } else if (op == 1) {  // x * inverse(y)
        for (int i = 0; i < lx; ++i) n = push_reduced(nw, n, x[i]);
        for (int i = ly - 1; i >= 0; --i) n = push_reduced(nw, n, (int8_t)-y[i]);
    } else if (op == 2) {  // conj0_(x, g) = g^-1 x g
        n = push_reduced(nw, n, (int8_t)-g);
        for (int i = 0; i < lx; ++i) n = push_reduced(nw, n, x[i]);
        n = push_reduced(nw, n, (int8_t)g);
    } else {  // inverse
        for (int i = lx - 1; i >= 0; --i) n = push_reduced(nw, n, (int8_t)-x[i]);
    }
    return n;
}

// one thread per candidate: child, canonical order, candidate buffer
__global__ void __launch_bounds__(kBallThreads) ball_expand_kernel(const BallArgs A) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= A.nparents * A.K) return;
    const uint64_t p = A.lo + c / A.K;
    const int t = (int)(c % A.K);
    const int L = A.L;
    const int8_t* r1 = A.nodes + p * 2 * L;
    const int8_t* r2 = r1 + L;
    const int l1 = A.lens[2 * p], l2 = A.lens[2 * p + 1];
    int8_t nw[1026];  // local memory; L <= 512
    int8_t tmp[1026];  // second buffer of the literal reduction (untouched on the fast path)
    int which;
    const int n = ball_move(r1, l1, r2, l2, t, A.classic != 0, nw, which, A.literal != 0, tmp);
    uint16_t o1 = 0xFFFF, o2 = 0xFFFF;
    if (n > L) {
        // with a size cap the stride IS the cap: such a child is simply too long (ac_bfs.cpp:60); without one
        // the stride was sized from the radius and this cannot happen short of the 512-letter limit
        if (A.size_cap <= 0) atomicExch(&A.ctrl[0], 1ull);
    } else {
        const int8_t* a = which == 0 ? nw : r1;
        const int la = which == 0 ? n : l1;
        const int8_t* b = which == 0 ? r2 : nw;
        const int lb = which == 0 ? l2 : n;
        if (!(A.size_cap > 0 && la + lb > A.size_cap)) {
            const bool keep = rel_less(a, la, b, lb);  // sort_: (a, b) if a < b else (b, a)
            const int8_t* f = keep ? a : b;
            const int lf = keep ? la : lb;
            const int8_t* s = keep ? b : a;
            const int ls = keep ? lb : la;
            int8_t* dst = A.cand + c * 2 * L;
            for (int i = 0; i < lf; ++i) dst[i] = f[i];
            for (int i = 0; i < ls; ++i) dst[L + i] = s[i];
            o1 = (uint16_t)lf;
            o2 = (uint16_t)ls;
        }
    }
    A.cand_lens[2 * c] = o1;
    A.cand_lens[2 * c + 1] = o2;
}

__device__ __forceinline__ bool ball_same(const int8_t* x, const uint16_t* xl, const int8_t* y, const uint16_t* yl, int L) {
    if (xl[0] != yl[0] || xl[1] != yl[1]) return false;
    for (int i = 0; i < xl[0]; ++i)
        if (x[i] != y[i]) return false;
    for (int i = 0; i < xl[1]; ++i)
        if (x[L + i] != y[L + i]) return false;
    return true;
}

// exact dedup, smallest candidate id wins among the candidates of the chunk
__global__ void __launch_bounds__(kBallThreads) ball_insert_kernel(const BallArgs A) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= A.nparents * A.K) return;
    const int L = A.L;
    const uint16_t* cl = A.cand_lens + 2 * c;
    uint32_t my_slot = 0xFFFFFFFFu;
    if (cl[0] != 0xFFFF) {
        const int8_t* me = A.cand + c * 2 * L;
        const uint32_t my_root = A.root_of[A.lo + c / A.K];
        const uint64_t h = ball_hash(me, cl[0], me + L, cl[1], my_root);
        const uint64_t fp = h >> 40;
        const uint64_t mine = (fp << 40) | (A.n_nodes + c + 1);
        for (uint64_t s = h & A.tmask;; s = (s + 1) & A.tmask) {
            uint64_t cur = __ldcg(&A.table[s]);
            if (cur == 0) {
                cur = atomicCAS((unsigned long long*)&A.table[s], 0ull, (unsigned long long)mine);
                if (cur == 0) {
                    my_slot = (uint32_t)s;
                    break;
                }
            }
            if ((cur >> 40) == fp) {
                const uint64_t idx = (cur & kBallIdxMask) - 1;
                const bool same = idx < A.n_nodes
                                      ? (A.root_of[idx] == my_root && ball_same(me, cl, A.nodes + idx * 2 * L, A.lens + 2 * idx, L))
                                      : (A.root_of[A.lo + (idx - A.n_nodes) / A.K] == my_root &&
                                         ball_same(me, cl, A.cand + (idx - A.n_nodes) * 2 * L, A.cand_lens + 2 * (idx - A.n_nodes), L));
                if (same) {
                    if (idx >= A.n_nodes) atomicMin((unsigned long long*)&A.table[s], (unsigned long long)mine);
                    my_slot = (uint32_t)s;
                    break;
                }
            }
        }
    }
    A.cand_slot[c] = my_slot;
}

// winners (the candidate whose id the slot still holds), single-block exclusive prefix
__global__ void __launch_bounds__(1024) ball_rank_kernel(const BallArgs A) {
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t carry;
    const uint64_t n = A.nparents * A.K;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint64_t base = 0; base < n; base += blockDim.x) {
        const uint64_t c = base + threadIdx.x;
        bool w = false;
        if (c < n && A.cand_slot[c] != 0xFFFFFFFFu) {
            const uint64_t idx = (__ldcg(&A.table[A.cand_slot[c]]) & kBallIdxMask) - 1;
            w = idx == A.n_nodes + c;
        }
        if (c < n) A.win[c] = w ? 1 : 0;
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, w);
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        if (lane == 0) warp_sum[wid] = __popc(bal);
        __syncthreads();
        uint32_t before = carry + __popc(bal & ((1u << lane) - 1u)), tot = 0;
        for (int k = 0; k < 32; ++k) {
            if (k < wid) before += warp_sum[k];
            tot += warp_sum[k];
        }
        if (c < n) A.rank[c] = before;
        __syncthreads();
        if (threadIdx.x == 0) carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        A.rank[n] = carry;
        A.ctrl[1] = carry;
    }
}

// node index of every candidate's state; winners are appended in candidate order (FIFO discovery order)
__global__ void __launch_bounds__(kBallThreads) ball_commit_kernel(const BallArgs A, int next_level) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= A.nparents * A.K) return;
    const uint32_t slot = A.cand_slot[c];
    if (slot == 0xFFFFFFFFu) {
        A.cand_node[c] = 0xFFFFFFFFu;
        return;
    }
    const uint64_t cur = __ldcg(&A.table[slot]);
    const uint64_t idx = (cur & kBallIdxMask) - 1;
    if (idx < A.n_nodes) {
        A.cand_node[c] = (uint32_t)idx;  // already visited
        return;
    }
    const uint64_t holder = idx - A.n_nodes;  // the winning candidate of this state
    const uint64_t node = A.n_nodes + A.rank[holder];
    A.cand_node[c] = (uint32_t)node;
    if (holder == c) {
        const int L = A.L;
        const int8_t* src = A.cand + c * 2 * L;
        int8_t* dst = A.nodes + node * 2 * L;
        const int l1 = A.cand_lens[2 * c], l2 = A.cand_lens[2 * c + 1];
        for (int i = 0; i < l1; ++i) dst[i] = src[i];
        for (int i = 0; i < l2; ++i) dst[L + i] = src[L + i];
        A.lens[2 * node] = (uint16_t)l1;
        A.lens[2 * node + 1] = (uint16_t)l2;
        A.level[node] = (uint8_t)next_level;
        A.root_of[node] = A.root_of[A.lo + c / A.K];
    }
}
// second pass (after every winner's rank is final): re-point the table slots at the nodes
__global__ void __launch_bounds__(kBallThreads) ball_fix_kernel(const BallArgs A) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= A.nparents * A.K || !A.win[c]) return;
    const uint32_t slot = A.cand_slot[c];
    const uint64_t cur = A.table[slot];
    A.table[slot] = (cur & ~kBallIdxMask) | (A.n_nodes + A.rank[c] + 1);
}

// 1-simplices in the reference's output order (ac_bfs.cpp:73-80): one per candidate with cn < cc
__global__ void __launch_bounds__(1024) ball_edges_kernel(const BallArgs A, uint64_t edge_base) {
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t carry;
    const uint64_t n = A.nparents * A.K;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint64_t base = 0; base < n; base += blockDim.x) {
        const uint64_t c = base + threadIdx.x;
        bool e = false;
        uint32_t cn = 0, cc = 0;
        if (c < n && A.cand_node[c] != 0xFFFFFFFFu) {
            cn = (uint32_t)(A.lo + c / A.K);
            cc = A.cand_node[c];
            e = cn < cc;
        }
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, e);
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        if (lane == 0) warp_sum[wid] = __popc(bal);
        __syncthreads();
        uint32_t before = carry + __popc(bal & ((1u << lane) - 1u)), tot = 0;
        for (int k = 0; k < 32; ++k) {
            if (k < wid) before += warp_sum[k];
            tot += warp_sum[k];
        }
        if (e) {
            uint32_t* o = A.edges + (edge_base + before) * 3;
            const uint32_t sp = (uint32_t)A.lens[2 * cn] + A.lens[2 * cn + 1];
            const uint32_t sc = (uint32_t)A.cand_lens[2 * c] + A.cand_lens[2 * c + 1];
            o[0] = cn;
            o[1] = cc;
            o[2] = max(sp, sc);
        }
        __syncthreads();
        if (threadIdx.x == 0) carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) A.ctrl[2] = carry;
}

// the start presentations (nodes 0 .. n_roots-1) enter the visited table
__global__ void __launch_bounds__(256) ball_roots_kernel(const BallArgs A, int n_roots) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_roots) return;
    const int8_t* row = A.nodes + (uint64_t)r * 2 * A.L;
    const uint64_t h = ball_hash(row, A.lens[2 * r], row + A.L, A.lens[2 * r + 1], (uint32_t)r);
    const unsigned long long v = ((h >> 40) << 40) | (unsigned long long)(r + 1);
    for (uint64_t s = h & A.tmask;; s = (s + 1) & A.tmask)  // distinct (root, state) keys: plain linear probing
        if (atomicCAS((unsigned long long*)&A.table[s], 0ull, v) == 0ull) break;
}

// nodes per start presentation
__global__ void __launch_bounds__(256) ball_count_kernel(const uint32_t* root_of, uint64_t n, unsigned long long* counts) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(&counts[root_of[i]], 1ull);
}

}  // namespace acs

using namespace acs;

namespace {

// Breadth-first exploration from n_roots start presentations at once (each node carries its root's index, and
// the visited set is keyed by (root, state), so the runs are independent but share every kernel launch).
// Root r: letters h_letters[off[2r] .. off[2r+1]) and [off[2r+1] .. off[2r+2]).
int ball_run(int device, const int8_t* h_letters, const int64_t* off, int n_roots, int radius, int size_cap, int classic,
             int64_t max_nodes, int64_t* n_nodes_out, int64_t* h_counts, uint16_t* h_sizes, uint8_t* h_levels,
             int64_t cap_nodes, uint32_t* h_edges, int64_t cap_edges, int64_t* n_edges_out) {
    if (!h_letters || !off || n_roots < 1 || max_nodes < n_roots) return fail(ACS_ERR_INVALID, "ball: bad argument");
    if (max_nodes > (int64_t)3500000000ll) return fail(ACS_ERR_UNSUPPORTED, "ball: node indices are 32-bit (max_nodes <= 3.5e9)");
    if (const int rc = open_device(device, "ball")) return rc;
    int max_len = 1;
    for (int r = 0; r < n_roots; ++r) {
        const int64_t a = off[2 * r], b = off[2 * r + 1], c = off[2 * r + 2];
        if (a > b || b > c) return fail(ACS_ERR_INVALID, "ball: offsets must be non-decreasing");
        max_len = std::max<int>(max_len, (int)std::max(b - a, c - b));
    }
    for (int64_t i = 0; i < off[2 * n_roots]; ++i)
        if (h_letters[i] == 0 || h_letters[i] < -2 || h_letters[i] > 2) return fail(ACS_ERR_INVALID, "ball: letters must be +-1, +-2");
    bool literal = false;  // a start word with an adjacent inverse pair: the whole run follows the reference's reduce_ literally
    for (int k = 0; k < 2 * n_roots && !literal; ++k)
        for (int64_t i = off[k]; i + 1 < off[k + 1]; ++i)
            if (h_letters[i] + h_letters[i + 1] == 0) literal = true;
    const int K = classic ? 14 : 12;
    // stride: a relator at most doubles per move (concatenation); radius-bounded runs size it from the start
    int L = size_cap > 0 ? size_cap : max_len;
    if (size_cap <= 0) {
        int a = max_len, b = max_len;
        for (int r = 0; r < std::max(radius, 0); ++r) {  // concatenation adds the other relator, conjugation 2 letters
            const int s2 = std::max(a + b, std::max(a, b) + 2);
            b = std::max(a, b);
            a = s2;
        }
        L = std::max(a, b) + 2;
    }
    L = (std::min(std::max(L, 4), 512) + 3) / 4 * 4;
    const uint64_t cap = (uint64_t)max_nodes + 16;
    uint64_t tcap = 1024;
    const uint64_t chunk = n_roots > 1 ? 32768 : 8192;
    const uint64_t ccap = chunk * K;
    while (tcap < 2 * (cap + ccap)) tcap <<= 1;  // committed nodes + the tentative entries of one chunk, half full
    BallArgs A{};
    uint32_t* d_edges = nullptr;
    unsigned long long* d_counts = nullptr;
    auto free_all = [&]() {
        cudaFree(A.nodes);
        cudaFree(A.lens);
        cudaFree(A.level);
        cudaFree(A.root_of);
        cudaFree(A.table);
        cudaFree(A.cand);
        cudaFree(A.cand_lens);
        cudaFree(A.cand_slot);
        cudaFree(A.cand_node);
        cudaFree(A.rank);
        cudaFree(A.win);
        cudaFree(A.ctrl);
        cudaFree(d_edges);
        cudaFree(d_counts);
    };
    struct FreeOnExit {  // every return from here on releases the device buffers
        decltype(free_all)& f;
        ~FreeOnExit() { f(); }
    } free_on_exit{free_all};
    ACS_CUDA(cudaMalloc((void**)&A.nodes, cap * 2 * L));
    ACS_CUDA(cudaMalloc((void**)&A.lens, cap * 4));
    ACS_CUDA(cudaMalloc((void**)&A.level, cap));
    ACS_CUDA(cudaMalloc((void**)&A.root_of, cap * 4));
    ACS_CUDA(cudaMalloc((void**)&A.table, tcap * 8));
    ACS_CUDA(cudaMalloc((void**)&A.cand, ccap * 2 * L));
    ACS_CUDA(cudaMalloc((void**)&A.cand_lens, ccap * 4));
    ACS_CUDA(cudaMalloc((void**)&A.cand_slot, ccap * 4));
    ACS_CUDA(cudaMalloc((void**)&A.cand_node, ccap * 4));
    ACS_CUDA(cudaMalloc((void**)&A.rank, (ccap + 1) * 4));
    ACS_CUDA(cudaMalloc((void**)&A.win, ccap));
    ACS_CUDA(cudaMalloc((void**)&A.ctrl, 4 * 8));
    const bool want_edges = h_edges != nullptr && cap_edges > 0;
    if (want_edges) ACS_CUDA(cudaMalloc((void**)&d_edges, ccap * 3 * 4));
    A.edges = d_edges;
    A.tmask = tcap - 1;
    A.L = L;
    A.K = K;
    A.classic = classic ? 1 : 0;
    A.size_cap = size_cap;
    A.want_edges = want_edges ? 1 : 0;
    A.literal = literal ? 1 : 0;
    ACS_CUDA(cudaMemset(A.table, 0, tcap * 8));
    ACS_CUDA(cudaMemset(A.ctrl, 0, 32));
    // roots: the sorted pairs (sort_, AC_UTILS_no_hash.cpp:131-147) as nodes 0 .. n_roots-1, level 0
    {
        std::vector<int8_t> rows((size_t)n_roots * 2 * L, 0);
        std::vector<uint16_t> lens((size_t)n_roots * 2);
        std::vector<uint32_t> roots((size_t)n_roots);
        auto less = [](const int8_t* p, int lp, const int8_t* q, int lq) {
            if (lp != lq) return lp < lq;
            for (int i = 0; i < lp; ++i)
                if (p[i] != q[i]) return p[i] < q[i];
            return false;
        };
        for (int r = 0; r < n_roots; ++r) {
            const int8_t* x = h_letters + off[2 * r];
            const int8_t* y = h_letters + off[2 * r + 1];
            const int len1 = (int)(off[2 * r + 1] - off[2 * r]), len2 = (int)(off[2 * r + 2] - off[2 * r + 1]);
            const bool keep = less(x, len1, y, len2);
            const int8_t* f = keep ? x : y;
            const int lf = keep ? len1 : len2;
            const int8_t* sd = keep ? y : x;
            const int ls = keep ? len2 : len1;
            if (lf > L || ls > L)
                return fail(ACS_ERR_UNSUPPORTED, "ball: relators longer than 512 letters are not supported");
            int8_t* row = rows.data() + (size_t)r * 2 * L;
            std::memcpy(row, f, lf);
            std::memcpy(row + L, sd, ls);
            lens[2 * r] = (uint16_t)lf;
            lens[2 * r + 1] = (uint16_t)ls;
            roots[r] = (uint32_t)r;
        }
        ACS_CUDA(cudaMemcpy(A.nodes, rows.data(), rows.size(), cudaMemcpyHostToDevice));
        ACS_CUDA(cudaMemcpy(A.lens, lens.data(), lens.size() * 2, cudaMemcpyHostToDevice));
        ACS_CUDA(cudaMemset(A.level, 0, n_roots));
        ACS_CUDA(cudaMemcpy(A.root_of, roots.data(), roots.size() * 4, cudaMemcpyHostToDevice));
        ball_roots_kernel<<<(n_roots + 255) / 256, 256>>>(A, n_roots);
    }
    uint64_t n_nodes = (uint64_t)n_roots, head = 0, level_end = (uint64_t)n_roots;
    int level = 0;
    int64_t n_edges = 0;
    while (head < n_nodes) {
        if (head == level_end) {
            level_end = n_nodes;
            ++level;
        }
        if (radius >= 0 && level >= radius) break;  // nodes at distance `radius` are not expanded
        const uint64_t F = std::min<uint64_t>(level_end - head, chunk);
        A.lo = head;
        A.nparents = F;
        A.n_nodes = n_nodes;
        const unsigned blocks = (unsigned)((F * K + kBallThreads - 1) / kBallThreads);
        ball_expand_kernel<<<blocks, kBallThreads>>>(A);
        ball_insert_kernel<<<blocks, kBallThreads>>>(A);
        ball_rank_kernel<<<1, 1024>>>(A);
        ball_commit_kernel<<<blocks, kBallThreads>>>(A, level + 1);
        ball_fix_kernel<<<blocks, kBallThreads>>>(A);
        if (want_edges) ball_edges_kernel<<<1, 1024>>>(A, 0);
        unsigned long long ctrl[4];
        ACS_CUDA(cudaMemcpy(ctrl, A.ctrl, 32, cudaMemcpyDeviceToHost));
        if (ctrl[0])
            return fail(ACS_ERR_UNSUPPORTED, "ball: a relator outgrew the 512-letter stride");
        if (n_nodes + ctrl[1] > cap) return fail(ACS_ERR_NOMEM, "ball: more states than max_nodes");
        if (want_edges && ctrl[2]) {
            const int64_t ne = (int64_t)ctrl[2];
            if (n_edges + ne > cap_edges)
                return fail(ACS_ERR_NOMEM, "ball: more edges than cap_edges");
            ACS_CUDA(cudaMemcpy(h_edges + 3 * n_edges, d_edges, (size_t)ne * 12, cudaMemcpyDeviceToHost));
            n_edges += ne;
        }
        n_nodes += ctrl[1];
        head += F;
    }
    if (n_nodes_out) *n_nodes_out = (int64_t)n_nodes;
    if (n_edges_out) *n_edges_out = n_edges;
    if (h_counts) {
        ACS_CUDA(cudaMalloc((void**)&d_counts, (size_t)n_roots * 8));
        ACS_CUDA(cudaMemset(d_counts, 0, (size_t)n_roots * 8));
        ball_count_kernel<<<(unsigned)((n_nodes + 255) / 256), 256>>>(A.root_of, n_nodes, d_counts);
        ACS_CUDA(cudaMemcpy(h_counts, d_counts, (size_t)n_roots * 8, cudaMemcpyDeviceToHost));
    }
    const uint64_t ncopy = std::min<uint64_t>(n_nodes, (uint64_t)std::max<int64_t>(cap_nodes, 0));
    if (h_sizes && ncopy) {
        std::vector<uint16_t> lens(2 * ncopy);
        ACS_CUDA(cudaMemcpy(lens.data(), A.lens, ncopy * 4, cudaMemcpyDeviceToHost));
        for (uint64_t i = 0; i < ncopy; ++i) h_sizes[i] = (uint16_t)(lens[2 * i] + lens[2 * i + 1]);
    }
    if (h_levels && ncopy) ACS_CUDA(cudaMemcpy(h_levels, A.level, ncopy, cudaMemcpyDeviceToHost));
    return ACS_OK;
}

}  // namespace

extern "C" {

/* Explores the AC graph of the barcode_analysis state model breadth first from (r1, r2).
 *   radius >= 0 : all states within `radius` moves (neibourhoods.cpp:18-54); size_cap == 0
 *   size_cap > 0: all states of total length <= size_cap reachable through such states
 *                 (ac_bfs.cpp:36-91, radius < 0 = unbounded)
 * h_letters: r1 then r2 as int8 letters (lengths len1, len2), classic = 14 moves, else the 12 prime moves.
 * Outputs (any may be NULL): *n_nodes; node sizes / levels in discovery order (capacity cap_nodes);
 * edges (cn, cc, filtration) triples in the reference's output order (capacity cap_edges), *n_edges.
 * Returns ACS_ERR_NOMEM if max_nodes is exceeded. */
int acs_ball_explore(int device, const int8_t* h_letters, int len1, int len2, int radius, int size_cap, int classic,
                     int64_t max_nodes, int64_t* n_nodes_out, uint16_t* h_sizes, uint8_t* h_levels, int64_t cap_nodes,
                     uint32_t* h_edges, int64_t cap_edges, int64_t* n_edges_out) {
    if (!h_letters || len1 < 0 || len2 < 0 || max_nodes < 1) return fail(ACS_ERR_INVALID, "ball: bad argument");
    const int64_t off[3] = {0, len1, (int64_t)len1 + len2};
    return ball_run(device, h_letters, off, 1, radius, size_cap, classic, max_nodes, n_nodes_out, nullptr, h_sizes, h_levels,
                    cap_nodes, h_edges, cap_edges, n_edges_out);
}

/* neibourhoods.cpp read_do_and_write (:58-103) for a whole input file at once: the radius-`radius` ball sizes of
 * n_roots presentations in ONE exploration (all balls advance level by level in the same kernel launches).
 * Root r = letters [h_off[2r], h_off[2r+1]) and [h_off[2r+1], h_off[2r+2]) of h_letters; h_counts[n_roots].
 * max_nodes bounds the SUM of the ball sizes (ACS_ERR_NOMEM if exceeded: split the batch). */
int acs_ball_sizes(int device, const int8_t* h_letters, const int64_t* h_off, int n_roots, int radius, int classic,
                   int64_t max_nodes, int64_t* h_counts) {
    if (!h_counts || radius < 0) return fail(ACS_ERR_INVALID, "ball: bad argument");
    return ball_run(device, h_letters, h_off, n_roots, radius, 0, classic, max_nodes, nullptr, h_counts, nullptr, nullptr, 0,
                    nullptr, 0, nullptr);
}

}  // extern "C"
