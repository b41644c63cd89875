// mb_host.cuh -- the host half of the engines built on MbEngine (mbfs.cu, beam.cu): the driver's stream,
// events and pinned ring, the common device arrays, root packing, the run prologue and epilogue, the lagging
// poll of the run state, paths, visited rows and goal sets.  Each engine keeps its own plan, its extra arrays
// and the kernel launches of its chunk; the launches here are instantiated in the engine's translation unit.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "ac_keys.cuh"
#include "ac_sym.cuh"
#include "acs_internal.h"
#include "goalset.cuh"
#include "mb_engine.cuh"

namespace acs {

// the host enqueues chunks ahead of the device and reads the run state copied kMbLag chunks earlier
constexpr int kMbRing = 4, kMbLag = 2;

struct MbHost {
    int device = 0, n_search = 0, mrl = 0, W = 1, cyclical = 0;
    std::vector<int64_t> budgets;
    std::vector<MbSearch> h_final;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ring_ev[kMbRing] = {};
    MbState* h_ring = nullptr;  // pinned [kMbRing]
    int sms = 148;
    uint64_t* d_roots = nullptr;
    int32_t* d_paths = nullptr;
    int32_t* d_plen = nullptr;
    int d_path_cap = 0;
    int expand_blocks = 148, expand_wpb = 8, insert_blocks = 148;
    size_t expand_smem = 0;
    bool ran = false;
    const acs_goalset* goals = nullptr;  // the goal set of the next runs
};

// the engine's shape and node budgets
inline void mb_init(MbHost& h, int device, int n_search, int mrl, int W, int cyclical, const int64_t* max_nodes) {
    h.device = device;
    h.n_search = n_search;
    h.mrl = mrl;
    h.W = W;
    h.cyclical = cyclical ? 1 : 0;
    h.budgets.assign(max_nodes, max_nodes + n_search);
}

// the pinned ring, the stream, the events and the SM count
inline int mb_open(MbHost& h, const char* who) {
    if (cudaMallocHost((void**)&h.h_ring, kMbRing * sizeof(MbState)) != cudaSuccess)
        return fail(ACS_ERR_NOMEM, std::string(who) + ": cudaMallocHost");
    if (cudaStreamCreateWithFlags(&h.stream, cudaStreamNonBlocking) != cudaSuccess)
        return fail(ACS_ERR_CUDA, std::string(who) + ": cudaStreamCreate");
    cudaEventCreate(&h.ev0);
    cudaEventCreate(&h.ev1);
    for (auto& e : h.ring_ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, h.device) == cudaSuccess) h.sms = prop.multiProcessorCount;
    return ACS_OK;
}

// blocks of `kernel` that fill the GPU: its resident blocks per SM (at least one) on every SM
template <class K>
int mb_blocks(const MbHost& h, K kernel, int threads, size_t smem) {
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
    return h.sms * std::max(per_sm, 1);
}

// the arrays every engine needs; the caller frees what was allocated (mb_close) when this fails.  `b` is a
// pointer and `E` is named E because ACS_ALLOC's error text names the array as written: "cudaMalloc(b->d_roots)".
inline int mb_alloc(MbHost* b, MbEngine& E, int64_t nodes, uint64_t tcap, int64_t rec_cap, int64_t bitmap_words) {
    const int n_search = b->n_search, W = b->W;
    E.rec_cap = rec_cap;
    ACS_ALLOC(E.st, sizeof(MbState), (void)0);
    ACS_ALLOC(E.srch, (size_t)n_search * sizeof(MbSearch), (void)0);
    ACS_ALLOC(E.nodes, (size_t)nodes * 8 * node_words(W), (void)0);
    ACS_ALLOC(E.table, (size_t)tcap * 8, (void)0);
    ACS_ALLOC(E.log_keys, (size_t)rec_cap * 16 * W, (void)0);
    ACS_ALLOC(E.log_c, (size_t)rec_cap * 4, (void)0);
    ACS_ALLOC(E.log_s, (size_t)rec_cap * 4, (void)0);
    ACS_ALLOC(E.cursor, 8, (void)0);
    ACS_ALLOC(E.bitmap, (size_t)bitmap_words * 4, (void)0);
    ACS_ALLOC(E.ctrl, (size_t)n_search * kMbCtrl * 8, (void)0);
    ACS_ALLOC(E.seg_search, (size_t)n_search * 4, (void)0);
    ACS_ALLOC(E.seg_head, (size_t)n_search * 8, (void)0);
    ACS_ALLOC(E.seg_off, (size_t)(n_search + 1) * 8, (void)0);
    ACS_ALLOC(E.seg_limit, (size_t)n_search * 8, (void)0);
    ACS_ALLOC(E.seg_base, (size_t)n_search * 8, (void)0);
    ACS_ALLOC(E.seg_of, (size_t)n_search * 4, (void)0);
    ACS_ALLOC(b->d_roots, (size_t)n_search * 16 * W, (void)0);
    return ACS_OK;
}

// waits for the stream and frees every MbEngine array and the driver's own resources; the engine frees its extras
inline void mb_close(MbHost& h, MbEngine& E) {
    cudaSetDevice(h.device);
    if (h.stream) {
        cudaStreamSynchronize(h.stream);
        cudaStreamDestroy(h.stream);
    }
    if (h.ev0) cudaEventDestroy(h.ev0);
    if (h.ev1) cudaEventDestroy(h.ev1);
    for (auto e : h.ring_ev)
        if (e) cudaEventDestroy(e);
    void* ptrs[] = {E.st, E.srch, E.nodes, E.table, E.log_keys, E.log_c, E.log_s, E.rec_slot, E.cursor, E.bitmap, E.rt,
                    E.bsums, E.ctrl, E.seg_search, E.seg_head, E.seg_off, E.seg_limit, E.seg_base, E.seg_of,
                    E.goal_hit, E.goal_hit_g, E.log_g, h.d_roots, h.d_paths, h.d_plen};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (h.h_ring) cudaFreeHost(h.h_ring);
    cudaGetLastError();
}

// the host side of a run's roots
struct MbRoots {
    std::vector<MbSearch> init;  // [n_search] the searches' initial state
    std::vector<uint64_t> keys;  // [n_search][2W] the packed roots
    std::vector<uint8_t> g;      // [n_search] orbit search: the element that canonicalized each root
    int64_t n_valid = 0;         // roots that are searched
};

// Packs every row before any device work.  Search s gets a slab of budget + slack nodes; a row that is not a
// valid presentation gets status ACS_ROW_ASSERT and is not searched.  A letter outside {+-1,+-2} refuses the run.
template <int W>
int mb_pack_roots(const MbHost& h, const int8_t* h_pres, int64_t slack, bool symmetric, const char* who, MbRoots& R) {
    const int n = h.n_search, mrl = h.mrl;
    R.init.assign((size_t)n, MbSearch{});
    R.keys.assign((size_t)n * 2 * W, 0);
    R.g.assign((size_t)n, 0);
    R.n_valid = 0;
    int64_t slab = 0;
    for (int s = 0; s < n; ++s) {
        MbSearch& M = R.init[s];
        M.budget = h.budgets[s];
        M.cap = h.budgets[s] + slack;
        M.slab = slab;
        slab += M.cap;
        M.n_nodes = 1;
        M.level_end = 1;
        M.sol_gid = -1;
        Key<W> root;
        int lens[2];
        const RootCheck rc = pack_root<W>(h_pres + (size_t)s * 2 * mrl, mrl, root, lens);
        if (rc == RootCheck::bad_letter)
            return fail(ACS_ERR_UNSUPPORTED, std::string(who) + ": letters outside {+-1,+-2} are not supported by the packed search");
        if (rc != RootCheck::ok) {  // breadth_first.py:36-38 asserts is_array_valid_presentation
            M.status = ACS_ROW_ASSERT;
            M.done = 1;
            M.n_nodes = 0;
            continue;
        }
        M.min_len = lens[0] + lens[1];
        if (symmetric) {
            int g0 = 0;
            root = canonical<W>(root, g0);
            R.g[s] = (uint8_t)g0;
        }
        for (int i = 0; i < 2 * W; ++i) R.keys[(size_t)s * 2 * W + i] = root.k[i];
        ++R.n_valid;
    }
    return ACS_OK;
}

// The prologue of a run: clears the visited table and the goal hits, uploads the run state `st`, the searches
// and the roots (with d_root_g, each root's element of an orbit search), and launches the root kernels.
template <int W>
int mb_run_begin(MbHost& h, MbEngine& E, const MbState& st, const MbRoots& R, uint8_t* d_root_g) {
    const int n = h.n_search;
    cudaStream_t s = h.stream;
    ACS_CUDA(cudaSetDevice(h.device));
    ACS_CUDA(cudaMemsetAsync(E.table, 0, (st.tmask + 1) * sizeof(uint64_t), s));
    if (E.goal_hit) ACS_CUDA(cudaMemsetAsync(E.goal_hit, 0xFF, (size_t)n * sizeof(int64_t), s));
    if (E.goal_hit_g) ACS_CUDA(cudaMemsetAsync(E.goal_hit_g, 0xFF, (size_t)n * sizeof(int32_t), s));
    h.h_ring[0] = st;  // pinned staging for the async upload
    ACS_CUDA(cudaMemcpyAsync(E.st, &h.h_ring[0], sizeof(MbState), cudaMemcpyHostToDevice, s));
    ACS_CUDA(cudaMemcpyAsync(E.srch, R.init.data(), R.init.size() * sizeof(MbSearch), cudaMemcpyHostToDevice, s));
    ACS_CUDA(cudaMemcpyAsync(h.d_roots, R.keys.data(), R.keys.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    if (d_root_g) ACS_CUDA(cudaMemcpyAsync(d_root_g, R.g.data(), R.g.size(), cudaMemcpyHostToDevice, s));
    E.root_g = d_root_g;
    ACS_CUDA(cudaStreamSynchronize(s));  // the staging copies above read host memory that goes out of scope
    ACS_CUDA(cudaEventRecord(h.ev0, s));
    mb_init_kernel<W><<<(n + 127) / 128, 128, 0, s>>>(E, h.d_roots);
    if (h.goals) mb_goal_roots_kernel<W><<<(n + 127) / 128, 128, 0, s>>>(E);
    ACS_CUDA(cudaGetLastError());
    return ACS_OK;
}

// Before chunk `chunk` is enqueued: 1 when the run state copied kMbLag chunks earlier says the run is done,
// 0 when the chunk is to be enqueued, or an error code.
inline int mb_ring_done(MbHost& h, int64_t chunk) {
    if (chunk < kMbLag) return 0;
    ACS_CUDA(cudaEventSynchronize(h.ring_ev[(chunk - kMbLag) % kMbRing]));
    return h.h_ring[(chunk - kMbLag) % kMbRing].done ? 1 : 0;
}

// After chunk `chunk` is enqueued: a copy of the run state for mb_ring_done
inline int mb_ring_publish(MbHost& h, const MbEngine& E, int64_t chunk) {
    ACS_CUDA(cudaMemcpyAsync(&h.h_ring[chunk % kMbRing], E.st, sizeof(MbState), cudaMemcpyDeviceToHost, h.stream));
    ACS_CUDA(cudaEventRecord(h.ring_ev[chunk % kMbRing], h.stream));
    return ACS_OK;
}

// Paths of the solved searches of the last run into h_paths [n_search, path_cap, 2]; plen gets every search's
// path length (0 if not solved).  A path longer than path_cap is an error, never truncated.
template <int W>
int mb_paths(MbHost& h, const MbEngine& E, bool symmetric, const char* who, int32_t* h_paths, int path_cap,
             std::vector<int32_t>& plen) {
    const int n = h.n_search;
    cudaStream_t s = h.stream;
    ACS_CUDA(cudaSetDevice(h.device));
    const int cap = std::max(path_cap, 1);  // the kernel writes the first pair of every solved path
    if (!h.d_paths || cap > h.d_path_cap) {
        if (h.d_paths) cudaFree(h.d_paths);
        h.d_paths = nullptr;
        h.d_path_cap = 0;
        ACS_CUDA(cudaMalloc((void**)&h.d_paths, (size_t)n * cap * 2 * sizeof(int32_t)));
        h.d_path_cap = cap;
    }
    if (!h.d_plen) ACS_CUDA(cudaMalloc((void**)&h.d_plen, (size_t)n * sizeof(int32_t)));
    if (symmetric) mb_path_kernel<W, true><<<(n + 127) / 128, 128, 0, s>>>(E, h.d_paths, cap, h.d_plen);
    else mb_path_kernel<W, false><<<(n + 127) / 128, 128, 0, s>>>(E, h.d_paths, cap, h.d_plen);
    ACS_CUDA(cudaGetLastError());
    plen.resize((size_t)n);
    ACS_CUDA(cudaMemcpyAsync(plen.data(), h.d_plen, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < n; ++i)
        if (plen[i] > path_cap)
            return fail(ACS_ERR_INVALID, std::string(who) + ": a solution path is longer than path_cap (see path_len)");
    if (h_paths && path_cap > 0) {
        ACS_CUDA(cudaMemcpyAsync(h_paths, h.d_paths, (size_t)n * path_cap * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        ACS_CUDA(cudaStreamSynchronize(s));
    }
    return ACS_OK;
}

// the paths of the last run again, into a buffer of another size
inline int mb_paths_again(MbHost& h, const MbEngine& E, bool symmetric, const char* who, int32_t* h_paths, int path_cap) {
    if (!h.ran) return fail(ACS_ERR_INVALID, std::string(who) + ": no completed run");
    std::vector<int32_t> plen;
    return h.W == 1 ? mb_paths<1>(h, E, symmetric, who, h_paths, path_cap, plen)
                    : mb_paths<2>(h, E, symmetric, who, h_paths, path_cap, plen);
}

// The epilogue of a run, once its last chunk is enqueued: the final run state and searches.  ierr gets the run's
// internal error bits (MB_IERR_*); when they are set nothing else is done and the caller reports them.  Otherwise
// the run counts as completed, and its paths and results are fetched.
template <int W>
int mb_run_end(MbHost& h, const MbEngine& E, bool symmetric, const char* who, int32_t* h_paths, int path_cap,
               acs_search_result* results, int& ierr) {
    const int n = h.n_search;
    cudaStream_t s = h.stream;
    ACS_CUDA(cudaEventRecord(h.ev1, s));
    MbState fin{};
    h.h_final.resize((size_t)n);
    ACS_CUDA(cudaMemcpyAsync(&fin, E.st, sizeof(MbState), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaMemcpyAsync(h.h_final.data(), E.srch, (size_t)n * sizeof(MbSearch), cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaStreamSynchronize(s));
    ierr = fin.ierr;
    if (ierr) return ACS_OK;
    h.ran = true;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h.ev0, h.ev1);
    std::vector<int32_t> plen((size_t)n);
    const int rc = mb_paths<W>(h, E, symmetric, who, h_paths, path_cap, plen);
    for (int i = 0; i < n; ++i) {
        const MbSearch& f = h.h_final[i];
        acs_search_result* r = results + i;
        std::memset(r, 0, sizeof(*r));
        r->solved = f.solved;
        r->status = f.status;
        r->budget_hit = f.budget_hit;
        r->path_len = plen[i];
        r->seconds_device = ms * 1e-3;
        if (f.status == ACS_ROW_ASSERT && f.n_nodes == 0) continue;  // invalid root: the reference asserts before searching
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

// the visited nodes of one search of the last run, in order, as int8 rows
inline int mb_visited(const MbHost& h, const MbEngine& E, const char* who, int search, int8_t* h_out, int64_t cap_rows,
                      int64_t* n_out) {
    if (!h.ran) return fail(ACS_ERR_INVALID, std::string(who) + ": no completed run");
    ACS_CUDA(cudaSetDevice(h.device));
    const MbSearch& f = h.h_final[search];
    const int64_t n = std::min<int64_t>(f.n_nodes, std::max<int64_t>(cap_rows, 0));
    if (n_out) *n_out = n;
    const uint64_t* slab = E.nodes + (size_t)f.slab * node_words(h.W);
    return records_to_host(h.W, slab, node_words(h.W), n, h.mrl, h_out, nullptr, h.stream);
}

// binds the goal set g (checked by goalset_check), or none, to the next runs
inline int mb_set_goals(MbHost& h, MbEngine& E, const acs_goalset* g) {
    if (g) {
        if (!E.goal_hit) {
            ACS_CUDA(cudaSetDevice(h.device));
            ACS_CUDA(cudaMalloc((void**)&E.goal_hit, (size_t)h.n_search * sizeof(int64_t)));
            ACS_CUDA(cudaMemset(E.goal_hit, 0xFF, (size_t)h.n_search * sizeof(int64_t)));
            ACS_CUDA(cudaMalloc((void**)&E.goal_hit_g, (size_t)h.n_search * sizeof(int32_t)));
            ACS_CUDA(cudaMemset(E.goal_hit_g, 0xFF, (size_t)h.n_search * sizeof(int32_t)));
        }
        E.goals = g->view();
    } else {
        E.goals = GoalView{nullptr, nullptr, 0, 0};
    }
    h.goals = g;
    return ACS_OK;
}

// per search of the last run, the goal entry it stopped at (E.goal_hit) or the goal element (E.goal_hit_g);
// -1 for every search when no goal set was ever bound
template <class T>
int mb_goal_hits(const MbHost& h, const T* d_hits, T* h_out, const char* who) {
    if (!h.ran) return fail(ACS_ERR_INVALID, std::string(who) + ": no completed run");
    if (!d_hits) {
        std::fill(h_out, h_out + h.n_search, (T)-1);
        return ACS_OK;
    }
    ACS_CUDA(cudaSetDevice(h.device));
    ACS_CUDA(cudaMemcpyAsync(h_out, d_hits, (size_t)h.n_search * sizeof(T), cudaMemcpyDeviceToHost, h.stream));
    ACS_CUDA(cudaStreamSynchronize(h.stream));
    return ACS_OK;
}

}  // namespace acs
