// goalset.cu -- goal sets: device-resident sets of states keyed by the state alone, for the goal test
// of the batched breadth-first search (mbfs.cu).  Built from int8 rows here, or from a finished
// batched run (acs_goalset_from_bfs_batch in mbfs.cu).  Layout and lookup: goalset.cuh.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "ac_keys.cuh"
#include "acs_internal.h"
#include "bfs_common.cuh"
#include "goalset.cuh"

namespace acs {

// every entry claims the first free slot of its probe sequence, or displaces a larger entry index of the
// same state (slots only ever pass between entries of one state, so a state never holds two slots)
template <int W>
__global__ void __launch_bounds__(256) gs_insert_kernel(uint64_t* table, uint64_t tmask, const uint64_t* nodes, uint64_t n,
                                                        int* overflow) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const Key<W> key = node_key<W>(nodes, i);
        const uint64_t h = pb_hash<W>(key), fp = h >> 41;
        const uint64_t mine = (fp << 40) | (i + 1);
        uint64_t base = (h & tmask) & ~3ull;
        bool finished = false;
        for (uint64_t probes = 0; !finished; probes += 4, base = (base + 4) & tmask) {
            if (probes > tmask) {  // cannot happen: the table is at most half full
                atomicOr(overflow, 1);
                break;
            }
            uint64_t vv[4];
            load_bucket(table + base, vv);
            for (int j = 0; j < 4 && !finished; ++j) {
                unsigned long long* sp = (unsigned long long*)&table[base + j];
                uint64_t cur = vv[j];
                if (cur == 0) {
                    cur = atomicCAS(sp, 0ull, (unsigned long long)mine);
                    if (cur == 0) {
                        finished = true;
                        break;
                    }
                }
                if ((cur >> 40) != fp || !key_eq<W>(node_key<W>(nodes, (cur & kGsIdx) - 1), key)) continue;
                while ((cur & kGsIdx) - 1 > i) {  // the same state under a larger index: take its slot
                    const uint64_t old = atomicCAS(sp, (unsigned long long)cur, (unsigned long long)mine);
                    if (old == cur) break;
                    cur = old;  // another entry of this state took it meanwhile: compare again
                }
                finished = true;
            }
        }
    }
}

__global__ void __launch_bounds__(256) gs_count_kernel(const uint64_t* table, uint64_t n, unsigned long long* count) {
    __shared__ unsigned long long sum;
    if (threadIdx.x == 0) sum = 0;
    __syncthreads();
    uint64_t c = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        c += table[i] != 0;
    if (c) atomicAdd(&sum, (unsigned long long)c);
    __syncthreads();
    if (threadIdx.x == 0 && sum) atomicAdd(count, sum);
}

// path of one entry from its root: (-1, L_root), (action, L), ...; out[0] = length, out[1] = root, out[2] = the
// frame H of the path's end: end state = H.(stored state).  In a symmetric set entry j stores c_j = g_j.(the state
// its move made from c_j-1), the actual states are a_j = h_j.c_j with h_0 = g_0^-1 and h_j = h_j-1.g_j^-1, so
// h_j = (g_j ... g_0)^-1, and the actual move into node j is pi_{h_j-1}(m_j) with h_j-1 = P^-1.(g_k ... g_j),
// P = g_k ... g_0: one pass for P, one pass back from the entry accumulating g_k ... g_j.
template <int W>
__global__ void gs_path_kernel(const uint64_t* nodes, int64_t entry, int32_t* path, int path_cap, int32_t* out) {
    int depth = 0;
    int64_t root = 0;
    int P = 0;
    for (int64_t e = entry; e >= 0; ++depth) {
        Key<W> k;
        int64_t pl;
        node_load<W>(nodes, (uint64_t)e, k, pl, root);
        P = sym_mul(P, (int)((uint64_t)root >> 32) & 15);
        e = pl < 0 ? -1 : (pl >> 4);
    }
    out[0] = depth;
    out[1] = (int32_t)(root & 0xFFFFFFFFll);
    out[2] = sym_inv(P);
    int pos = depth - 1, Q = 0;
    for (int64_t e = entry; e >= 0; --pos) {
        Key<W> k;
        int64_t pl, r;
        node_load<W>(nodes, (uint64_t)e, k, pl, r);
        Q = sym_mul(Q, (int)((uint64_t)r >> 32) & 15);
        if (pos < path_cap) {
            path[2 * pos] = pl < 0 ? -1 : sym_pi(sym_mul(sym_inv(P), Q), (int)(pl & 15));
            path[2 * pos + 1] = key_total_len<W>(k);
        }
        e = pl < 0 ? -1 : (pl >> 4);
    }
}

int goalset_check(const acs_goalset* g, int mrl, int cyclical, int device, bool orbit, const char* who) {
    const std::string w = std::string(who) + "_set_goals: ";
    if (g->mrl != mrl) return fail(ACS_ERR_INVALID, w + "the goal set's max_relator_length differs from the engine's");
    if (g->cyclical != cyclical) return fail(ACS_ERR_INVALID, w + "the goal set's cyclical flag differs from the engine's");
    if (g->device != device) return fail(ACS_ERR_INVALID, w + "the goal set lives on another device");
    if (orbit && !g->symmetric)  // an orbit search knows only the orbit of a child
        return fail(ACS_ERR_INVALID, w + "an orbit search needs a symmetric goal set");
    if (g->n_entries >= (int64_t)0xFFFFFFFF)  // a hit packs the entry into 32 bits beside its candidate id
        return fail(ACS_ERR_UNSUPPORTED, w + "goal sets of 2^32 - 1 entries or more are not supported");
    return ACS_OK;
}

int goalset_index(acs_goalset* g, cudaStream_t s) {
    uint64_t t = 1024;
    while (t < 2 * (uint64_t)g->n_entries) t <<= 1;
    g->tcap = t;
    if (cudaMalloc((void**)&g->table, t * 8) != cudaSuccess) {
        cudaGetLastError();
        return fail(ACS_ERR_NOMEM, "goalset: cudaMalloc of the index failed");
    }
    int* d_flag = nullptr;
    unsigned long long* d_count = nullptr;
    cudaError_t e = cudaMalloc((void**)&d_flag, 16);
    if (e == cudaSuccess) {
        d_count = reinterpret_cast<unsigned long long*>(d_flag + 2);
        e = cudaMemsetAsync(d_flag, 0, 16, s);
    }
    if (e == cudaSuccess) e = cudaMemsetAsync(g->table, 0, t * 8, s);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g->device);
    if (e == cudaSuccess && g->n_entries > 0) {
        const unsigned grid = (unsigned)std::min<int64_t>((g->n_entries + 255) / 256, (int64_t)sms * 8);
        if (g->W == 1) gs_insert_kernel<1><<<grid, 256, 0, s>>>(g->table, t - 1, g->nodes, (uint64_t)g->n_entries, d_flag);
        else gs_insert_kernel<2><<<grid, 256, 0, s>>>(g->table, t - 1, g->nodes, (uint64_t)g->n_entries, d_flag);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) {
        const unsigned grid = (unsigned)std::min<uint64_t>((t + 255) / 256, (uint64_t)sms * 8);
        gs_count_kernel<<<grid, 256, 0, s>>>(g->table, t, d_count);
        e = cudaGetLastError();
    }
    int flag = 0;
    unsigned long long count = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&count, d_count, 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (d_flag) cudaFree(d_flag);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ACS_ERR_CUDA, std::string("goalset: building the index: ") + cudaGetErrorString(e));
    }
    if (flag) return fail(ACS_ERR_CUDA, "goalset: internal error: index full");
    g->n_states = (int64_t)count;
    return ACS_OK;
}

void goalset_free(acs_goalset* g) {
    if (!g) return;
    cudaSetDevice(g->device);
    if (g->nodes) cudaFree(g->nodes);
    if (g->table) cudaFree(g->table);
    cudaGetLastError();
    delete g;
}

}  // namespace acs

using namespace acs;

namespace {

// "" if row k is a state a search can generate: letters in {+-1,+-2}, each relator non-empty,
// right-padded and freely reduced, and cyclically reduced when `cyclical`
std::string gs_row_problem(const int8_t* p, int mrl, int cyclical) {
    for (int h = 0; h < 2; ++h) {
        const int8_t* r = p + h * mrl;
        int n = 0;
        while (n < mrl && r[n] != 0) ++n;
        if (n == 0) return "an empty relator";
        for (int t = n; t < mrl; ++t)
            if (r[t] != 0) return "zeros inside a relator (padding must be on the right)";
        for (int t = 0; t < n; ++t)
            if (r[t] < -2 || r[t] > 2) return "a letter outside {+-1, +-2}";
        for (int t = 0; t + 1 < n; ++t)
            if (r[t] == -r[t + 1]) return "a relator that is not freely reduced";
        if (cyclical && n > 1 && r[0] == -r[n - 1]) return "a relator that is not cyclically reduced";
    }
    return "";
}

template <int W>
void gs_pack(const int8_t* h_rows, int64_t n, int mrl, int symmetric, std::vector<uint64_t>& nodes) {
    nodes.assign((size_t)std::max<int64_t>(n, 1) * node_words(W), 0);
    for (int64_t i = 0; i < n; ++i) {
        Key<W> key;
        int lens[2];
        pack_root<W>(h_rows + (size_t)i * 2 * mrl, mrl, key, lens);  // gs_row_problem has accepted the row
        int g = 0;
        if (symmetric) key = canonical<W>(key, g);
        node_pack<W>(key, -1, i | (int64_t)g << 32, nodes.data() + (size_t)i * node_words(W));
    }
}

}  // namespace

extern "C" {

namespace {
int gs_from_rows(int device, int mrl, int cyclical, int symmetric, const int8_t* h_rows, int64_t n, acs_goalset** out) {
    if (!out) return ACS_ERR_INVALID;
    *out = nullptr;
    if (const int rc = check_key_mrl(mrl, "goalset")) return rc;
    if (n < 0 || (n > 0 && !h_rows)) return fail(ACS_ERR_INVALID, "goalset: bad row count or rows");
    if (n >= (int64_t)kGsIdx) return fail(ACS_ERR_UNSUPPORTED, "goalset: too many rows");
    for (int64_t i = 0; i < n; ++i) {
        const std::string why = gs_row_problem(h_rows + (size_t)i * 2 * mrl, mrl, cyclical);
        if (!why.empty())
            return fail(ACS_ERR_INVALID, "goalset: row " + std::to_string(i) + " has " + why +
                                                ", so no search can generate it");
    }
    if (const int rc = open_device(device, "goalset")) return rc;
    acs_goalset* g = new acs_goalset();
    g->device = device;
    g->mrl = mrl;
    g->W = key_words(mrl);
    g->cyclical = cyclical ? 1 : 0;
    g->symmetric = symmetric ? 1 : 0;
    g->n_entries = n;
    std::vector<uint64_t> h;
    if (g->W == 1) gs_pack<1>(h_rows, n, mrl, g->symmetric, h);
    else gs_pack<2>(h_rows, n, mrl, g->symmetric, h);
    if (cudaMalloc((void**)&g->nodes, h.size() * 8) != cudaSuccess) {
        cudaGetLastError();
        goalset_free(g);
        return fail(ACS_ERR_NOMEM, "goalset: cudaMalloc of the entries failed");
    }
    if (cudaMemcpy(g->nodes, h.data(), h.size() * 8, cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaGetLastError();
        goalset_free(g);
        return fail(ACS_ERR_CUDA, "goalset: uploading the entries failed");
    }
    const int rc = goalset_index(g, 0);
    if (rc != ACS_OK) {
        goalset_free(g);
        return rc;
    }
    *out = g;
    return ACS_OK;
}
}  // namespace

int acs_goalset_from_rows(int device, int mrl, int cyclical, const int8_t* h_rows, int64_t n, acs_goalset** out) {
    return gs_from_rows(device, mrl, cyclical, 0, h_rows, n, out);
}

int acs_goalset_from_rows_symmetric(int device, int mrl, int cyclical, const int8_t* h_rows, int64_t n,
                                    acs_goalset** out) {
    return gs_from_rows(device, mrl, cyclical, 1, h_rows, n, out);
}

int acs_goalset_is_symmetric(const acs_goalset* g, int* symmetric) {
    if (!g || !symmetric) return ACS_ERR_INVALID;
    *symmetric = g->symmetric;
    return ACS_OK;
}

int acs_goalset_size(const acs_goalset* g, int64_t* n_entries, int64_t* n_states, int64_t* bytes) {
    if (!g) return ACS_ERR_INVALID;
    if (n_entries) *n_entries = g->n_entries;
    if (n_states) *n_states = g->n_states;
    if (bytes) *bytes = std::max<int64_t>(g->n_entries, 1) * 8 * node_words(g->W) + (int64_t)g->tcap * 8;
    return ACS_OK;
}

int acs_goalset_path(const acs_goalset* g, int64_t entry, int* root, int32_t* h_path, int path_cap, int* path_len) {
    return acs_goalset_path_frame(g, entry, root, h_path, path_cap, path_len, nullptr);
}

int acs_goalset_path_frame(const acs_goalset* g, int64_t entry, int* root, int32_t* h_path, int path_cap, int* path_len,
                           int* frame) {
    if (!g || path_cap < 0 || (!h_path && path_cap > 0)) return ACS_ERR_INVALID;
    if (entry < 0 || entry >= g->n_entries) return fail(ACS_ERR_INVALID, "goalset_path: entry out of range");
    if (cudaSetDevice(g->device) != cudaSuccess) {
        cudaGetLastError();
        return fail(ACS_ERR_CUDA, "goalset_path: cudaSetDevice failed");
    }
    const int cap = std::max(path_cap, 1);
    int32_t* d = nullptr;
    cudaError_t e = cudaMalloc((void**)&d, ((size_t)cap * 2 + 4) * sizeof(int32_t));
    int32_t res[4] = {0, 0, 0, 0};
    if (e == cudaSuccess) {
        if (g->W == 1) gs_path_kernel<1><<<1, 1>>>(g->nodes, entry, d + 4, cap, d);
        else gs_path_kernel<2><<<1, 1>>>(g->nodes, entry, d + 4, cap, d);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(res, d, sizeof(res), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && res[0] <= path_cap && path_cap > 0)
        e = cudaMemcpy(h_path, d + 4, (size_t)res[0] * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost);
    if (d) cudaFree(d);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ACS_ERR_CUDA, std::string("goalset_path: ") + cudaGetErrorString(e));
    }
    if (path_len) *path_len = res[0];
    if (root) *root = res[1];
    if (frame) *frame = res[2];
    if (res[0] > path_cap) return fail(ACS_ERR_INVALID, "goalset_path: the path is longer than path_cap (see path_len)");
    return ACS_OK;
}

void acs_goalset_destroy(acs_goalset* g) { goalset_free(g); }

}  // extern "C"
