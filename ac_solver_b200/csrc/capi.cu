// capi.cu -- the C ABI of libacsolver_b200.so (see include/acsolver_b200.h).
// Host-side runtime only: argument checks, the context (streams + grow-only scratch) and
// the chunked H2D -> kernel -> D2H pipelines behind the *_host entry points.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "ac_keys.cuh"
#include "acs_internal.h"

using acs::cuda_fail;
using acs::fail;

namespace {

thread_local std::string g_err;

constexpr int kStreams = 3;
constexpr int64_t kChunkRows = 1 << 17;  // rows per pipeline chunk of the *_host calls
constexpr int64_t kEnvChunkRows = 1 << 18;  // acs_env_step_host: 4 chunks per 1 Mi rows (131072 .. 1048576 measure the same at N = 1)
constexpr size_t kSmallCall = 64 * 1024;   // single-call API: everything goes through one pinned staging buffer

struct Scratch {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return ACS_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(scratch)");
        cap = bytes;
        return ACS_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace

namespace acs {
void set_last_error(const char* msg) { g_err = msg ? msg : ""; }

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

int cuda_fail(cudaError_t e, const std::string& what) {
    cudaGetLastError();
    return fail(e == cudaErrorMemoryAllocation ? ACS_ERR_NOMEM : ACS_ERR_CUDA, what + ": " + cudaGetErrorString(e));
}

int open_device(int device, const char* who) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(ACS_ERR_NO_DEVICE, "no CUDA device visible; there is no CPU fallback");
    }
    if (device < 0 || device >= n) return fail(ACS_ERR_INVALID, std::string(who) + ": device index out of range");
    ACS_CUDA(cudaSetDevice(device));
    return ACS_OK;
}

int check_key_mrl(int mrl, const char* who) {
    if (mrl >= 1 && mrl <= kMaxKeyMrl) return ACS_OK;
    return fail(ACS_ERR_UNSUPPORTED, std::string(who) + " needs 1 <= max_relator_length <= " + std::to_string(kMaxKeyMrl));
}

int records_to_host(int W, const uint64_t* d_recs, int stride, int64_t n, int mrl, int8_t* h_rows, int64_t* h_gid,
                    cudaStream_t s) {
    if (n <= 0) return ACS_OK;
    int8_t* d = nullptr;
    int64_t* dg = nullptr;
    ACS_ALLOC(d, n * 2 * mrl, (void)0);
    if (h_gid) ACS_ALLOC(dg, n * 8, cudaFree(d));
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (W == 1) records_unpack_kernel<1><<<grid, 256, 0, s>>>(d_recs, stride, dg, d, (uint64_t)n, mrl);
    else records_unpack_kernel<2><<<grid, 256, 0, s>>>(d_recs, stride, dg, d, (uint64_t)n, mrl);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_rows, d, (size_t)n * 2 * mrl, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && h_gid) e = cudaMemcpyAsync(h_gid, dg, (size_t)n * 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(dg);
    cudaFree(d);
    return e == cudaSuccess ? ACS_OK : cuda_fail(e, "visited rows");
}
}  // namespace acs

struct acs_ctx {
    int device = 0;
    cudaStream_t streams[kStreams] = {};
    Scratch scratch[kStreams];
    unsigned long long* d_err = nullptr;  // {count, min row}
    unsigned long long* h_err = nullptr;  // pinned: [0..1] reset values, [2..3] read-back
    uint8_t* h_stage = nullptr;            // pinned staging of the small-call path of acs_generic_host (kSmallCall bytes)
    Scratch out;                           // acs_env_step_host: actions | reward | done | truncated of the whole call
    cudaEvent_t ev_start = nullptr, ev_done[kStreams] = {};
    std::mutex mu;  // the *_host calls share streams and scratch: one caller at a time per context
};

extern "C" {

int acs_version(void) { return 100; }
const char* acs_last_error(void) { return g_err.c_str(); }

int acs_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int acs_ctx_create(int device, acs_ctx** out) {
    if (!out) return fail(ACS_ERR_INVALID, "out is null");
    *out = nullptr;
    if (const int rc = acs::open_device(device, "acs_ctx_create")) return rc;
    acs_ctx* c = new acs_ctx();
    c->device = device;
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < kStreams && e == cudaSuccess; ++k)
        e = cudaStreamCreateWithFlags(&c->streams[k], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_err, 2 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMallocHost(&c->h_err, 4 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMallocHost(&c->h_stage, kSmallCall);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_start, cudaEventDisableTiming);
    for (int k = 0; k < kStreams && e == cudaSuccess; ++k) e = cudaEventCreateWithFlags(&c->ev_done[k], cudaEventDisableTiming);
    if (e != cudaSuccess) {  // release whatever was created
        acs_ctx_destroy(c);
        return cuda_fail(e, "acs_ctx_create");
    }
    *out = c;
    return ACS_OK;
}

void acs_ctx_destroy(acs_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (int k = 0; k < kStreams; ++k) {
        if (c->streams[k]) {
            cudaStreamSynchronize(c->streams[k]);
            cudaStreamDestroy(c->streams[k]);
        }
        c->scratch[k].release();
    }
    c->out.release();
    if (c->ev_start) cudaEventDestroy(c->ev_start);
    for (int k = 0; k < kStreams; ++k)
        if (c->ev_done[k]) cudaEventDestroy(c->ev_done[k]);
    if (c->d_err) cudaFree(c->d_err);
    if (c->h_err) cudaFreeHost(c->h_err);
    if (c->h_stage) cudaFreeHost(c->h_stage);
    delete c;
}

// ---------------------------------------------------------------- device-pointer API
int acs_moves_batch(const int8_t* d_in, const uint8_t* d_action, int8_t* d_out, uint8_t* d_lens,
                    uint8_t* d_status, uint64_t* d_err, int64_t n, int mrl, int flags, void* stream) {
    if (n < 0 || (n > 0 && (!d_in || !d_action || !d_out))) return fail(ACS_ERR_INVALID, "null buffer");
    if (mrl < 1 || mrl > 64) return fail(ACS_ERR_UNSUPPORTED, "packed kernels need 1 <= mrl <= 64");
    acs::StepParams P{};
    P.in = d_in;
    P.out = d_out;
    P.action = d_action;
    P.lens = d_lens;
    P.status = d_status;
    P.err = reinterpret_cast<unsigned long long*>(d_err);
    P.n = n;
    P.mrl = mrl;
    P.cyclical = (flags & ACS_FLAG_CYCLICAL) ? 1 : 0;
    P.trusted = (flags & ACS_FLAG_NORMALIZED) ? 1 : 0;
    P.lens_valid = ((flags & ACS_FLAG_LENS_VALID) && P.trusted && d_lens) ? 1 : 0;
    P.bulk_ok = aligned16(d_in) && aligned16(d_out);
    ACS_CUDA(acs::launch_step(P, static_cast<cudaStream_t>(stream)));
    return ACS_OK;
}

int acs_env_step_batch(int8_t* d_state, const uint8_t* d_action, int32_t* d_reward, uint8_t* d_done,
                       uint8_t* d_truncated, int32_t* d_step_count, uint8_t* d_lens, uint8_t* d_status,
                       uint64_t* d_err, int64_t n, int mrl, int horizon, int flags, void* stream) {
    if (n < 0 || (n > 0 && (!d_state || !d_action || !d_reward || !d_done || !d_truncated || !d_step_count)))
        return fail(ACS_ERR_INVALID, "null buffer");
    if (mrl < 1 || mrl > 64) return fail(ACS_ERR_UNSUPPORTED, "packed kernels need 1 <= mrl <= 64");
    acs::StepParams P{};
    P.in = d_state;
    P.out = d_state;
    P.action = d_action;
    P.lens = d_lens;
    P.status = d_status;
    P.err = reinterpret_cast<unsigned long long*>(d_err);
    P.reward = d_reward;
    P.done = d_done;
    P.truncated = d_truncated;
    P.step_count = d_step_count;
    P.n = n;
    P.mrl = mrl;
    P.cyclical = 1;  // ac_env.py:97-99 uses ACMove's default cyclical=True
    P.trusted = (flags & ACS_FLAG_NORMALIZED) ? 1 : 0;
    P.lens_valid = ((flags & ACS_FLAG_LENS_VALID) && P.trusted && d_lens) ? 1 : 0;
    P.horizon = horizon;
    P.max_reward = horizon * mrl * 2;  // ac_env.py:80
    P.bulk_ok = aligned16(d_state);
    ACS_CUDA(acs::launch_step(P, static_cast<cudaStream_t>(stream)));
    return ACS_OK;
}

int acs_vecenv_step(int8_t* d_state, const int8_t* d_initial_state, const uint8_t* d_action, int32_t* d_reward,
                    uint8_t* d_done, uint8_t* d_truncated, int32_t* d_step_count, uint8_t* d_lens,
                    const uint8_t* d_initial_lens, uint8_t* d_action_log, int log_stride, int8_t* d_final_obs,
                    int32_t* d_final_steps, uint64_t* d_err, int64_t n, int mrl, int horizon, int flags, void* stream) {
    if (n < 0 || (n > 0 && (!d_state || !d_initial_state || !d_action || !d_reward || !d_done || !d_truncated ||
                            !d_step_count)))
        return fail(ACS_ERR_INVALID, "null buffer");
    if (mrl < 1 || mrl > 64) return fail(ACS_ERR_UNSUPPORTED, "packed kernels need 1 <= mrl <= 64");
    if (d_action_log && log_stride < 1) return fail(ACS_ERR_INVALID, "the action log needs log_stride >= 1");
    if (d_lens && !d_initial_lens) return fail(ACS_ERR_INVALID, "d_lens needs d_initial_lens for the auto-reset");
    acs::StepParams P{};
    P.in = d_state;
    P.out = d_state;
    P.action = d_action;
    P.lens = d_lens;
    P.err = reinterpret_cast<unsigned long long*>(d_err);
    P.reward = d_reward;
    P.done = d_done;
    P.truncated = d_truncated;
    P.step_count = d_step_count;
    P.n = n;
    P.mrl = mrl;
    P.cyclical = 1;
    P.trusted = (flags & ACS_FLAG_NORMALIZED) ? 1 : 0;
    P.lens_valid = ((flags & ACS_FLAG_LENS_VALID) && P.trusted && d_lens) ? 1 : 0;
    P.horizon = horizon;
    P.max_reward = horizon * mrl * 2;
    P.bulk_ok = aligned16(d_state);
    P.action_log = d_action_log;
    P.log_stride = log_stride;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    ACS_CUDA(acs::launch_step(P, s));
    ACS_CUDA(acs::launch_autoreset(d_state, d_initial_state, d_final_obs, d_done, d_truncated, d_step_count,
                                   d_final_steps, d_lens, d_initial_lens, n, mrl, s));
    return ACS_OK;
}

int acs_reward_transform(const int32_t* d_reward, const uint8_t* d_done, double* d_stats, float* d_out, int64_t n,
                         double gamma, double eps, int normalize, int clip, double lo, double hi, void* stream) {
    if (n < 0 || (n > 0 && (!d_reward || !d_out || (normalize && (!d_stats || !d_done)))))
        return fail(ACS_ERR_INVALID, "null buffer");
    ACS_CUDA(acs::launch_reward_transform(d_reward, d_done, d_stats, d_out, n, gamma, eps, normalize, clip, lo, hi,
                                          static_cast<cudaStream_t>(stream)));
    return ACS_OK;
}

int acs_vecenv_curriculum_step(const acs_curriculum_args* a, void* stream) {
    if (!a || a->n < 0) return fail(ACS_ERR_INVALID, "null argument block");
    if (a->n > 0 && (!a->state || !a->pool || !a->pool_lens || !a->lens || !a->action || !a->reward || !a->done ||
                     !a->truncated || !a->step_count || !a->cur_state || !a->solved || !a->solved_list || !a->best ||
                     !a->best_actions || !a->action_log || !a->counters))
        return fail(ACS_ERR_INVALID, "null buffer");
    if (a->mrl < 1 || a->mrl > 64) return fail(ACS_ERR_UNSUPPORTED, "packed kernels need 1 <= mrl <= 64");
    if (a->n_states < 1 || a->log_stride < 1) return fail(ACS_ERR_INVALID, "bad pool size / log stride");
    acs::StepParams P{};
    P.in = a->state;
    P.out = a->state;
    P.action = a->action;
    P.lens = a->lens;
    P.err = reinterpret_cast<unsigned long long*>(a->err);
    P.reward = a->reward;
    P.done = a->done;
    P.truncated = a->truncated;
    P.step_count = a->step_count;
    P.n = a->n;
    P.mrl = a->mrl;
    P.cyclical = 1;
    P.trusted = (a->flags & ACS_FLAG_NORMALIZED) ? 1 : 0;
    P.lens_valid = ((a->flags & ACS_FLAG_LENS_VALID) && P.trusted) ? 1 : 0;
    P.horizon = a->horizon;
    P.max_reward = a->horizon * a->mrl * 2;
    P.bulk_ok = aligned16(a->state);
    P.action_log = a->action_log;
    P.log_stride = a->log_stride;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    ACS_CUDA(acs::launch_step(P, s));
    acs::CurriculumParams C{};
    C.state = a->state;
    C.pool = a->pool;
    C.pool_lens = a->pool_lens;
    C.lens = a->lens;
    C.done = a->done;
    C.trunc = a->truncated;
    C.step_count = a->step_count;
    C.cur_state = a->cur_state;
    C.solved = a->solved;
    C.solved_list = a->solved_list;
    C.best = reinterpret_cast<unsigned long long*>(a->best);
    C.best_actions = a->best_actions;
    C.action_log = a->action_log;
    C.final_obs = a->final_obs;
    C.final_steps = a->final_steps;
    C.counters = reinterpret_cast<long long*>(a->counters);
    C.n = a->n;
    C.n_states = a->n_states;
    C.mrl = a->mrl;
    C.log_stride = a->log_stride;
    C.repeat_solved_prob = a->repeat_solved_prob;
    C.seed = a->seed;
    ACS_CUDA(acs::launch_curriculum(C, s));
    return ACS_OK;
}

int acs_validate_batch(const int8_t* d_in, uint8_t* d_flags, int64_t n, int mrl, void* stream) {
    if (n < 0 || (n > 0 && (!d_in || !d_flags)) || mrl < 1) return fail(ACS_ERR_INVALID, "bad argument");
    ACS_CUDA(acs::launch_validate(d_in, d_flags, n, mrl, static_cast<cudaStream_t>(stream)));
    return ACS_OK;
}

int acs_generic_batch(int op, const int8_t* d_in, const uint8_t* d_action, int8_t* d_out, int32_t* d_aux,
                      uint8_t* d_status, int64_t n, int width, int i, int j, int sign, int cyclical,
                      void* stream) {
    if (n < 0 || (n > 0 && (!d_in || !d_out || !d_aux))) return fail(ACS_ERR_INVALID, "null buffer");
    if (op < 0 || op > 4) return fail(ACS_ERR_INVALID, "unknown op");
    if (op == ACS_OP_ACMOVE && n > 0 && !d_action) return fail(ACS_ERR_INVALID, "ACMOVE needs actions");
    if (width < 1 || width > 254 || (op != ACS_OP_SIMPLIFY_RELATOR && (width & 1)))
        return fail(ACS_ERR_UNSUPPORTED, "generic kernels need 1 <= width <= 254 (even for presentations)");
    acs::GenericParams G{};
    G.op = op;
    G.in = d_in;
    G.action = d_action;
    G.out = d_out;
    G.aux = d_aux;
    G.status = d_status;
    G.n = n;
    G.width = width;
    G.i = i;
    G.j = j;
    G.sign = sign;
    G.cyclical = cyclical ? 1 : 0;
    ACS_CUDA(acs::launch_generic(G, static_cast<cudaStream_t>(stream)));
    return ACS_OK;
}

// ---------------------------------------------------------------- host-pointer API
int acs_moves_batch_host(acs_ctx* c, const int8_t* h_in, const uint8_t* h_action, int8_t* h_out, uint8_t* h_lens,
                         uint8_t* h_status, int64_t n, int mrl, int flags) {
    if (!c) return fail(ACS_ERR_INVALID, "ctx is null");
    std::lock_guard<std::mutex> lock(c->mu);
    if (n < 0 || (n > 0 && (!h_in || !h_action || !h_out))) return fail(ACS_ERR_INVALID, "null buffer");
    if (mrl < 1 || mrl > 64) return fail(ACS_ERR_UNSUPPORTED, "packed kernels need 1 <= mrl <= 64");
    ACS_CUDA(cudaSetDevice(c->device));
    const size_t rowb = 2 * (size_t)mrl;
    const int64_t chunk = n < kChunkRows ? (n > 0 ? n : 1) : kChunkRows;
    // per-stream scratch: state (in place) | action | lens | status, each 256-byte aligned
    const size_t o_act = align_up((size_t)chunk * rowb, 256);
    const size_t o_len = o_act + align_up((size_t)chunk, 256);
    const size_t o_st = o_len + align_up((size_t)chunk * 2, 256);
    const size_t total = o_st + align_up((size_t)chunk, 256);
    int64_t ci = 0;
    for (int64_t r0 = 0; r0 < n; r0 += chunk, ++ci) {
        const int k = (int)(ci % kStreams);
        const int64_t m = (n - r0) < chunk ? (n - r0) : chunk;
        int rc = c->scratch[k].reserve(total);
        if (rc != ACS_OK) return rc;
        uint8_t* base = static_cast<uint8_t*>(c->scratch[k].p);
        cudaStream_t s = c->streams[k];
        ACS_CUDA(cudaMemcpyAsync(base, h_in + r0 * rowb, (size_t)m * rowb, cudaMemcpyHostToDevice, s));
        ACS_CUDA(cudaMemcpyAsync(base + o_act, h_action + r0, (size_t)m, cudaMemcpyHostToDevice, s));
        rc = acs_moves_batch(reinterpret_cast<int8_t*>(base), base + o_act, reinterpret_cast<int8_t*>(base),
                             h_lens ? base + o_len : nullptr, h_status ? base + o_st : nullptr, nullptr, m, mrl,
                             flags, s);
        if (rc != ACS_OK) return rc;
        ACS_CUDA(cudaMemcpyAsync(h_out + r0 * rowb, base, (size_t)m * rowb, cudaMemcpyDeviceToHost, s));
        if (h_lens) ACS_CUDA(cudaMemcpyAsync(h_lens + 2 * r0, base + o_len, (size_t)m * 2, cudaMemcpyDeviceToHost, s));
        if (h_status) ACS_CUDA(cudaMemcpyAsync(h_status + r0, base + o_st, (size_t)m, cudaMemcpyDeviceToHost, s));
    }
    for (int k = 0; k < kStreams; ++k) ACS_CUDA(cudaStreamSynchronize(c->streams[k]));
    return ACS_OK;
}

int acs_env_step_host(acs_ctx* c, int8_t* d_state, int32_t* d_step_count, const uint8_t* h_action, int8_t* h_obs,
                      int32_t* h_reward, uint8_t* h_done, uint8_t* h_truncated, int64_t n, int mrl, int horizon,
                      int flags, int64_t* n_bad) {
    if (!c) return fail(ACS_ERR_INVALID, "ctx is null");
    std::lock_guard<std::mutex> lock(c->mu);
    if (n < 0 || (n > 0 && (!d_state || !d_step_count || !h_action || !h_reward || !h_done || !h_truncated)))
        return fail(ACS_ERR_INVALID, "null buffer");
    if (mrl < 1 || mrl > 64) return fail(ACS_ERR_UNSUPPORTED, "packed kernels need 1 <= mrl <= 64");
    ACS_CUDA(cudaSetDevice(c->device));
    const size_t rowb = 2 * (size_t)mrl;
    // The link to the host is the bound of this call (78 bytes per move come back), so the pipeline is
    // built to keep it busy from the first microsecond to the last: rows go through the step kernel
    // in chunks on kStreams streams, each chunk's observation copy starts as soon as its kernel is
    // done, and the per-row scalars (reward, done, truncated) live in one whole-call buffer and come
    // back in three large copies behind the last observation chunk -- 11 device-to-host copies per
    // 1 Mi rows instead of 32, no synchronisation before the final one.
    static const int64_t chunk_rows = [] {  // ACS_HOST_CHUNK_ROWS: rows per pipeline chunk of this call (multiple of 128)
        const char* e = std::getenv("ACS_HOST_CHUNK_ROWS");
        const long long v = e ? std::atoll(e) : 0;
        return (v >= 128 && v % 128 == 0) ? (int64_t)v : kEnvChunkRows;
    }();
    const int64_t chunk = n < chunk_rows ? (n > 0 ? n : 1) : chunk_rows;
    const size_t o_rew = align_up((size_t)n, 256);
    const size_t o_done = o_rew + align_up((size_t)n * 4, 256);
    const size_t o_tr = o_done + align_up((size_t)n, 256);
    const size_t total = o_tr + align_up((size_t)n, 256);
    {
        const int rc = c->out.reserve(total > 0 ? total : 256);
        if (rc != ACS_OK) return rc;
    }
    uint8_t* base = static_cast<uint8_t*>(c->out.p);
    c->h_err[0] = 0;
    c->h_err[1] = ~0ull;
    ACS_CUDA(cudaMemcpyAsync(c->d_err, c->h_err, 16, cudaMemcpyHostToDevice, c->streams[0]));
    ACS_CUDA(cudaEventRecord(c->ev_start, c->streams[0]));
    for (int k = 1; k < kStreams; ++k) ACS_CUDA(cudaStreamWaitEvent(c->streams[k], c->ev_start, 0));
    int64_t ci = 0;
    for (int64_t r0 = 0; r0 < n; r0 += chunk, ++ci) {
        const int k = (int)(ci % kStreams);
        const int64_t m = (n - r0) < chunk ? (n - r0) : chunk;
        cudaStream_t s = c->streams[k];
        ACS_CUDA(cudaMemcpyAsync(base + r0, h_action + r0, (size_t)m, cudaMemcpyHostToDevice, s));
        const int rc = acs_env_step_batch(d_state + r0 * rowb, base + r0, reinterpret_cast<int32_t*>(base + o_rew) + r0,
                                          base + o_done + r0, base + o_tr + r0, d_step_count + r0, nullptr, nullptr,
                                          reinterpret_cast<uint64_t*>(c->d_err), m, mrl, horizon, flags, s);
        if (rc != ACS_OK) return rc;
        if (h_obs) ACS_CUDA(cudaMemcpyAsync(h_obs + r0 * rowb, d_state + r0 * rowb, (size_t)m * rowb, cudaMemcpyDeviceToHost, s));
    }
    for (int k = 1; k < kStreams; ++k) {
        ACS_CUDA(cudaEventRecord(c->ev_done[k], c->streams[k]));
        ACS_CUDA(cudaStreamWaitEvent(c->streams[0], c->ev_done[k], 0));
    }
    if (n > 0) {
        cudaStream_t s = c->streams[0];
        ACS_CUDA(cudaMemcpyAsync(h_reward, base + o_rew, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        ACS_CUDA(cudaMemcpyAsync(h_done, base + o_done, (size_t)n, cudaMemcpyDeviceToHost, s));
        ACS_CUDA(cudaMemcpyAsync(h_truncated, base + o_tr, (size_t)n, cudaMemcpyDeviceToHost, s));
    }
    ACS_CUDA(cudaMemcpyAsync(c->h_err + 2, c->d_err, 16, cudaMemcpyDeviceToHost, c->streams[0]));
    ACS_CUDA(cudaStreamSynchronize(c->streams[0]));  // stream 0 waited for every other stream's work
    if (n_bad) *n_bad = (int64_t)c->h_err[2];
    return ACS_OK;
}

int acs_validate_batch_host(acs_ctx* c, const int8_t* h_in, uint8_t* h_flags, int64_t n, int mrl) {
    if (!c) return fail(ACS_ERR_INVALID, "ctx is null");
    std::lock_guard<std::mutex> lock(c->mu);
    if (n < 0 || (n > 0 && (!h_in || !h_flags)) || mrl < 1) return fail(ACS_ERR_INVALID, "bad argument");
    if (n == 0) return ACS_OK;
    ACS_CUDA(cudaSetDevice(c->device));
    const size_t bytes = (size_t)n * 2 * mrl;
    const size_t o_f = align_up(bytes, 256);
    int rc = c->scratch[0].reserve(o_f + (size_t)n);
    if (rc != ACS_OK) return rc;
    uint8_t* base = static_cast<uint8_t*>(c->scratch[0].p);
    cudaStream_t s = c->streams[0];
    ACS_CUDA(cudaMemcpyAsync(base, h_in, bytes, cudaMemcpyHostToDevice, s));
    rc = acs_validate_batch(reinterpret_cast<int8_t*>(base), base + o_f, n, mrl, s);
    if (rc != ACS_OK) return rc;
    ACS_CUDA(cudaMemcpyAsync(h_flags, base + o_f, (size_t)n, cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaStreamSynchronize(s));
    return ACS_OK;
}

int acs_generic_host(acs_ctx* c, int op, const int8_t* h_in, const uint8_t* h_action, int8_t* h_out, int32_t* h_aux,
                     uint8_t* h_status, int64_t n, int width, int i, int j, int sign, int cyclical) {
    if (!c) return fail(ACS_ERR_INVALID, "ctx is null");
    std::lock_guard<std::mutex> lock(c->mu);
    if (n < 0 || (n > 0 && (!h_in || !h_out || !h_aux || !h_status))) return fail(ACS_ERR_INVALID, "null buffer");
    if (n == 0) return ACS_OK;
    ACS_CUDA(cudaSetDevice(c->device));
    const size_t bytes = (size_t)n * width;
    const int aux_per_row = (op == ACS_OP_ACMOVE || op == ACS_OP_SIMPLIFY_PRESENTATION) ? 2 : 1;
    {
        // Small calls (the reference's one-presentation-at-a-time API: ACMove, ACEnv.step, simplify_*): the cost is
        // API calls and latency, not bytes.  Layout [in | action | aux | out | status] in a pinned staging buffer and
        // on the device: ONE upload of the prefix (aux arrives zeroed), the kernel, ONE download of the suffix.
        const size_t s_act = align_up(bytes, 16), s_aux = s_act + align_up((size_t)n, 16);
        const size_t s_out = s_aux + align_up((size_t)n * 4 * aux_per_row, 16), s_st = s_out + align_up(bytes, 16);
        const size_t s_end = s_st + align_up((size_t)n, 16);
        if (s_end <= kSmallCall) {
            int rc = c->scratch[0].reserve(kSmallCall);
            if (rc != ACS_OK) return rc;
            uint8_t* d = static_cast<uint8_t*>(c->scratch[0].p);
            uint8_t* h = c->h_stage;
            cudaStream_t s = c->streams[0];
            std::memcpy(h, h_in, bytes);
            if (h_action) std::memcpy(h + s_act, h_action, (size_t)n);
            std::memset(h + s_aux, 0, s_out - s_aux);
            ACS_CUDA(cudaMemcpyAsync(d, h, s_out, cudaMemcpyHostToDevice, s));
            rc = acs_generic_batch(op, reinterpret_cast<int8_t*>(d), h_action ? d + s_act : nullptr,
                                   reinterpret_cast<int8_t*>(d + s_out), reinterpret_cast<int32_t*>(d + s_aux), d + s_st, n,
                                   width, i, j, sign, cyclical, s);
            if (rc != ACS_OK) return rc;
            ACS_CUDA(cudaMemcpyAsync(h + s_aux, d + s_aux, s_end - s_aux, cudaMemcpyDeviceToHost, s));
            ACS_CUDA(cudaStreamSynchronize(s));
            std::memcpy(h_out, h + s_out, bytes);
            std::memcpy(h_aux, h + s_aux, (size_t)n * 4 * aux_per_row);
            std::memcpy(h_status, h + s_st, (size_t)n);
            return ACS_OK;
        }
    }
    const size_t o_out = align_up(bytes, 256);
    const size_t o_act = o_out + align_up(bytes, 256);
    const size_t o_aux = o_act + align_up((size_t)n, 256);
    const size_t o_st = o_aux + align_up((size_t)n * 4 * aux_per_row, 256);
    int rc = c->scratch[0].reserve(o_st + (size_t)n);
    if (rc != ACS_OK) return rc;
    uint8_t* base = static_cast<uint8_t*>(c->scratch[0].p);
    cudaStream_t s = c->streams[0];
    ACS_CUDA(cudaMemcpyAsync(base, h_in, bytes, cudaMemcpyHostToDevice, s));
    if (h_action) ACS_CUDA(cudaMemcpyAsync(base + o_act, h_action, (size_t)n, cudaMemcpyHostToDevice, s));
    ACS_CUDA(cudaMemsetAsync(base + o_aux, 0, (size_t)n * 4 * aux_per_row, s));
    rc = acs_generic_batch(op, reinterpret_cast<int8_t*>(base), h_action ? base + o_act : nullptr,
                           reinterpret_cast<int8_t*>(base + o_out), reinterpret_cast<int32_t*>(base + o_aux),
                           base + o_st, n, width, i, j, sign, cyclical, s);
    if (rc != ACS_OK) return rc;
    ACS_CUDA(cudaMemcpyAsync(h_out, base + o_out, bytes, cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaMemcpyAsync(h_aux, base + o_aux, (size_t)n * 4 * aux_per_row, cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaMemcpyAsync(h_status, base + o_st, (size_t)n, cudaMemcpyDeviceToHost, s));
    ACS_CUDA(cudaStreamSynchronize(s));
    return ACS_OK;
}

}  // extern "C"
