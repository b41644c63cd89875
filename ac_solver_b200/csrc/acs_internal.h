// acs_internal.h -- declarations shared by the translation units of libacsolver_b200.so.
#pragma once
#include <cstdint>
#include <string>

#include <cuda_runtime.h>

// return the error of a failed CUDA call (acs::cuda_fail)
#define ACS_CUDA(call)                                                \
    do {                                                              \
        const cudaError_t e__ = (call);                               \
        if (e__ != cudaSuccess) return ::acs::cuda_fail(e__, #call);  \
    } while (0)
// cudaMalloc, or run `cleanup` and return ACS_ERR_NOMEM with the text "cudaMalloc(<ptr>): <CUDA error string>"
#define ACS_ALLOC(ptr, bytes, cleanup)                                                                     \
    do {                                                                                                   \
        const cudaError_t e__ = cudaMalloc((void**)&(ptr), (size_t)(bytes));                               \
        if (e__ != cudaSuccess) {                                                                          \
            cudaGetLastError();                                                                            \
            cleanup;                                                                                       \
            return ::acs::fail(ACS_ERR_NOMEM, std::string("cudaMalloc(" #ptr "): ") + cudaGetErrorString(e__)); \
        }                                                                                                  \
    } while (0)

namespace acs {

// Arguments of the batched move / env-step kernels (moves_kernel.cu).
struct StepParams {
    const int8_t* in;       // [n, 2*mrl]
    int8_t* out;            // [n, 2*mrl], may alias in
    const uint8_t* action;  // [n]
    uint8_t* lens;          // [n,2] or null
    uint8_t* status;        // [n] or null
    unsigned long long* err;  // {count, min row} or null
    int32_t* reward;        // [n] or null  (null => plain ACMove, no env bookkeeping)
    uint8_t* done;          // [n]
    uint8_t* truncated;     // [n]
    int32_t* step_count;    // [n] in/out
    int64_t n;
    int mrl;
    int cyclical;
    int horizon;
    int max_reward;
    int bulk_ok;            // in/out are 16-byte aligned: TMA bulk copies allowed
    int trusted;            // rows are normal forms for `cyclical` (see ac_core.cuh apply_move)
    int lens_valid;         // `lens` holds the current relator lengths on entry (in/out)
    uint8_t* action_log;    // [n, log_stride] or null: action written at the pre-step counter (env only)
    int log_stride;
};

// thread-local error text behind acs_last_error() (capi.cu)
void set_last_error(const char* msg);
// sets the error text and returns code
int fail(int code, const std::string& msg);
// a failed CUDA call: clears the runtime's last error and returns ACS_ERR_NOMEM for an allocation failure,
// ACS_ERR_CUDA for any other, with the text "<what>: <CUDA error string>"
int cuda_fail(cudaError_t e, const std::string& what);
// selects `device` for the calling thread: ACS_ERR_NO_DEVICE without a visible device, ACS_ERR_INVALID
// for an index out of range ("<who>: device index out of range")
int open_device(int device, const char* who);
// ACS_ERR_UNSUPPORTED unless a packed key holds relators of mrl letters
// ("<who> needs 1 <= max_relator_length <= 61")
int check_key_mrl(int mrl, const char* who);
// n visited records of `stride` words (see records_unpack_kernel, ac_keys.cuh) -> int8 rows in host memory,
// and with h_gid the global id word of each node record; synchronises `s`
int records_to_host(int W, const uint64_t* d_recs, int stride, int64_t n, int mrl, int8_t* h_rows, int64_t* h_gid,
                    cudaStream_t s);

cudaError_t launch_step(const StepParams& P, cudaStream_t s);

// byte-domain reference-semantics kernel for any int8 alphabet (generic_kernel.cu)
enum GenericOp : int {
    OP_ACMOVE = 0,
    OP_CONCAT_RAW = 1,
    OP_CONJ_RAW = 2,
    OP_SIMPLIFY_RELATOR = 3,
    OP_SIMPLIFY_PRESENTATION = 4,
};
struct GenericParams {
    int op;
    const int8_t* in;       // [n, width]
    const uint8_t* action;  // [n] (OP_ACMOVE)
    int8_t* out;            // [n, width]
    int32_t* aux;           // OP_ACMOVE / SIMPLIFY_PRESENTATION: [n,2] lengths; RAW: [n] new size or -1/-2;
                            // SIMPLIFY_RELATOR: [n] length
    uint8_t* status;        // [n]
    int64_t n;
    int width;              // letters per row (2*mrl, or the relator width for SIMPLIFY_RELATOR)
    int i, j, sign;         // RAW ops
    int cyclical;
};
cudaError_t launch_generic(const GenericParams& P, cudaStream_t s);
cudaError_t launch_validate(const int8_t* in, uint8_t* flags, int64_t n, int mrl, cudaStream_t s);
cudaError_t launch_autoreset(int8_t* state, const int8_t* init, int8_t* final_obs, const uint8_t* done,
                             const uint8_t* trunc, int32_t* step_count, int32_t* final_steps, uint8_t* lens,
                             const uint8_t* init_lens, int64_t n, int mrl, cudaStream_t s);

cudaError_t launch_reward_transform(const int32_t* reward, const uint8_t* done, double* stats, float* out, int64_t n,
                                    double gamma, double eps, int normalize, int clip, double lo, double hi,
                                    cudaStream_t s);
struct CurriculumParams {
    int8_t* state;            // [n, 2*mrl]
    const int8_t* pool;       // [n_states, 2*mrl]
    const uint8_t* pool_lens; // [n_states, 2]
    uint8_t* lens;            // [n, 2]
    const uint8_t* done;
    const uint8_t* trunc;
    int32_t* step_count;
    int32_t* cur_state;       // [n]   index into the pool of each environment's episode
    uint8_t* solved;          // [n_states]
    int32_t* solved_list;     // [n_states] solved states in the order they were first solved
    unsigned long long* best; // [n_states] (path length << 32 | env) of the shortest solving episode, ~0 = none
    uint8_t* best_actions;    // [n_states, log_stride]
    const uint8_t* action_log;  // [n, log_stride]
    int8_t* final_obs;        // [n, 2*mrl] or null
    int32_t* final_steps;     // [n] or null
    long long* counters;      // [0] next unprocessed state, [1] number solved, [2] draws made, [3] episodes finished
    int64_t n;
    int n_states, mrl, log_stride;
    float repeat_solved_prob;
    unsigned long long seed;
};

cudaError_t launch_curriculum(const CurriculumParams& P, cudaStream_t s);

}  // namespace acs
