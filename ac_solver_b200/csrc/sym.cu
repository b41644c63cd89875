// sym.cu -- canonical forms of presentations under the symmetry group G (ac_sym.cuh), one thread per row.
#include <cstdint>
#include <string>

#include <cuda_runtime.h>

#include "../../include/acsolver_b200.h"
#include "ac_core.cuh"
#include "ac_keys.cuh"
#include "ac_sym.cuh"
#include "acs_internal.h"

namespace acs {

template <int W>
__global__ void canonical_form_kernel(const int8_t* in, int8_t* out, uint8_t* elem, int64_t n, int mrl) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Rel<2 * W> r0 = pack_bytes<2 * W>(in + i * 2 * mrl, mrl), r1 = pack_bytes<2 * W>(in + i * 2 * mrl + mrl, mrl);
    int g = 0;
    const Key<W> c = canonical<W>(make_key<W>(r0, r1), g);
    Rel<2 * W> c0, c1;
    split_key<W>(c, c0, c1);
    unpack_bytes<2 * W>(out + i * 2 * mrl, c0, mrl);
    unpack_bytes<2 * W>(out + i * 2 * mrl + mrl, c1, mrl);
    elem[i] = (uint8_t)g;
}

}  // namespace acs

using namespace acs;

extern "C" int acs_canonical_form(int device, int mrl, const int8_t* h_rows, int64_t n, int8_t* h_out, uint8_t* h_elem) {
    if (n < 0 || (n > 0 && (!h_rows || !h_out || !h_elem))) return ACS_ERR_INVALID;
    if (const int rc = check_key_mrl(mrl, "canonical_form")) return rc;
    for (int64_t r = 0; r < n; ++r) {  // right-padded rows of letters in {+-1, +-2}
        for (int h = 0; h < 2; ++h) {
            bool pad = false;
            for (int t = 0; t < mrl; ++t) {
                const int v = h_rows[r * 2 * mrl + h * mrl + t];
                if ((v != 0 && pad) || v < -2 || v > 2) {
                    set_last_error("canonical_form: rows must be right-padded with letters in {+-1, +-2}");
                    return ACS_ERR_INVALID;
                }
                pad = pad || v == 0;
            }
        }
    }
    if (n == 0) return ACS_OK;
    if (const int rc = open_device(device, "canonical_form")) return rc;
    const size_t bytes = (size_t)n * 2 * mrl;
    int8_t *d_in = nullptr, *d_out = nullptr;
    uint8_t* d_elem = nullptr;
    cudaError_t e = cudaMalloc((void**)&d_in, bytes);
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_out, bytes);
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_elem, (size_t)n);
    if (e == cudaSuccess) e = cudaMemcpy(d_in, h_rows, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        const unsigned grid = (unsigned)((n + 255) / 256);
        if (key_words(mrl) == 1) canonical_form_kernel<1><<<grid, 256>>>(d_in, d_out, d_elem, n, mrl);
        else canonical_form_kernel<2><<<grid, 256>>>(d_in, d_out, d_elem, n, mrl);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(h_out, d_out, bytes, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(h_elem, d_elem, (size_t)n, cudaMemcpyDeviceToHost);
    cudaFree(d_in);
    cudaFree(d_out);
    cudaFree(d_elem);
    return e == cudaSuccess ? ACS_OK : cuda_fail(e, "canonical_form");
}
