// sym_host.cpp -- TEST HARNESS: compiles csrc/ac_sym.cuh (the symmetry group on packed keys) for the
// HOST, on top of core_host.cpp's shims, so canonical forms and the group tables can be checked against
// tests/sym_oracle.py on a machine without a GPU.  Test infrastructure only.
#include "core_host.cpp"

// ac_keys.cuh also defines a kernel; it is never called here
static const uint3 blockIdx{}, blockDim{}, threadIdx{};

#include "ac_keys.cuh"
#include "ac_sym.cuh"

template <int W>
static void unpack_key(const Key<W>& q, int8_t* out, int mrl) {
    static const int8_t letter[4] = {2, 1, -2, -1};
    for (int h = 0; h < 2; ++h) {
        const int len = (int)(q.k[h * W + W - 1] >> 58);
        for (int t = 0; t < mrl; ++t)
            out[h * mrl + t] = t < len ? letter[(q.k[h * W + t / 32] >> (2 * (t % 32))) & 3] : 0;
    }
}

template <int W>
static int run_canonical(const int8_t* in, const uint8_t* apply, int8_t* out, uint8_t* elem, int64_t n, int mrl) {
    for (int64_t r = 0; r < n; ++r) {
        Key<W> q;
        int lens[2];
        bool valid;
        if (!pack_root<W>(in + r * 2 * mrl, mrl, q, lens, valid)) return -1;
        int g = apply ? apply[r] : 0;
        const Key<W> c = apply ? sym_apply<W>(q, g) : canonical<W>(q, g);
        unpack_key<W>(c, out + r * 2 * mrl, mrl);
        elem[r] = (uint8_t)g;
    }
    return 0;
}

// apply == NULL: out = canonical form of each row, elem = its element; else out = apply[r] . row r
extern "C" int hostsim_canonical(const int8_t* in, const uint8_t* apply, int8_t* out, uint8_t* elem, int64_t n,
                                 int mrl) {
    if (mrl < 1 || mrl > 61) return -1;
    return mrl <= 29 ? run_canonical<1>(in, apply, out, elem, n, mrl) : run_canonical<2>(in, apply, out, elem, n, mrl);
}

// mul [16][16], inv [16], pi [16][12]
extern "C" void hostsim_sym_tables(uint8_t* mul, uint8_t* inv, uint8_t* pi) {
    for (int g = 0; g < 16; ++g) {
        inv[g] = (uint8_t)sym_inv(g);
        for (int h = 0; h < 16; ++h) mul[16 * g + h] = (uint8_t)sym_mul(g, h);
        for (int m = 0; m < 12; ++m) pi[12 * g + m] = (uint8_t)sym_pi(g, m);
    }
}
