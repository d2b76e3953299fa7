// Philox4x32-10 (Salmon et al., SC'11) and the 53-bit uniform map shared by the nested-sampling
// walks (nested.cu) and the multivariate-normal draws (mvn.cu).  Restated on the CPU in
// oracle/philox.py.
#pragma once

namespace abr {

struct U4 { unsigned x, y, z, w; };

__device__ __forceinline__ U4 philox(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return U4{c0, c1, c2, c3};
}

// two 32-bit words -> double in [0, 1) with 53 random bits
__device__ __forceinline__ double u53(unsigned hi, unsigned lo) {
    return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) / 9007199254740992.0;
}

}  // namespace abr
