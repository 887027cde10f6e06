// Philox4x32-10 (Salmon et al. 2011): the counter-based generator behind every in-kernel Gaussian draw of the loop.
#pragma once
#include <stdint.h>

namespace kpd {

__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}

}  // namespace kpd
