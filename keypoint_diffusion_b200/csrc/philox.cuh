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

// standard normal for (seed, step, atom, channel, word): counter = (atom, step+1, ch/4, word), key = seed; one counter
// gives channels 4k..4k+3 by Box-Muller on (0,1] x [0,1).  Word 0 is the plain loop, 3u+kind an inpainting pass.
__device__ __forceinline__ float philox_normal(uint64_t seed, int step, int atom, int ch, uint32_t word = 0) {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)atom, (uint32_t)(step + 1), (uint32_t)(ch >> 2), word),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const int q = ch & 3;
    const uint32_t ua = q < 2 ? r.x : r.z, ub = q < 2 ? r.y : r.w;
    const float u1 = ((float)ua + 1.0f) * 2.3283064365386963e-10f;
    const float u2 = (float)ub * 2.3283064365386963e-10f;
    const float rad = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincosf(6.283185307179586f * u2, &sn, &cs);
    return (q & 1) ? rad * sn : rad * cs;
}

}  // namespace kpd
