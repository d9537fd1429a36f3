// Counter-based generator shared by the device samplers (predict.cu, ss_sample.cu): Philox-4x32-10 (Salmon et al. 2011).
// A draw depends only on (counter, key), so every sampler is reproducible per seed whatever its launch geometry.
#pragma once
#include <cuda_runtime.h>

namespace gpcc {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// Two standard normals from one Philox output (Box-Muller on two 53-bit uniforms in (0, 1)): the state-space samplers.
__device__ __forceinline__ double2 box_muller(uint4 r) {
    const double u1 = ((double)(((unsigned long long)(r.x >> 5) << 26) | (r.y >> 6)) + 0.5) * (1.0 / 9007199254740992.0);
    const double u2 = ((double)(((unsigned long long)(r.z >> 5) << 26) | (r.w >> 6)) + 0.5) * (1.0 / 9007199254740992.0);
    const double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    return make_double2(rad * cs, rad * sn);
}

}  // namespace gpcc
