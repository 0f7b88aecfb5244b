// Counter-based uniforms shared by the samplers (gt_lse_sample, gt_child_sample) and the resampler (gt_resample): one
// Philox4x32-10 block per row, counter = (offset + row, stream), key = seed, so a draw depends only on (seed, offset + row)
// and not on the launch.  The samplers use stream 0 and the resampler stream 1: one (seed, offset) can drive both
// without correlated draws.
#pragma once
#include <cstdint>

namespace gt {

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// 53-bit uniform in [0, 1) from the first two words of the block for counter (`ctr`, `stream`) under key `seed`: the
// counter's first two words hold `ctr`, the third `stream`, the fourth 0
__device__ __forceinline__ double philox_uniform53(uint64_t seed, uint64_t ctr, uint32_t stream = 0u) {
    uint32_t r[4];
    philox4x32_10((uint32_t)ctr, (uint32_t)(ctr >> 32), stream, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    return (double)(((uint64_t)(r[0] >> 5) << 26) | (uint64_t)(r[1] >> 6)) * (1.0 / 9007199254740992.0);
}

}  // namespace gt
