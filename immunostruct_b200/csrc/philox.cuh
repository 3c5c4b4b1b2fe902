// Philox4x32-10 (Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC 2011): the counter-based
// stream of the seeded analyses.  Counter (c0, c1, c2, c3), key (k0, k1) -> four uint32 words v0..v3.  Users keep their
// streams apart by counter word 3: item 0 and 1 are the coordinate perturbations of csrc/coordnoise.cu, 2 the Shapley
// permutation keys of csrc/shapley.cu.
#pragma once

#include <cstdint>

namespace is {

struct Philox4 {
    uint32_t v[4];
};

// ten rounds of the 4x32 S-box, the key bumped by the Weyl constants between rounds
__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int round = 0; round < 10; ++round) {
        if (round > 0) { k0 += W0; k1 += W1; }
        const uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
    }
    return Philox4{{c0, c1, c2, c3}};
}

}  // namespace is
