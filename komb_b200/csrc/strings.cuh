// strings.cuh — byte-string helpers shared by the text stages (sam.cu interns SAM names, fasta.cu indexes and joins
// FASTA records by name).
#pragma once

#include "common.cuh"

namespace kg {

#ifdef __CUDACC__

// 64-bit seeded hash of the bytes [p, p + len).  Equal hashes never decide equality on their own: every user
// compares the bytes of the strings a hash brings together.
__device__ __forceinline__ uint64_t hash_span(const unsigned char *__restrict__ p, uint32_t len, uint64_t seed) {
    uint64_t h = seed ^ ((uint64_t)len * 0xff51afd7ed558ccdull);
    uint32_t i = 0;
    for (; i + 8 <= len; i += 8) {
        uint64_t w = 0;
#pragma unroll
        for (int b = 0; b < 8; ++b) w |= (uint64_t)p[i + b] << (8 * b);
        h = (h ^ w) * 0xc2b2ae3d27d4eb4full;
        h ^= h >> 29;
    }
    uint64_t w = 0;
    for (int b = 0; i < len; ++i, ++b) w |= (uint64_t)p[i] << (8 * b);
    h = (h ^ w) * 0x165667b19e3779f9ull;
    h ^= h >> 32;
    h *= 0xd6e8feb86659fd93ull;
    h ^= h >> 32;
    return h;
}

#endif  // __CUDACC__

namespace {
// launch geometry of the text kernels: grid-stride loops over at most 16 blocks per SM
constexpr int kThreads = 256;
inline uint32_t grid_for(uint64_t n, int per_block, int sms) {
    const uint64_t g = (n + per_block - 1) / per_block;
    const uint64_t cap = (uint64_t)sms * 16u;
    return (uint32_t)(g < 1 ? 1 : (g > cap ? cap : g));
}
}  // namespace

}  // namespace kg
