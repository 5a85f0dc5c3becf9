// Philox4x32-10 counter-based generator shared by the device simulator (simulate.cu) and the held-out edge split
// (edge_split.cu): one definition, so that a stream keyed by (seed, purpose, a, b, c) means the same words in both.
// Purposes in use: 1-4 simulate.cu, 5 edge_split.cu.
#pragma once
#include <stdint.h>

namespace pangnn {

struct Philox {
    uint32_t key[2];
    uint32_t ctr[4];
    uint32_t out[4];
    int have;
    // one stream per (purpose, genome, gene, draw): 2^32 blocks of 4 words each, never shared between draws
    __device__ Philox(uint64_t seed, uint32_t purpose, uint32_t a, uint32_t b, uint32_t c = 0) : have(0) {
        key[0] = (uint32_t)seed;
        key[1] = (uint32_t)(seed >> 32) ^ (purpose * 0x9E3779B9u);
        ctr[0] = 0; ctr[1] = a; ctr[2] = b; ctr[3] = c;
    }
    __device__ void round10() {
        uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
            c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
        ++ctr[0];
    }
    __device__ uint32_t next() {
        if (have == 0) { round10(); have = 4; }
        return out[4 - have--];
    }
    // uniform in (0, 1): 53 bits
    __device__ double uniform() {
        const uint64_t hi = next(), lo = next();
        return ((double)(((hi << 32) | lo) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    }
    __device__ double normal() {
        const double u1 = uniform(), u2 = uniform();
        return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
    }
};

}  // namespace pangnn
