// xxh64.cuh -- XXH64 (seed 0) of one buffer by a group of four lanes, the hashing core of k_xxh64 (content checksum of decoded
// frames) and k_cxxh64 (content checksum of frames being compressed).  The four accumulators of XXH64 are independent chains
// over every 4th 8-byte word: lane k of the group walks accumulator k over the 32-byte stripes; lane 0 merges and finishes the
// tail.  Every lane of the warp must call it (the merge shuffles over the full warp); the result is valid on lane k == 0.
#pragma once
#include <stdint.h>

namespace b200z {

__device__ __forceinline__ uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
__device__ __forceinline__ uint64_t ld_u64_unaligned(const uint8_t *p) {
    uintptr_t a = (uintptr_t)p;
    if ((a & 7) == 0) return *reinterpret_cast<const uint64_t *>(p);
    const uint64_t *q = reinterpret_cast<const uint64_t *>(a & ~(uintptr_t)7);
    uint32_t sh = (uint32_t)(a & 7) * 8u;
    return (q[0] >> sh) | (q[1] << (64u - sh));
}
__device__ __forceinline__ uint64_t xxh64_group4(const uint8_t *p, const uint64_t len, const uint32_t k) {
    const uint64_t P1 = 0x9E3779B185EBCA87ull, P2 = 0xC2B2AE3D27D4EB4Full, P3 = 0x165667B19E3779F9ull, P4 = 0x85EBCA77C2B2AE63ull, P5 = 0x27D4EB2F165667C5ull;
    const uint64_t nstripes = len >> 5;
    uint64_t v = k == 0 ? P1 + P2 : (k == 1 ? P2 : (k == 2 ? 0ull : 0ull - P1));
    const uint8_t *q = p + 8 * k;
    // the accumulator is a serial chain, the loads are not: 16 stripes' words are requested together (the loop is bound by
    // memory latency otherwise: 1 ms per GiB with one load in flight per lane)
    uint64_t s = 0;
    if ((((uintptr_t)q) & 7) == 0) {
        // software pipelined: the next 16 stripes' words are in flight while this batch goes through the (serial) rounds -- what a
        // lone huge frame needs (four lanes cannot hide a DRAM round trip any other way), and more bytes in flight for many frames
        if (s + 16 <= nstripes) {
            uint64_t w[16];
#pragma unroll
            for (int i = 0; i < 16; i++) w[i] = *reinterpret_cast<const uint64_t *>(q + 32 * i);
            s += 16; q += 512;
            for (; s + 16 <= nstripes; s += 16, q += 512) {
                uint64_t n[16];
#pragma unroll
                for (int i = 0; i < 16; i++) n[i] = *reinterpret_cast<const uint64_t *>(q + 32 * i);
#pragma unroll
                for (int i = 0; i < 16; i++) { v += w[i] * P2; v = rotl64(v, 31) * P1; }
#pragma unroll
                for (int i = 0; i < 16; i++) w[i] = n[i];
            }
#pragma unroll
            for (int i = 0; i < 16; i++) { v += w[i] * P2; v = rotl64(v, 31) * P1; }
        }
    } else {
        const uint32_t sh = (uint32_t)(((uintptr_t)q) & 7) * 8u;
        const uint64_t *qa = reinterpret_cast<const uint64_t *>(((uintptr_t)q) & ~(uintptr_t)7);
        for (; s + 16 <= nstripes; s += 16, q += 512, qa += 64) {
            uint64_t lo[16], hi[16];
#pragma unroll
            for (int i = 0; i < 16; i++) { lo[i] = qa[4 * i]; hi[i] = qa[4 * i + 1]; }
#pragma unroll
            for (int i = 0; i < 16; i++) { const uint64_t w = (lo[i] >> sh) | (hi[i] << (64u - sh)); v += w * P2; v = rotl64(v, 31) * P1; }
        }
    }
    for (; s < nstripes; s++, q += 32) {
        v += ld_u64_unaligned(q) * P2;
        v = rotl64(v, 31) * P1;
    }
    const uint32_t gbase = (threadIdx.x & 31u) & ~3u;
    uint64_t v0 = __shfl_sync(0xffffffffu, v, gbase), v1 = __shfl_sync(0xffffffffu, v, gbase + 1), v2 = __shfl_sync(0xffffffffu, v, gbase + 2),
             v3 = __shfl_sync(0xffffffffu, v, gbase + 3);
    if (k != 0) return 0;
    uint64_t h;
    if (len >= 32) {
        h = rotl64(v0, 1) + rotl64(v1, 7) + rotl64(v2, 12) + rotl64(v3, 18);
        uint64_t vs[4] = {v0, v1, v2, v3};
#pragma unroll
        for (int i = 0; i < 4; i++) { uint64_t x = rotl64(vs[i] * P2, 31) * P1; h ^= x; h = h * P1 + P4; }
    } else h = P5;   // seed 0 + PRIME64_5
    h += len;
    const uint8_t *r = p + (nstripes << 5), *end = p + len;
    while (r + 8 <= end) { uint64_t x = rotl64(ld_u64_unaligned(r) * P2, 31) * P1; h ^= x; h = rotl64(h, 27) * P1 + P4; r += 8; }
    if (r + 4 <= end) { uint32_t w = (uint32_t)r[0] | ((uint32_t)r[1] << 8) | ((uint32_t)r[2] << 16) | ((uint32_t)r[3] << 24); h ^= (uint64_t)w * P1; h = rotl64(h, 23) * P2 + P3; r += 4; }
    while (r < end) { h ^= (uint64_t)(*r) * P5; h = rotl64(h, 11) * P1; r++; }
    h ^= h >> 33; h *= P2; h ^= h >> 29; h *= P3; h ^= h >> 32;
    return h;
}


}  // namespace b200z
