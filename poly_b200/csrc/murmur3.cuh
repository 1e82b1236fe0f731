// murmur3.cuh -- MurmurHash3_x86_32 (seed 0) device primitives.
//
// Replaces github.com/spaolacci/murmur3 v1.1.0 Sum32 at its only call site on the
// hot path, /root/reference/search/mash/mash.go:76.  The block pre-mix
// K(w) = rotl(w*c1,15)*c2 depends only on the 4 bytes at a position, so kernels
// compute it once per position and share it between the k/4 k-mers that consume it
// (DESIGN.md "K1").
#pragma once
#include <stdint.h>

namespace pg {

constexpr uint32_t MM3_C1 = 0xcc9e2d51u;
constexpr uint32_t MM3_C2 = 0x1b873593u;
constexpr uint32_t MM3_N = 0xe6546b64u;

__device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return __funnelshift_l(x, x, r); }

// block pre-mix of one little-endian 4-byte word (also the tail mix of 1..3 bytes
// once the unused high bytes are masked to zero)
__device__ __forceinline__ uint32_t mm3_kmix(uint32_t w) {
    w *= MM3_C1;
    w = rotl32(w, 15);
    w *= MM3_C2;
    return w;
}
// first body round with h == seed == 0:  h ^ k == k
__device__ __forceinline__ uint32_t mm3_round0(uint32_t kq) { return rotl32(kq, 13) * 5u + MM3_N; }
__device__ __forceinline__ uint32_t mm3_round(uint32_t h, uint32_t kq) {
    h ^= kq;
    h = rotl32(h, 13);
    return h * 5u + MM3_N;
}
__device__ __forceinline__ uint32_t mm3_fmix(uint32_t h) {
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return h;
}

// Hash k raw bytes at an arbitrary (unaligned) address, byte loads only.  Used by
// the generic (any k, ragged) path.
template <typename LoadByte>
__device__ __forceinline__ uint32_t mm3_bytes(LoadByte ld, uint32_t k) {
    uint32_t h = 0;
    uint32_t nb = k >> 2;
    for (uint32_t b = 0; b < nb; ++b) {
        uint32_t w = (uint32_t)ld(4 * b) | ((uint32_t)ld(4 * b + 1) << 8) |
                     ((uint32_t)ld(4 * b + 2) << 16) | ((uint32_t)ld(4 * b + 3) << 24);
        h = mm3_round(h, mm3_kmix(w));
    }
    uint32_t t = k & 3u;
    if (t) {
        uint32_t w = 0;
        for (uint32_t j = 0; j < t; ++j) w |= (uint32_t)ld(4 * nb + j) << (8 * j);
        h ^= mm3_kmix(w);
    }
    h ^= k;
    return mm3_fmix(h);
}

}  // namespace pg
