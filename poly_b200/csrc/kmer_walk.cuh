// kmer_walk.cuh -- the register-ring k-mer walk shared by K1 (sketch_fill.cu) and K2
// (sketch_select.cu): one thread walks consecutive k-mer positions of a byte string staged in
// shared memory, 4 bytes (= 4 k-mers) per step.  The murmur3 block pre-mix K(p) of the 4 bytes at
// position p is computed once and kept in a register ring shared by the k/4 k-mers that use it.
//
// PG_KMER_STEP(U, CHECKED, EMIT) is one word step (ring slot U); PG_K1_STEP is the same with the
// positional store.  It uses these locals of the enclosing
// scope (K, NB = K/4, TAIL = K%4, TAILMASK, LUT = (TAIL == 1) are compile-time):
//   w_cur, w_nxt          the realigned words at the current / next word position
//   raw_a, raw_b, swp, sh  raw staged words one step ahead of their use, funnel-shift amount
//   ring[4][NB]            pre-mixes of the last NB word steps
//   sb                     byte pointer: the tail byte of k-mer i is sb[i]      (LUT only)
//   lut_stride, lut_base   shared-memory tail table (256 x kmix(byte)); the stride (4) is a
//                          runtime value so byte*4 + base stays an IMAD on the FMA pipe
//   my_out, i, nk          hashes of k-mers i .. i+3 go to my_out[i ..]; CHECKED guards i+r < nk
#pragma once
#include <stdint.h>

#include "murmur3.cuh"

namespace pg {

__device__ __forceinline__ uint32_t lds_u32(uint32_t saddr) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}

// kmix(b) for a single tail byte b, built at compile time
struct KmixTable {
    uint32_t v[256];
};
constexpr uint32_t c_rotl(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
constexpr KmixTable make_kmix_table() {
    KmixTable t{};
    for (uint32_t b = 0; b < 256; ++b) t.v[b] = c_rotl(b * MM3_C1, 15) * MM3_C2;
    return t;
}
static __device__ __align__(16) const KmixTable g_kmix_byte = make_kmix_table();

// One word step = 4 k-mers (ring slot U).  EMIT(r, value) consumes the hash of k-mer i + r.
#define PG_KMER_STEP(U, CHECKED, EMIT)                                                         \
    {                                                                                          \
        uint32_t w[4];                                                                         \
        w[0] = w_cur;                                                                          \
        w[1] = __funnelshift_r(w_cur, w_nxt, 8);                                               \
        w[2] = __funnelshift_r(w_cur, w_nxt, 16);                                              \
        w[3] = __funnelshift_r(w_cur, w_nxt, 24);                                              \
        uint32_t h[4];                                                                         \
        _Pragma("unroll") for (int r = 0; r < 4; ++r) {                                        \
            uint32_t x = mm3_round0(ring[r][U]);                                               \
            _Pragma("unroll") for (int j = 1; j < NB; ++j)                                     \
                x = mm3_round(x, ring[r][((U) + j) % NB]);                                     \
            if (LUT) x ^= lds_u32(sb[i + r] * lut_stride + lut_base);                          \
            else if (TAIL) x ^= mm3_kmix(w[r] & TAILMASK);                                     \
            x ^= (uint32_t)K;                                                                  \
            h[r] = mm3_fmix(x);                                                                \
            ring[r][U] = mm3_kmix(w[r]);                                                       \
        }                                                                                      \
        EMIT(0, h[0]);                                                                         \
        if (!(CHECKED) || i + 1 < nk) EMIT(1, h[1]);                                           \
        if (!(CHECKED) || i + 2 < nk) EMIT(2, h[2]);                                           \
        if (!(CHECKED) || i + 3 < nk) EMIT(3, h[3]);                                           \
        w_cur = w_nxt;                                                                         \
        w_nxt = __funnelshift_r(raw_a, raw_b, sh);                                             \
        raw_a = raw_b;                                                                         \
        raw_b = *swp++;                                                                        \
        i += 4;                                                                                \
    }
// The same word step with a ROLLED ring: slot 0 is always the oldest pre-mix and the ring is shifted by one
// after the step ((NB - 1) x 4 register moves), so a loop over steps needs ONE step of code instead of NB
// (k = 31: 15 KB of SASS -> 2.5 KB).  For kernels whose unrolled body no longer fits the instruction caches.
#define PG_KMER_STEP_ROLLED(CHECKED, EMIT)                                                     \
    {                                                                                          \
        uint32_t w[4];                                                                         \
        w[0] = w_cur;                                                                          \
        w[1] = __funnelshift_r(w_cur, w_nxt, 8);                                               \
        w[2] = __funnelshift_r(w_cur, w_nxt, 16);                                              \
        w[3] = __funnelshift_r(w_cur, w_nxt, 24);                                              \
        uint32_t h[4];                                                                         \
        _Pragma("unroll") for (int r = 0; r < 4; ++r) {                                        \
            uint32_t x = mm3_round0(ring[r][0]);                                               \
            _Pragma("unroll") for (int j = 1; j < NB; ++j) x = mm3_round(x, ring[r][j]);       \
            if (LUT) x ^= lds_u32(sb[i + r] * lut_stride + lut_base);                          \
            else if (TAIL) x ^= mm3_kmix(w[r] & TAILMASK);                                     \
            x ^= (uint32_t)K;                                                                  \
            h[r] = mm3_fmix(x);                                                                \
            _Pragma("unroll") for (int j = 0; j + 1 < NB; ++j) ring[r][j] = ring[r][j + 1];    \
            ring[r][NB - 1] = mm3_kmix(w[r]);                                                  \
        }                                                                                      \
        EMIT(0, h[0]);                                                                         \
        if (!(CHECKED) || i + 1 < nk) EMIT(1, h[1]);                                           \
        if (!(CHECKED) || i + 2 < nk) EMIT(2, h[2]);                                           \
        if (!(CHECKED) || i + 3 < nk) EMIT(3, h[3]);                                           \
        w_cur = w_nxt;                                                                         \
        w_nxt = __funnelshift_r(raw_a, raw_b, sh);                                             \
        raw_a = raw_b;                                                                         \
        raw_b = *swp++;                                                                        \
        i += 4;                                                                                \
    }
// Rotate the ring by G slots (slot G becomes slot 0).  A loop body of G unrolled PG_KMER_STEP(0..G-1) followed by
// this rotation is the middle ground between the fully unrolled NB-step body (no moves, NB steps of code) and the
// rolled one ((NB - 1) x 4 moves per step): about (NB + 1) x 4 / G moves per step.
#define PG_RING_ROTATE(G)                                                                      \
    {                                                                                          \
        _Pragma("unroll") for (int r = 0; r < 4; ++r) {                                        \
            uint32_t t_[NB];                                                                   \
            _Pragma("unroll") for (int q = 0; q < NB; ++q) t_[q] = ring[r][(q + (G)) % NB];    \
            _Pragma("unroll") for (int q = 0; q < NB; ++q) ring[r][q] = t_[q];                 \
        }                                                                                      \
    }
// positional store: hash of k-mer i + r -> my_out[i + r]
#define PG_EMIT_POSITIONAL(R_, H_) my_out[i + (R_)] = (H_)
#define PG_K1_STEP(U, CHECKED) PG_KMER_STEP(U, CHECKED, PG_EMIT_POSITIONAL)

}  // namespace pg
