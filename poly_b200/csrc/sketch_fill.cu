// sketch_fill.cu -- K1: mash.Sketch in the fill regime (L-k < s): every k-mer hash is
// written positionally (/root/reference/search/mash/mash.go:73-84).
//
// Fast path (fixed-length reads, k in the instantiated set, compact output):
//   * one CTA = one warp = one tile of 32 reads; the 32*L input bytes are contiguous in HBM and are
//     brought in by ONE 1-D TMA bulk copy (cp.async.bulk + mbarrier; SASS UBLKCP);
//   * one THREAD per read walks the read 4 bytes per step.  The murmur3 block pre-mix
//     K(p) = rotl(w(p)*c1,15)*c2 of the 4 bytes at position p is computed ONCE and kept
//     in a register ring shared by the k/4 k-mers that consume it, so the cost per
//     k-mer is the body chain + fmix, not k/4 pre-mixes.  The kernel is bound by the
//     ALU pipe (SHF/LOP3 issue at one warp instruction per 2 cycles per SM sub-partition,
//     tools/pipe_bench.cu), i.e. by ALU instruction COUNT, so everything that is not
//     murmur3 arithmetic is kept off that pipe: for k % 4 == 1 the tail pre-mix comes from
//     a 256-entry shared-memory table (2 LSU instructions, table address formed by IMAD on
//     the FMA pipe), the main loop has no bounds tests or predicated stores, and raw words
//     are fetched one step ahead (DESIGN.md "K1", profiles/);
//   * hashes are staged in shared memory ([read][pos], stride L-k words: bank-conflict
//     free when L-k is odd) and leave as ONE bulk store per tile (the compact output
//     [n][L-k] of a tile is contiguous in HBM).
// All global traffic is therefore full-line TMA traffic; the SM only touches smem.
//
// Generic path (any k >= 0, ragged reads, any row stride): one warp per read, every
// k-mer hashed from scratch.  Slower, same results.
#include <algorithm>

#include "common.cuh"
#include "murmur3.cuh"
#include "tma.cuh"
#include "kmer_walk.cuh"

namespace pg {

// ---- K1 fast path ----------------------------------------------------------------
// smem: in tile (32*L bytes + 16 B over-read pad, 16-B rounded) | out tile [32][nk]
// (+ 1 KB static table when k % 4 == 1)
__host__ __device__ inline uint32_t k1_in_bytes(uint32_t L) {
    return (32u * L + 16u + 15u) & ~15u;
}

// lut_stride == 4 arrives as a kernel argument so that the table address byte*4 + base
// stays an IMAD (FMA pipe) instead of being strength-reduced to LEA (ALU pipe).
template <int K>
__global__ void __launch_bounds__(32)
sketch_fill_uniform_kernel(const uint8_t *__restrict__ bases, const SketchDst dst,
                           uint32_t L, uint32_t nk, uint32_t lut_stride) {
    constexpr int NB = K / 4;    // 4-byte body blocks per k-mer
    constexpr int TAIL = K % 4;  // tail bytes per k-mer
    constexpr uint32_t TAILMASK = TAIL == 1 ? 0xffu : TAIL == 2 ? 0xffffu : 0xffffffu;
    constexpr bool LUT = TAIL == 1;
    static_assert(NB >= 1, "fast path needs k >= 4");

    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(16) uint32_t s_lut[LUT ? 256 : 4];
    __shared__ __align__(8) uint64_t s_bar[2];  // [0]: the tile; [1]: the table
    uint8_t *s_in = smem;
    uint32_t *s_out = reinterpret_cast<uint32_t *>(smem + k1_in_bytes(L));

    const uint32_t tid = threadIdx.x;  // lane == read within the tile
    const uint64_t tile = blockIdx.x;
    const uint32_t in_bytes = 32u * L;  // multiple of 16 (host guarantees)

    if (tid == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        fence_mbar_init();
        mbar_expect_tx(&s_bar[0], in_bytes);
        bulk_g2s(s_in, bases + tile * in_bytes, in_bytes, &s_bar[0]);
        if (LUT) {
            mbar_expect_tx(&s_bar[1], 1024u);
            bulk_g2s(s_lut, &g_kmix_byte, 1024u, &s_bar[1]);
        }
    }
    __syncwarp();  // barrier init visible to every lane
    mbar_wait(&s_bar[0], 0);
    if (LUT) mbar_wait(&s_bar[1], 0);

    // my read: bytes [tid*L, tid*L+L) of the tile, realigned to words on the fly
    const uint32_t b0 = tid * L;
    const uint32_t *sw = reinterpret_cast<const uint32_t *>(s_in) + (b0 >> 2);
    const uint8_t *sb = s_in + b0 + 4 * NB;  // tail byte of k-mer i is sb[i]
    const uint32_t sh = (b0 & 3u) * 8u;
    uint32_t *my_out = s_out + tid * nk;
    const uint32_t lut_base = smem_u32(s_lut);

    uint32_t raw_a = sw[0], raw_b = sw[1];
    uint32_t w_cur = __funnelshift_r(raw_a, raw_b, sh);  // bytes 4Q .. 4Q+3 of the read
    raw_a = raw_b; raw_b = sw[2];
    uint32_t w_nxt = __funnelshift_r(raw_a, raw_b, sh);  // bytes 4Q+4 .. 4Q+7
    raw_a = raw_b; raw_b = sw[3];                        // one word ahead of its use
    const uint32_t *swp = sw + 4;

    uint32_t ring[4][NB];  // ring[r][*]: pre-mixes K(4q+r) of the last NB word steps
    // prologue: word steps 0 .. NB-1 only fill the ring
#pragma unroll
    for (int q = 0; q < NB; ++q) {
        ring[0][q] = mm3_kmix(w_cur);
        ring[1][q] = mm3_kmix(__funnelshift_r(w_cur, w_nxt, 8));
        ring[2][q] = mm3_kmix(__funnelshift_r(w_cur, w_nxt, 16));
        ring[3][q] = mm3_kmix(__funnelshift_r(w_cur, w_nxt, 24));
        w_cur = w_nxt;
        w_nxt = __funnelshift_r(raw_a, raw_b, sh);
        raw_a = raw_b;
        raw_b = *swp++;
    }

    // At word step Q = NB + i/4 the k-mers i+r (r = 0..3) complete: their body blocks are
    // ring[r][oldest .. newest], their tail bytes start at position i + r + 4*NB.
    uint32_t i = 0;
    const uint32_t n_main = (nk / (4 * NB)) * (4 * NB);
    while (i < n_main) {  // full groups of NB word steps: no bounds tests
#pragma unroll
        for (int u = 0; u < NB; ++u) PG_K1_STEP(u, false)
    }
#pragma unroll
    for (int u = 0; u < NB; ++u) {  // remainder: < NB full steps plus possibly a partial one
        if (i < nk) PG_K1_STEP(u, true)
    }

    // hand the staged tile to the async proxy and bulk-store it (positional, mash.go:81-84)
    fence_async_smem();
    __syncwarp();
    if (tid == 0) {
        // one bulk store per destination: the local buffer, or (fused all-gather) the gathered
        // buffer of every rank, peers reached through their NVLink-mapped addresses
#pragma unroll
        for (int p = 0; p < PG_MAX_PEERS; ++p)  // static indices: the struct stays in parameter space
            if (p < dst.n) bulk_s2g(dst.ptr[p] + tile * (uint64_t)(32u * nk), s_out, 32u * nk * 4u);  // multiple of 16
        bulk_wait_read0();
    }
}

// ---- K1r: the same walk for RAGGED reads (every read in the fill regime) --------------------
// A warp owns 32 consecutive reads; their bytes [offsets[r0], offsets[r0+32]) are contiguous and
// arrive by one TMA bulk copy (16-byte aligned body; the < 16 tail bytes by plain loads).  Each
// thread walks its own read with its own length, so lanes only diverge at the end of the shorter
// reads.  Output rows have a common stride (>= the longest row); the words beyond a row's count
// are written as zeros (the zero tail of a fresh Mash, as far as the stride reaches), so the whole
// [32][stride] tile leaves as one bulk store.
template <int K>
__global__ void __launch_bounds__(32)
sketch_fill_ragged_kernel(const uint8_t *__restrict__ bases, const uint64_t *__restrict__ offsets,
                          uint32_t *__restrict__ out, uint32_t stride, uint32_t in_cap,
                          uint32_t *__restrict__ count, int32_t *__restrict__ status, uint32_t lut_stride) {
    constexpr int NB = K / 4;
    constexpr int TAIL = K % 4;
    constexpr uint32_t TAILMASK = TAIL == 1 ? 0xffu : TAIL == 2 ? 0xffffu : 0xffffffu;
    constexpr bool LUT = TAIL == 1;
    static_assert(NB >= 1, "fast path needs k >= 4");

    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(16) uint32_t s_lut[LUT ? 256 : 4];
    __shared__ __align__(8) uint64_t s_bar[2];
    uint8_t *s_in = smem;                                        // [in_cap] (16-byte multiple, >= range + 47)
    uint32_t *s_out = reinterpret_cast<uint32_t *>(smem + in_cap);  // [32][stride]

    const uint32_t tid = threadIdx.x;
    const uint64_t r0 = (uint64_t)blockIdx.x * 32;
    const uint64_t t_beg = offsets[r0], t_end = offsets[r0 + 32];
    const uint32_t head = (uint32_t)((uintptr_t)(bases + t_beg) & 15u);
    const uint32_t range = (uint32_t)(t_end - t_beg);
    const uint32_t body = (head + range) & ~15u;
    if (tid == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        fence_mbar_init();
        mbar_expect_tx(&s_bar[0], body);
        if (body) bulk_g2s(s_in, bases + t_beg - head, body, &s_bar[0]);
        if (LUT) {
            mbar_expect_tx(&s_bar[1], 1024u);
            bulk_g2s(s_lut, &g_kmix_byte, 1024u, &s_bar[1]);
        }
    }
    for (uint32_t i = body + tid; i < head + range + 32; i += 32)  // unaligned tail + over-read pad
        s_in[i] = i < head + range ? __ldg(bases + t_beg - head + i) : (uint8_t)0;
    __syncwarp();
    mbar_wait(&s_bar[0], 0);
    if (LUT) mbar_wait(&s_bar[1], 0);

    const uint64_t my_beg = offsets[r0 + tid];
    const uint32_t L = (uint32_t)(offsets[r0 + tid + 1] - my_beg);
    const uint32_t nk = L > (uint32_t)K ? L - (uint32_t)K : 0u;  // mash.go:73
    const uint32_t b0 = head + (uint32_t)(my_beg - t_beg);
    const uint32_t *sw = reinterpret_cast<const uint32_t *>(s_in) + (b0 >> 2);
    const uint8_t *sb = s_in + b0 + 4 * NB;
    const uint32_t sh = (b0 & 3u) * 8u;
    uint32_t *my_out = s_out + tid * stride;
    const uint32_t lut_base = smem_u32(s_lut);

    if (nk > 0) {
        uint32_t raw_a = sw[0], raw_b = sw[1];
        uint32_t w_cur = __funnelshift_r(raw_a, raw_b, sh);
        raw_a = raw_b; raw_b = sw[2];
        uint32_t w_nxt = __funnelshift_r(raw_a, raw_b, sh);
        raw_a = raw_b; raw_b = sw[3];
        const uint32_t *swp = sw + 4;
        uint32_t ring[4][NB];
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            ring[0][q] = mm3_kmix(w_cur);
            ring[1][q] = mm3_kmix(__funnelshift_r(w_cur, w_nxt, 8));
            ring[2][q] = mm3_kmix(__funnelshift_r(w_cur, w_nxt, 16));
            ring[3][q] = mm3_kmix(__funnelshift_r(w_cur, w_nxt, 24));
            w_cur = w_nxt;
            w_nxt = __funnelshift_r(raw_a, raw_b, sh);
            raw_a = raw_b;
            raw_b = *swp++;
        }
        uint32_t i = 0;
        const uint32_t n_main = (nk / (4 * NB)) * (4 * NB);
        while (i < n_main) {
#pragma unroll
            for (int u = 0; u < NB; ++u) PG_K1_STEP(u, false)
        }
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            if (i < nk) PG_K1_STEP(u, true)
        }
    }
    for (uint32_t i = nk; i < stride; ++i) my_out[i] = 0u;  // zero tail up to the row stride
    if (count) count[r0 + tid] = nk;
    if (status) status[r0 + tid] = PG_ITEM_OK;

    fence_async_smem();
    __syncwarp();
    if (tid == 0) {
        bulk_s2g(out + r0 * stride, s_out, 32u * stride * 4u);
        bulk_wait_read0();
    }
}

// ---- generic fill path -----------------------------------------------------------
// One warp per read.  Handles reads with n = max(len-k,0) < s (others are left to the
// select kernel).  Also writes count / zero padding / status for those reads.
__global__ void __launch_bounds__(256)
sketch_fill_generic_kernel(const uint8_t *__restrict__ bases, const uint64_t *__restrict__ offsets,
                           uint32_t uniform_len, uint64_t n_reads, uint64_t first_read, uint32_t k,
                           uint32_t s, uint32_t flags, uint32_t *__restrict__ out,
                           uint64_t row_stride, uint32_t *__restrict__ count,
                           int32_t *__restrict__ status, const SketchDst extra) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); r < n_reads;
         r += warps) {
        const uint64_t row = first_read + r;
        uint64_t beg, len;
        if (offsets) {
            beg = offsets[row];
            len = offsets[row + 1] - beg;
        } else {
            beg = row * (uint64_t)uniform_len;
            len = uniform_len;
        }
        const uint64_t n = len > k ? len - k : 0;  // mash.go:73
        if (n >= s && !(n == 0 && s == 0)) continue;  // select regime (incl. s in {0,1} panics)
        const uint8_t *seq = bases + beg;
        uint32_t *dst = out + row * row_stride;
        for (uint64_t i = lane; i < row_stride; i += 32) {
            // hash, then the zero tail of a fresh Mash as far as the caller's row reaches (at least s
            // words with PG_SKETCH_PAD_ZERO): rows are fully defined whichever kernel produced them
            uint32_t h = 0u;
            if (i < n) {
                const uint8_t *p = seq + i;
                h = mm3_bytes([p](uint32_t j) { return __ldg(p + j); }, k);
            }
            if (extra.n == 0) {
                dst[i] = h;
            } else {  // fused all-gather: the row goes to every destination (out is one of them)
#pragma unroll
                for (int pr = 0; pr < PG_MAX_PEERS; ++pr)
                    if (pr < extra.n) extra.ptr[pr][row * row_stride + i] = h;
            }
        }
        if (lane == 0) {
            if (count) count[row] = (uint32_t)n;
            if (status) status[row] = PG_ITEM_OK;
        }
    }
}

// ---- launchers -------------------------------------------------------------------
template <int K>
static int launch_k1(const uint8_t *d_bases, uint64_t n_tiles, uint32_t L, uint32_t nk,
                     const SketchDst &dst, cudaStream_t st) {
    const size_t smem = k1_in_bytes(L) + (size_t)32 * nk * 4;
    { const int rc_ = func_smem((const void *)sketch_fill_uniform_kernel<K>, smem); if (rc_ != PG_OK) return rc_; }
    sketch_fill_uniform_kernel<K><<<(unsigned)n_tiles, 32, smem, st>>>(d_bases, dst, L, nk, 4u);
    PG_LAUNCH_CHECK("sketch_fill_uniform_kernel");
    return PG_OK;
}

static int dispatch_k1(int k, const uint8_t *d_bases, uint64_t n_tiles, uint32_t L, uint32_t nk,
                       const SketchDst &dst, cudaStream_t st, bool *handled) {
    *handled = true;
    switch (k) {
#define PG_K1_CASE(KK) \
    case KK: return launch_k1<KK>(d_bases, n_tiles, L, nk, dst, st);
        PG_K1_CASE(11) PG_K1_CASE(13) PG_K1_CASE(15) PG_K1_CASE(16) PG_K1_CASE(17) PG_K1_CASE(19)
        PG_K1_CASE(21) PG_K1_CASE(23) PG_K1_CASE(24) PG_K1_CASE(25) PG_K1_CASE(27) PG_K1_CASE(29)
        PG_K1_CASE(31) PG_K1_CASE(32)
#undef PG_K1_CASE
    default: *handled = false; return PG_OK;
    }
}

static int launch_fill_generic(const uint8_t *d_bases, const uint64_t *d_offsets, uint32_t ulen,
                               uint64_t n_reads, uint64_t first_read, int k, int s, uint32_t flags,
                               uint32_t *d_out, uint64_t row_stride, uint32_t *d_count,
                               int32_t *d_status, cudaStream_t st, const SketchDst *extra = nullptr) {
    if (n_reads == 0) return PG_OK;
    const uint64_t blocks = std::min<uint64_t>((n_reads + 7) / 8, (uint64_t)sm_count() * 32);
    SketchDst ex;
    ex.n = 0;
    if (extra) ex = *extra;
    sketch_fill_generic_kernel<<<(unsigned)blocks, 256, 0, st>>>(
        d_bases, d_offsets, ulen, n_reads, first_read, (uint32_t)k, (uint32_t)s, flags, d_out,
        row_stride, d_count, d_status, ex);
    PG_LAUNCH_CHECK("sketch_fill_generic_kernel");
    return PG_OK;
}

int launch_sketch_uniform(const uint8_t *d_bases, uint64_t n_reads, uint32_t L, int k, int s,
                          uint32_t flags, uint32_t *d_out, uint64_t row_stride, int32_t *d_status,
                          cudaStream_t st, const SketchDst *extra) {
    if (n_reads == 0) return PG_OK;
    const uint64_t n = L > (uint32_t)k ? L - (uint32_t)k : 0;
    if (n >= (uint64_t)s && !(n == 0 && s == 0))  // select regime, mash.go:87-102
        return launch_sketch_select(d_bases, nullptr, L, n_reads, k, s, flags, d_out, row_stride,
                                    nullptr, d_status, st, extra);
    // fill regime
    const uint32_t nk = (uint32_t)n;
    uint64_t done = 0;
    const bool compact = row_stride == nk && !(flags & PG_SKETCH_PAD_ZERO);
    bool aligned = ((uintptr_t)d_bases % 16 == 0) && ((uintptr_t)d_out % 16 == 0);
    if (extra)
        for (int p = 0; p < extra->n; ++p) aligned = aligned && ((uintptr_t)extra->ptr[p] % 16 == 0);
    // tiles of 32 reads, one per CTA
    const size_t smem1 = k1_in_bytes(L) + (size_t)32 * nk * 4;
    if (compact && aligned && nk > 0 && (32 * (uint64_t)L) % 16 == 0 && smem1 <= 100 * 1024 && n_reads >= 32) {
        const uint64_t tiles = n_reads / 32;
        bool handled = false;
        uint64_t t0 = 0;
        while (t0 < tiles) {
            const uint64_t nt = std::min<uint64_t>(tiles - t0, 0x7fffffffull);  // grid.x limit
            SketchDst dst;
            dst.n = extra ? extra->n : 1;
            for (int p = 0; p < dst.n; ++p)
                dst.ptr[p] = (extra ? extra->ptr[p] : d_out) + t0 * 32 * (uint64_t)nk;
            int rc = dispatch_k1(k, d_bases + t0 * 32 * (uint64_t)L, nt, L, nk, dst, st, &handled);
            if (rc != PG_OK) return rc;
            if (!handled) break;
            t0 += nt;
        }
        if (handled) {
            done = tiles * 32;
            if (d_status) PG_CUDA(cudaMemsetAsync(d_status, 0, done * sizeof(int32_t), st));
        }
    }
    if (done < n_reads)  // rows the TMA fast path does not take (k not instantiated, < 32 rows left, unaligned buffers)
        return launch_fill_generic(d_bases, nullptr, L, n_reads - done, done, k, s, flags, d_out,
                                   row_stride, nullptr, d_status, st, extra);
    return PG_OK;
}

template <int K>
static int launch_k1r(const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n_tiles, uint32_t stride,
                      uint32_t in_cap, uint32_t *d_out, uint32_t *d_count, int32_t *d_status, cudaStream_t st) {
    const size_t smem = (size_t)in_cap + (size_t)32 * stride * 4;
    { const int rc_ = func_smem((const void *)sketch_fill_ragged_kernel<K>, smem); if (rc_ != PG_OK) return rc_; }
    sketch_fill_ragged_kernel<K><<<(unsigned)n_tiles, 32, smem, st>>>(d_bases, d_offsets, d_out, stride, in_cap, d_count, d_status, 4u);
    PG_LAUNCH_CHECK("sketch_fill_ragged_kernel");
    return PG_OK;
}

int launch_sketch_ragged(const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n_reads,
                         uint64_t max_read_len, int k, int s, uint32_t flags, uint32_t *d_out,
                         uint64_t row_stride, uint32_t *d_count, int32_t *d_status,
                         cudaStream_t st) {
    if (n_reads == 0) return PG_OK;
    const uint64_t nmax = max_read_len > (uint64_t)k ? max_read_len - (uint64_t)k : 0;
    uint64_t done = 0;
    // K1r: every read in the fill regime, rows not wider than the staging allows
    const uint64_t in_cap = (32 * max_read_len + 48 + 15) & ~15ull;
    const uint64_t need_stride = (flags & PG_SKETCH_PAD_ZERO) ? (uint64_t)s : nmax;
    if (nmax > 0 && nmax < (uint64_t)s && row_stride >= need_stride && row_stride * 128 <= 96 * 1024 && in_cap <= 64 * 1024 &&
        (uintptr_t)d_out % 16 == 0 && n_reads >= 32 && (row_stride == need_stride || !(flags & PG_SKETCH_PAD_ZERO) || row_stride >= (uint64_t)s)) {
        const uint64_t tiles = n_reads / 32;
        bool handled = true;
        int rc = PG_OK;
        switch (k) {
#define PG_K1R_CASE(KK) \
    case KK: rc = launch_k1r<KK>(d_bases, d_offsets, tiles, (uint32_t)row_stride, (uint32_t)in_cap, d_out, d_count, d_status, st); break;
            PG_K1R_CASE(11) PG_K1R_CASE(13) PG_K1R_CASE(15) PG_K1R_CASE(16) PG_K1R_CASE(17) PG_K1R_CASE(19)
            PG_K1R_CASE(21) PG_K1R_CASE(23) PG_K1R_CASE(24) PG_K1R_CASE(25) PG_K1R_CASE(27) PG_K1R_CASE(29)
            PG_K1R_CASE(31) PG_K1R_CASE(32)
#undef PG_K1R_CASE
            default: handled = false;
        }
        if (rc != PG_OK) return rc;
        if (handled) done = tiles * 32;
    }
    if (done < n_reads) {
        int rc = launch_fill_generic(d_bases, d_offsets, 0, n_reads - done, done, k, s, flags, d_out, row_stride,
                                     d_count, d_status, st);
        if (rc != PG_OK) return rc;
        if (nmax >= (uint64_t)s && nmax > 0)  // some read may be in the select regime
            return launch_sketch_select(d_bases, d_offsets, 0, n_reads, k, s, flags, d_out, row_stride,
                                        d_count, d_status, st, nullptr, max_read_len);
    }
    return PG_OK;
}

}  // namespace pg
