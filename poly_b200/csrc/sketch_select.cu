// sketch_select.cu -- K2: mash.Sketch in the select regime (L-k >= s): the sketch is the
// ascending bottom-s MULTISET of all k-mer hashes (closed form of
// /root/reference/search/mash/mash.go:87-102: fill, sort once at i == s-1, then
// replace-max + re-sort; duplicates are kept, SURVEY.md 8a row a3).
//
// Three kernels share this file (dispatch at the bottom, launch_sketch_select):
//   K2t  sketch_thresh_walk_kernel + sketch_thresh_select_kernel -- the default for the instantiated k: a value
//        threshold admits ~s hashes per row into global candidate lists, a counting sort picks the bottom-s
//        (section "K2t" below); rows on which the estimate fails go to
//   K2w  sketch_select_walk_kernel -- exact streaming kernel with the register-ring walk, one CTA per row;
//   generic sketch_select_kernel -- any k <= 1024, described next.
// Sketches above 16384 words or k above 1024 leave this file for sketch_select_large.cu.
//
// The generic kernel: one CTA per read.  The read is streamed through shared memory in chunks:
//   stage    the chunk's bytes arrive by a 1-D TMA bulk copy (16-byte aligned body; the few
//            unaligned tail bytes by plain loads), double-buffered one chunk ahead
//   phase 1  pre-mix K(p) of every position of the chunk, once       (shared via smem)
//   phase 2  one k-mer per thread: body chain over K(i+4j), tail, fmix; hashes below
//            the current admission limit are appended to the candidate buffer
//   prune    when the buffer would overflow: exact radix-select of the s-th smallest
//            value, keep all smaller values plus the needed number of ties
//   final    bucket sort-select: histogram of the candidates over 2048 value buckets, scan,
//            scatter of the buckets below the one holding the s-th smallest value, rank inside
//            each (tiny) bucket -> the sorted bottom-s directly (O(candidates), exact for
//            ties).  Degenerate value distributions (a bucket that does not fit the scratch
//            area, e.g. a homopolymer read) take the general path: exact radix select to s,
//            bitonic sort in shared memory.
// Nothing but the read bytes and the s output words touches HBM.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "murmur3.cuh"
#include "tma.cuh"
#include "kmer_walk.cuh"

namespace pg {

namespace {

constexpr int SEL_THREADS = 512;
constexpr int SEL_CHUNK = 2048;     // k-mer positions per chunk
constexpr int SEL_MAX_S = 16384;    // largest sketch size of the shared-memory kernels (beyond: sketch_select_large.cu)
constexpr int SEL_LOOKAHEAD = 1024; // max k supported by the staged path (bytes beyond chunk)
constexpr int SEL_NBK = 2048;       // value buckets of the final sort-select (v >> 21)
constexpr int SEL_BSHIFT = 21;
constexpr int SEL_STAGE_WORDS = (SEL_CHUNK + SEL_LOOKAHEAD + 16 + 16) / 4;  // 15 B head + 8 B slack, 16-B multiple

struct SelSmem {
    uint32_t *cand;   // [cap]
    uint32_t *keep;   // [s]
    uint32_t *kv;     // [SEL_CHUNK + SEL_LOOKAHEAD]
    uint32_t *bytes;  // 2 x [SEL_STAGE_WORDS] staged read bytes (word view), double-buffered
    uint32_t *hist;   // [SEL_NBK + 1] (radix select uses the first 256 words)
    uint32_t *misc;   // [8]: 0 cnt, 1 prefix, 2 want, 3 kept_lt, 4 kept_eq, 5 hmin_later, 6 bt, 7 need (K2w: 8..10 per-chunk counters)
    uint32_t tmpcap;  // words available at keep[] for the final scatter (keep+kv+bytes are contiguous)
};

// atom.shared.add with the old value, as ONE instruction.  nvcc wraps atomicAdd(&shared[i], 1) whose result is
// used into a leader-election loop over the distinct addresses of the warp (ncu: ~12 instructions x up to 32
// rounds per call); the hardware resolves same-address lanes by itself.
__device__ __forceinline__ uint32_t smem_fetch_inc(uint32_t *p) {
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(p)) : "memory");
    return old;
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t saddr) {  // shared-space load from a 32-bit shared address
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void stg_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// acc += (x < e), n += (x == e): a compare and a predicated add each (nvcc's own code is add, select, move per counter)
__device__ __forceinline__ void count_lt_eq(uint32_t x, uint32_t e, uint32_t &acc, uint32_t &n) {
    asm("{\n\t.reg .pred p, q;\n\tsetp.lt.u32 p, %2, %3;\n\tsetp.eq.u32 q, %2, %3;\n\t@p add.u32 %0, %0, 1;\n\t@q add.u32 %1, %1, 1;\n\t}"
        : "+r"(acc), "+r"(n)
        : "r"(x), "r"(e));
}

__device__ __forceinline__ uint32_t smem_window(const uint32_t *bytes_w, uint32_t p) {
    // little-endian 4-byte window at byte position p of the staged bytes
    const uint32_t a = bytes_w[p >> 2], b = bytes_w[(p >> 2) + 1];
    return __funnelshift_r(a, b, (p & 3u) * 8u);
}

// exact selection: on return cand[0..s) holds the s smallest values (as a multiset) of
// cand[0..cnt); returns the s-th smallest value.  All threads must call.
template <int NT>
__device__ uint32_t prune_to_s(const SelSmem &m, uint32_t cnt, uint32_t s) {
    const uint32_t tid = threadIdx.x;
    uint32_t prefix = 0, mask = 0, want = s;  // want: 1-based rank inside the current bucket
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (uint32_t i = tid; i < 256; i += NT) m.hist[i] = 0;
        __syncthreads();
        for (uint32_t i = tid; i < cnt; i += NT) {
            const uint32_t e = m.cand[i];
            if ((e & mask) == prefix) atomicAdd(&m.hist[(e >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid < 32) {  // warp 0 scans the 256 bins (8 per lane)
            uint32_t loc[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { loc[j] = m.hist[tid * 8 + j]; sum += loc[j]; }
            uint32_t incl = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
                if ((int)tid >= d) incl += y;
            }
            uint32_t before = incl - sum;
            if (before < want && want <= incl) {  // the bucket lies in my 8 bins
                uint32_t w = want - before;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (w <= loc[j]) {
                        m.misc[1] = prefix | ((uint32_t)(tid * 8 + j) << shift);
                        m.misc[2] = w;
                        break;
                    }
                    w -= loc[j];
                }
            }
        }
        __syncthreads();
        prefix = m.misc[1];
        want = m.misc[2];
        mask |= 255u << shift;
        __syncthreads();
    }
    const uint32_t v = prefix;     // s-th smallest value
    const uint32_t need_eq = want; // copies of v that belong to the bottom-s multiset
    const uint32_t n_lt = s - need_eq;
    if (tid == 0) { m.misc[3] = 0; m.misc[4] = 0; }
    __syncthreads();
    for (uint32_t i0 = 0; i0 < cnt; i0 += NT) {
        const uint32_t i = i0 + tid;
        const uint32_t e = i < cnt ? m.cand[i] : 0xffffffffu;
        const bool lt = i < cnt && e < v;
        const bool eq = i < cnt && e == v;
        const uint32_t blt = __ballot_sync(0xffffffffu, lt), beq = __ballot_sync(0xffffffffu, eq);
        const uint32_t lane = tid & 31u, below = (1u << lane) - 1u;
        uint32_t base_lt = 0, base_eq = 0;
        if (lane == 0) {
            if (blt) base_lt = atomicAdd(&m.misc[3], __popc(blt));
            if (beq) base_eq = atomicAdd(&m.misc[4], __popc(beq));
        }
        base_lt = __shfl_sync(0xffffffffu, base_lt, 0);
        base_eq = __shfl_sync(0xffffffffu, base_eq, 0);
        if (lt) m.keep[base_lt + __popc(blt & below)] = e;
        if (eq) {
            const uint32_t q = base_eq + __popc(beq & below);
            if (q < need_eq) m.keep[n_lt + q] = e;
        }
    }
    __syncthreads();
    for (uint32_t i = tid; i < s; i += NT) m.cand[i] = m.keep[i];
    __syncthreads();
    return v;
}

template <int NT>
__device__ void bitonic_sort(uint32_t *x, uint32_t P) {
    const uint32_t tid = threadIdx.x;
    for (uint32_t k2 = 2; k2 <= P; k2 <<= 1) {
        for (uint32_t j = k2 >> 1; j > 0; j >>= 1) {
            for (uint32_t t = tid; t < (P >> 1); t += NT) {
                const uint32_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const uint32_t ixj = i | j;
                const bool up = (i & k2) == 0;
                const uint32_t a = x[i], b = x[ixj];
                if ((a > b) == up) { x[i] = b; x[ixj] = a; }
            }
            __syncthreads();
        }
    }
}

// Final stage, fast path.  cand[0..cnt) holds a superset of the bottom-s multiset (cnt >= s).
// Writes the ascending bottom-s to dst and returns true, or returns false (nothing written) if
// the buckets up to the threshold bucket do not fit the scratch area.  All threads must call.
template <int NT>
__device__ bool final_bucket_sort(const SelSmem &m, uint32_t cnt, uint32_t s, uint32_t *__restrict__ dst,
                                  const uint32_t bshift = SEL_BSHIFT) {
    const uint32_t tid = threadIdx.x;
    uint32_t *bstart = m.hist;  // counts, then exclusive starts; [SEL_NBK] = total
    uint32_t *tmp = m.keep;
    for (uint32_t i = tid; i <= SEL_NBK; i += NT) bstart[i] = 0;
    if (tid == 0) { m.misc[6] = 0xffffffffu; m.misc[7] = 0; }
    __syncthreads();
    for (uint32_t i = tid; i < cnt; i += NT) atomicAdd(&bstart[m.cand[i] >> bshift], 1u);
    __syncthreads();
    // exclusive scan: 4 buckets per thread, warp scan, then the 16 warp totals
    constexpr int PER = SEL_NBK / NT;
    uint32_t c[PER], sum = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) { c[j] = bstart[tid * PER + j]; sum += c[j]; }
    uint32_t incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
        if ((int)(tid & 31u) >= d) incl += y;
    }
    __shared__ uint32_t s_warp[NT / 32];
    if ((tid & 31u) == 31u) s_warp[tid >> 5] = incl;
    __syncthreads();
    uint32_t base = 0;
    for (uint32_t w = 0; w < (tid >> 5); ++w) base += s_warp[w];
    uint32_t run = base + incl - sum;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        bstart[tid * PER + j] = run;
        if (run < s && run + c[j] >= s) { m.misc[6] = tid * PER + j; m.misc[7] = run + c[j]; }  // threshold bucket
        run += c[j];
    }
    if (tid == NT - 1) bstart[SEL_NBK] = run;
    __syncthreads();
    const uint32_t bt = m.misc[6], need = m.misc[7];
    if (bt == 0xffffffffu || need > m.tmpcap) return false;
    // scatter buckets <= bt (slot order inside a bucket is arbitrary); the per-bucket cursors
    // sit right behind the scattered elements in the scratch area
    uint32_t *cursor = tmp + need;  // [bt + 1]
    if (need + bt + 1 > m.tmpcap) return false;
    for (uint32_t i = tid; i <= bt; i += NT) cursor[i] = 0;
    __syncthreads();
    for (uint32_t i = tid; i < cnt; i += NT) {
        const uint32_t e = m.cand[i], b = e >> bshift;
        if (b <= bt) tmp[bstart[b] + smem_fetch_inc(&cursor[b])] = e;
    }
    __syncthreads();
    // rank inside the bucket -> final position (ties keep distinct slots via the index tie-break)
    for (uint32_t p = tid; p < need; p += NT) {
        const uint32_t e = tmp[p], b = e >> bshift;
        const uint32_t lo = bstart[b], hi = bstart[b + 1];
        uint32_t r = 0;
        for (uint32_t q = lo; q < hi; ++q) {
            const uint32_t x = tmp[q];
            r += (x < e) || (x == e && q < p);
        }
        if (lo + r < s) dst[lo + r] = e;
    }
    __syncthreads();
    return true;
}

__global__ void __launch_bounds__(SEL_THREADS)
sketch_select_kernel(const uint8_t *__restrict__ bases, const uint64_t *__restrict__ offsets,
                     uint32_t uniform_len, uint64_t n_reads, uint32_t k, uint32_t s, uint32_t P,
                     uint32_t cap, uint32_t flags, uint32_t *__restrict__ out, uint64_t row_stride,
                     uint32_t *__restrict__ count, int32_t *__restrict__ status, const SketchDst extra) {
    extern __shared__ __align__(16) uint32_t smem_w[];
    SelSmem m;
    m.cand = smem_w;
    m.keep = m.cand + cap;
    m.kv = m.keep + ((s + 3u) & ~3u) + 4u;  // 16-byte granules keep the TMA stage buffers aligned
    m.bytes = m.kv + SEL_CHUNK + SEL_LOOKAHEAD;
    m.hist = m.bytes + 2 * SEL_STAGE_WORDS;
    m.misc = m.hist + SEL_NBK + 1;
    m.tmpcap = (uint32_t)(m.hist - m.keep);

    __shared__ __align__(8) uint64_t s_bar[2];
    uint32_t par0 = 0u, par1 = 0u;  // barrier parities (uniform across the CTA)
    const uint32_t tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    const uint32_t nb = k >> 2, tail = k & 3u;
    const uint32_t tailmask = tail == 1 ? 0xffu : tail == 2 ? 0xffffu : 0xffffffu;

    for (uint64_t row = blockIdx.x; row < n_reads; row += gridDim.x) {
        uint64_t beg, len;
        if (offsets) {
            beg = offsets[row];
            len = offsets[row + 1] - beg;
        } else {
            beg = row * (uint64_t)uniform_len;
            len = uniform_len;
        }
        const uint64_t n = len > k ? len - k : 0;
        if (n < s || n == 0) continue;  // fill regime: other kernel
        const uint8_t *seq = bases + beg;
        uint32_t *dst = out + row * row_stride;
        if (s == 0) {  // mash.go:96 reads Sketches[-1] on the first k-mer
            if (tid == 0) {
                if (status) status[row] = PG_ITEM_PANIC;
                if (count) count[row] = 0;
            }
            continue;
        }

        if (tid == 0) { m.misc[0] = 0; m.misc[5] = 0xffffffffu; }
        __syncthreads();
        uint64_t limit = 1ull << 32;  // admit h < limit
        uint32_t h_first = 0;

        // chunk c lives in stage buffer c & 1; its copy is issued one iteration ahead
        auto issue_stage = [&](uint64_t c0, uint32_t buf) {
            // bytes [c0, c0 + ch + k) of the read -> sb[head ..): 16-byte aligned body by TMA,
            // the (< 16) trailing bytes and 8 bytes of zero slack by plain stores
            const uint32_t ch = (uint32_t)min((uint64_t)SEL_CHUNK, n - c0);
            const uint32_t nbytes = ch + k;
            const uint8_t *src = seq + c0;
            const uint32_t head = (uint32_t)((uintptr_t)src & 15u);
            const uint32_t body = (head + nbytes) & ~15u;
            uint8_t *sb = reinterpret_cast<uint8_t *>(m.bytes + buf * SEL_STAGE_WORDS);
            if (tid == 0) {
                if (body) {
                    mbar_expect_tx(&s_bar[buf], body);
                    bulk_g2s(sb, src - head, body, &s_bar[buf]);
                } else {
                    mbar_expect_tx(&s_bar[buf], 0);
                }
            }
            for (uint32_t i = body + tid; i < head + nbytes + 8; i += SEL_THREADS)
                sb[i] = i < head + nbytes ? __ldg(src - head + i) : (uint8_t)0;
        };
        issue_stage(0, 0);
        uint32_t chunk_idx = 0;
        for (uint64_t c0 = 0; c0 < n; c0 += SEL_CHUNK, ++chunk_idx) {
            const uint32_t ch = (uint32_t)min((uint64_t)SEL_CHUNK, n - c0);
            const uint32_t buf = chunk_idx & 1u;
            if (c0 + SEL_CHUNK < n) issue_stage(c0 + SEL_CHUNK, buf ^ 1u);  // previous user of that buffer finished last iteration
            const uint32_t head = (uint32_t)((uintptr_t)(seq + c0) & 15u);
            const uint32_t *stage = m.bytes + buf * SEL_STAGE_WORDS;
            if (buf == 0) { mbar_wait(&s_bar[0], par0); par0 ^= 1u; }
            else          { mbar_wait(&s_bar[1], par1); par1 ^= 1u; }
            // make room: candidates after this chunk must fit
            uint32_t cnt = m.misc[0];
            __syncthreads();
            if (cnt + ch > cap) {
                limit = prune_to_s<SEL_THREADS>(m, cnt, s);
                if (tid == 0) m.misc[0] = s;
                __syncthreads();
            }
            // phase 1: block pre-mix of every position that some k-mer of the chunk uses
            const uint32_t npos = nb ? ch + 4 * (nb - 1) : 0;
            for (uint32_t p = tid; p < npos; p += SEL_THREADS) m.kv[p] = mm3_kmix(smem_window(stage, head + p));
            __syncthreads();
            // phase 2: one k-mer per thread.  Until the first prune every hash is a candidate and
            // its slot is known (base + position): no ballot / shared-memory atomic is needed.
            const bool unfiltered = limit == (1ull << 32);
            const uint32_t base_cnt = m.misc[0];
            for (uint32_t i0 = 0; i0 < ch; i0 += SEL_THREADS) {
                const uint32_t i = i0 + tid;
                bool take = false;
                uint32_t h = 0;
                if (i < ch) {
                    for (uint32_t j = 0; j < nb; ++j) h = mm3_round(h, m.kv[i + 4 * j]);
                    if (tail) h ^= mm3_kmix(smem_window(stage, head + i + 4 * nb) & tailmask);
                    h ^= k;
                    h = mm3_fmix(h);
                    take = (uint64_t)h < limit;
                    if (c0 + i == 0) h_first = h;  // thread 0 only
                }
                if (unfiltered) {
                    if (i < ch) m.cand[base_cnt + i] = h;
                } else {
                    const uint32_t b = __ballot_sync(0xffffffffu, take);
                    const uint32_t lane = tid & 31u;
                    uint32_t base = 0;
                    if (lane == 0 && b) base = atomicAdd(&m.misc[0], __popc(b));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    if (take) m.cand[base + __popc(b & ((1u << lane) - 1u))] = h;
                }
                if (s == 1 && i < ch && c0 + i > 0) atomicMin(&m.misc[5], h);
            }
            __syncthreads();
            if (unfiltered && tid == 0) m.misc[0] = base_cnt + ch;
            __syncthreads();
        }

        uint32_t cnt = m.misc[0];
        __syncthreads();
        if (!final_bucket_sort<SEL_THREADS>(m, cnt, s, dst)) {
            if (cnt > s) prune_to_s<SEL_THREADS>(m, cnt, s);
            for (uint32_t i = s + tid; i < P; i += SEL_THREADS) m.cand[i] = 0xffffffffu;
            __syncthreads();
            bitonic_sort<SEL_THREADS>(m.cand, P);
            for (uint32_t i = tid; i < s; i += SEL_THREADS) dst[i] = m.cand[i];
        }
        // fused all-gather: replicate the finished row into the gathered buffer of every rank
        if (extra.n > 0) {
            __syncthreads();
            for (int pr = 0; pr < extra.n; ++pr) {
                uint32_t *peer = extra.ptr[pr] + row * row_stride;
                if (peer == dst) continue;
                for (uint32_t i = tid; i < s; i += SEL_THREADS) peer[i] = dst[i];
            }
        }
        if (tid == 0) {
            int32_t st = PG_ITEM_OK;
            // s == 1: mash.go:96-98 indexes Sketches[-1] as soon as a later hash is
            // strictly below Sketches[0]
            if (s == 1 && m.misc[5] < h_first) st = PG_ITEM_PANIC;
            if (status) status[row] = st;
            if (count) count[row] = s;
        }
        __syncthreads();
    }
}

// ---- K2w: the select regime with the register-ring walk of K1 -----------------------------------
// Same CTA-per-read streaming, candidate buffer, prune and final stage as sketch_select_kernel, but
// the hashing of a chunk is K1's walk: thread t walks SELW_SEG consecutive k-mer positions of the
// staged chunk with the block pre-mixes in a register ring (kmer_walk.cuh), so a k-mer costs its
// body chain + fmix instead of k/4 shared-memory loads plus a loop, and no barrier separates a
// pre-mix phase from a hash phase.  Lanes read the staged bytes 20 bytes (5 words) apart, which
// is bank-conflict free.  While no prune has happened every hash is a candidate: full chunks store
// them transposed (k-mer j of thread t at [j][t]: conflict-free, order is irrelevant for a
// multiset), a partial last chunk stores them positionally; afterwards the walk itself tests each hash
// against the admission limit and appends the few that pass (one shared-memory atomic each) --
// for long sequences almost nothing passes, so the steady state is pure hashing.
// Half the instructions of the generic kernel (ncu: 0.74 G vs 1.46 G warp instructions on 20 k
// cfg3 reads); 256 threads x 3 CTAs per SM keep the issue slots busy.
constexpr int SELW_THREADS = 256;
constexpr int SELW_SEG = 20;  // bytes between the segments of adjacent lanes = 5 words: conflict-free smem reads
constexpr int SELW_CHUNK = SELW_THREADS * SELW_SEG;                      // 5120 k-mer positions
constexpr int SELW_ROOM = 8192;                                          // candidate room beyond s
constexpr int SELW_STAGE_WORDS = (15 + SELW_CHUNK + 32 + 48 + 15) / 16 * 4;  // head + chunk + k + over-read pad

#define PG_EMIT_ADMIT(R_, H_)                                              \
    if ((H_) < limit32) {                                                  \
        m.cand[cnt + atomicAdd(chunk_ctr, 1u)] = (H_);                     \
        if (s == 1) atomicMin(&m.misc[5], (H_));                           \
    }
// unfiltered, full chunk: k-mer i + r of this thread -> row i + r of a [SELW_SEG][SELW_THREADS] tile
#define PG_EMIT_TRANSPOSED(R_, H_) my_out[(i + (R_)) * SELW_THREADS] = (H_)
// unfiltered, partial chunk: positional (lane stride SELW_SEG words: 4-way conflicts, last chunk only)
#define PG_EMIT_APPEND(R_, H_) my_pos[i + (R_)] = (H_)

template <int K>
__global__ void __launch_bounds__(SELW_THREADS, 3)
sketch_select_walk_kernel(const uint8_t *__restrict__ bases, const uint64_t *__restrict__ offsets,
                          uint32_t uniform_len, uint64_t n_reads, uint32_t s, uint32_t P, uint32_t cap,
                          uint32_t *__restrict__ out, uint64_t row_stride, uint32_t *__restrict__ count,
                          int32_t *__restrict__ status, const SketchDst extra, uint32_t lut_stride,
                          const uint64_t *__restrict__ slice_beg, const uint32_t *__restrict__ slice_n,
                          unsigned long long *__restrict__ next_row, const uint32_t *__restrict__ row_list,
                          const uint32_t *__restrict__ n_list) {
    constexpr int NB = K / 4;
    constexpr int TAIL = K % 4;
    constexpr uint32_t TAILMASK = TAIL == 1 ? 0xffu : TAIL == 2 ? 0xffffu : 0xffffffu;
    constexpr bool LUT = TAIL == 1;
    constexpr uint32_t k = K;
    static_assert(NB >= 1 && K <= 32, "walk path: 4 <= k <= 32");
    static_assert(SELW_SEG % 4 == 0, "a segment is a whole number of word steps");

    extern __shared__ __align__(16) uint32_t smem_w[];
    SelSmem m;
    m.cand = smem_w;
    m.keep = m.cand + cap;
    m.kv = nullptr;
    m.bytes = m.keep + ((s + 3u) & ~3u) + 4u;  // 16-byte granules keep the TMA stage buffers aligned
    m.hist = m.bytes + 2 * SELW_STAGE_WORDS;
    m.misc = m.hist + SEL_NBK + 1;
    m.tmpcap = (uint32_t)(m.hist - m.keep);

    __shared__ __align__(16) uint32_t s_lut[LUT ? 256 : 4];
    __shared__ __align__(8) uint64_t s_bar[3];
    uint32_t par0 = 0u, par1 = 0u;
    const uint32_t tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        mbar_init(&s_bar[2], 1);
        fence_mbar_init();
        if (LUT) {
            mbar_expect_tx(&s_bar[2], 1024u);
            bulk_g2s(s_lut, &g_kmix_byte, 1024u, &s_bar[2]);
        }
    }
    __syncthreads();
    if (LUT) mbar_wait(&s_bar[2], 0);
    const uint32_t lut_base = smem_u32(s_lut);

    // rows are handed out dynamically (reads / slices differ in length): the grid is exactly the
    // resident CTA count, every CTA takes the next row when it is done
    __shared__ unsigned long long s_row;
    for (;;) {
        if (tid == 0) s_row = atomicAdd(next_row, 1ull);
        __syncthreads();
        uint64_t row = s_row;
        __syncthreads();
        if (row_list) {  // only the listed rows (the threshold path's retries); the list length lives on the device
            if (row >= *n_list) break;
            row = row_list[row];
        }
        if (row >= n_reads) break;
        uint64_t beg, n;
        if (slice_beg) {  // `row` is a slice of a long sequence: k-mer positions [beg, beg + n)
            beg = slice_beg[row];
            n = slice_n[row];
        } else {
            uint64_t len;
            if (offsets) {
                beg = offsets[row];
                len = offsets[row + 1] - beg;
            } else {
                beg = row * (uint64_t)uniform_len;
                len = uniform_len;
            }
            n = len > k ? len - k : 0;
        }
        if (n < s || n == 0) continue;  // fill regime: other kernel
        const uint8_t *seq = bases + beg;
        uint32_t *dst = out + row * row_stride;
        if (s == 0) {  // mash.go:96 reads Sketches[-1] on the first k-mer
            if (tid == 0) {
                if (status) status[row] = PG_ITEM_PANIC;
                if (count) count[row] = 0;
            }
            continue;
        }
        if (tid == 0) { m.misc[5] = 0xffffffffu; m.misc[8] = 0; m.misc[9] = 0; m.misc[10] = 0; }
        __syncthreads();
        uint64_t limit = 1ull << 32;  // admit h < limit
        uint32_t h_first = 0;
        uint32_t cnt = 0;  // candidates held (uniform across the CTA)

        // A chunk that is not the last of its row may over-read up to 15 bytes (they belong to the
        // same sequence): the whole stage is then one TMA copy.  Otherwise the 16-byte aligned body
        // comes by TMA and the tail by plain loads (+ a barrier before use).
        auto tail_by_tma = [&](uint64_t c0, uint32_t ch) { return n - (c0 + ch) >= 16; };
        auto issue_stage = [&](uint64_t c0, uint32_t buf) {
            const uint32_t ch = (uint32_t)min((uint64_t)SELW_CHUNK, n - c0);
            const uint32_t nbytes = ch + k;
            const uint8_t *src = seq + c0;
            const uint32_t head = (uint32_t)((uintptr_t)src & 15u);
            const bool all_tma = tail_by_tma(c0, ch);
            const uint32_t body = all_tma ? (head + nbytes + 15u) & ~15u : (head + nbytes) & ~15u;
            uint8_t *sb8 = reinterpret_cast<uint8_t *>(m.bytes + buf * SELW_STAGE_WORDS);
            if (tid == 0) {
                if (body) {
                    mbar_expect_tx(&s_bar[buf], body);
                    bulk_g2s(sb8, src - head, body, &s_bar[buf]);
                } else {
                    mbar_expect_tx(&s_bar[buf], 0);
                }
            }
            if (!all_tma)
                for (uint32_t i = body + tid; i < head + nbytes + 32; i += SELW_THREADS)  // tail + over-read pad
                    sb8[i] = i < head + nbytes ? __ldg(src - head + i) : (uint8_t)0;
        };
        issue_stage(0, 0);
        uint32_t chunk_idx = 0;
        for (uint64_t c0 = 0; c0 < n; c0 += SELW_CHUNK, ++chunk_idx) {
            const uint32_t ch = (uint32_t)min((uint64_t)SELW_CHUNK, n - c0);
            const uint32_t buf = chunk_idx & 1u;
            if (c0 + SELW_CHUNK < n) issue_stage(c0 + SELW_CHUNK, buf ^ 1u);  // its last readers passed the barrier below
            const uint32_t head = (uint32_t)((uintptr_t)(seq + c0) & 15u);
            const uint8_t *stage = reinterpret_cast<const uint8_t *>(m.bytes + buf * SELW_STAGE_WORDS);
            if (buf == 0) { mbar_wait(&s_bar[0], par0); par0 ^= 1u; }
            else          { mbar_wait(&s_bar[1], par1); par1 ^= 1u; }
            if (!tail_by_tma(c0, ch)) __syncthreads();  // plain-store part of this stage
            if (cnt + ch > cap) {  // worst case every hash of the chunk is admitted
                limit = prune_to_s<SELW_THREADS>(m, cnt, s);
                cnt = s;
            }
            uint32_t *chunk_ctr = &m.misc[8 + chunk_idx % 3u];  // admitted by this chunk (zeroed two chunks ago)
            const bool unfiltered = limit == (1ull << 32);
            const bool full_chunk = ch == SELW_CHUNK;
            const uint32_t limit32 = (uint32_t)limit;

            // the walk: my segment = positions [seg, seg + nk) of the chunk
            const uint32_t seg = tid * SELW_SEG;
            if (seg < ch) {
                const uint32_t nk = min((uint32_t)SELW_SEG, ch - seg);
                const uint32_t b0 = head + seg;
                const uint32_t *sw = reinterpret_cast<const uint32_t *>(stage) + (b0 >> 2);
                const uint8_t *sb = stage + b0 + 4 * NB;
                const uint32_t sh = (b0 & 3u) * 8u;
                uint32_t *my_out = m.cand + cnt + tid;  // transposed target (full chunk, unfiltered)
                uint32_t *my_pos = m.cand + cnt + seg;  // positional target (partial chunk, unfiltered)
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
    // a full segment is SELW_SEG / 4 word steps with no bounds tests; the last segment of a chunk is checked
#define PG_WALK_SEGMENT(EMIT)                                                          \
    if (nk == SELW_SEG) {                                                              \
        _Pragma("unroll") for (int q = 0; q < SELW_SEG / 4; ++q) PG_KMER_STEP(q % NB, false, EMIT) \
    } else {                                                                           \
        _Pragma("unroll") for (int q = 0; q < SELW_SEG / 4; ++q) {                     \
            if (i < nk) PG_KMER_STEP(q % NB, true, EMIT)                               \
        }                                                                              \
    }
                if (!unfiltered) PG_WALK_SEGMENT(PG_EMIT_ADMIT)
                else if (full_chunk) PG_WALK_SEGMENT(PG_EMIT_TRANSPOSED)
                else PG_WALK_SEGMENT(PG_EMIT_APPEND)
#undef PG_WALK_SEGMENT
            }
            __syncthreads();  // the one barrier per chunk: hashes / admissions of the chunk are in place
            if (unfiltered) {  // position 0 of the chunk is index 0 in both layouts
                if (c0 == 0 && tid == 0) h_first = m.cand[cnt];
                if (s == 1) {  // mash.go:96-98: a later hash strictly below Sketches[0] indexes Sketches[-1]
                    for (uint32_t q = tid; q < ch; q += SELW_THREADS)
                        if (c0 + q > 0) atomicMin(&m.misc[5], m.cand[cnt + q]);
                }
                cnt += ch;
            } else {
                cnt += *chunk_ctr;
            }
            if (tid == 0) m.misc[8 + (chunk_idx + 2) % 3u] = 0;  // next use: chunk_idx + 2, after the next barrier
        }
        __syncthreads();
        if (!final_bucket_sort<SELW_THREADS>(m, cnt, s, dst)) {
            if (cnt > s) prune_to_s<SELW_THREADS>(m, cnt, s);
            for (uint32_t i = s + tid; i < P; i += SELW_THREADS) m.cand[i] = 0xffffffffu;
            __syncthreads();
            bitonic_sort<SELW_THREADS>(m.cand, P);
            for (uint32_t i = tid; i < s; i += SELW_THREADS) dst[i] = m.cand[i];
        }
        if (extra.n > 0) {  // fused all-gather: replicate the finished row into every rank's buffer
            __syncthreads();
#pragma unroll
            for (int pr = 0; pr < PG_MAX_PEERS; ++pr) {  // static indices: the struct stays in parameter space
                if (pr >= extra.n) continue;
                uint32_t *peer = extra.ptr[pr] + row * row_stride;
                if (peer == dst) continue;
                for (uint32_t i = tid; i < s; i += SELW_THREADS) peer[i] = dst[i];
            }
        }
        if (tid == 0) {
            int32_t st = PG_ITEM_OK;
            if (s == 1 && m.misc[5] < h_first) st = PG_ITEM_PANIC;
            if (status) status[row] = st;
            if (count) count[row] = s;
        }
        __syncthreads();
    }
}
#undef PG_EMIT_ADMIT
#undef PG_EMIT_TRANSPOSED
#undef PG_EMIT_APPEND

// ---- merge of partial sketches (long sequences cut into slices) ---------------------------------
// The bottom-s multiset of a sequence is the bottom-s multiset of the union of the bottom-s multisets
// of its slices.  One CTA per row streams the row's partial sketches (slices are consecutive in
// `part`, s ascending words each) through the same candidate buffer / admission limit / prune /
// final stage as the hashing kernels.
constexpr int SELM_THREADS = 256;
constexpr int SELM_CHUNK = 4096;

__global__ void __launch_bounds__(SELM_THREADS)
select_merge_kernel(const uint32_t *__restrict__ part, const uint32_t *__restrict__ row_slice0, uint64_t n_rows,
                    uint32_t s, uint32_t P, uint32_t cap, uint32_t *__restrict__ out, uint64_t row_stride,
                    uint32_t *__restrict__ count, int32_t *__restrict__ status) {
    extern __shared__ __align__(16) uint32_t smem_w[];
    SelSmem m;
    m.cand = smem_w;
    m.keep = m.cand + cap;
    m.kv = nullptr;
    m.bytes = nullptr;
    m.hist = m.keep + s + SEL_NBK + 64;  // scratch of the final stage: s + ties + one cursor per bucket
    m.misc = m.hist + SEL_NBK + 1;
    m.tmpcap = (uint32_t)(m.hist - m.keep);
    const uint32_t tid = threadIdx.x;
    for (uint64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const uint32_t sl0 = row_slice0[row], sl1 = row_slice0[row + 1];
        if (sl1 == sl0) continue;  // not a select-regime row
        uint32_t *dst = out + row * row_stride;
        const uint32_t *src = part + (uint64_t)sl0 * s;
        if (sl1 - sl0 == 1) {  // a single slice is already the answer
            for (uint32_t i = tid; i < s; i += SELM_THREADS) dst[i] = src[i];
        } else {
            const uint64_t total = (uint64_t)(sl1 - sl0) * s;
            if (tid == 0) m.misc[0] = 0;
            __syncthreads();
            uint64_t limit = 1ull << 32;
            for (uint64_t c0 = 0; c0 < total; c0 += SELM_CHUNK) {
                const uint32_t ch = (uint32_t)min((uint64_t)SELM_CHUNK, total - c0);
                uint32_t cnt = m.misc[0];
                __syncthreads();
                if (cnt + ch > cap) {
                    limit = prune_to_s<SELM_THREADS>(m, cnt, s);
                    if (tid == 0) m.misc[0] = s;
                    cnt = s;
                    __syncthreads();
                }
                if (limit == (1ull << 32)) {
                    for (uint32_t q = tid; q < ch; q += SELM_THREADS) m.cand[cnt + q] = __ldg(src + c0 + q);
                    __syncthreads();
                    if (tid == 0) m.misc[0] = cnt + ch;
                } else {
                    const uint32_t limit32 = (uint32_t)limit;
                    for (uint32_t q = tid; q < ch; q += SELM_THREADS) {
                        const uint32_t h = __ldg(src + c0 + q);
                        if (h < limit32) m.cand[atomicAdd(&m.misc[0], 1u)] = h;
                    }
                }
                __syncthreads();
            }
            const uint32_t cnt = m.misc[0];
            __syncthreads();
            if (!final_bucket_sort<SELM_THREADS>(m, cnt, s, dst)) {
                if (cnt > s) prune_to_s<SELM_THREADS>(m, cnt, s);
                for (uint32_t i = s + tid; i < P; i += SELM_THREADS) m.cand[i] = 0xffffffffu;
                __syncthreads();
                bitonic_sort<SELM_THREADS>(m.cand, P);
                for (uint32_t i = tid; i < s; i += SELM_THREADS) dst[i] = m.cand[i];
            }
        }
        if (tid == 0) {
            if (status) status[row] = PG_ITEM_OK;
            if (count) count[row] = s;
        }
        __syncthreads();
    }
}

// ---- K2t: the select regime by a value threshold -------------------------------------------------
// The bottom-s multiset of n hashes is contained in {h < T} as soon as that set has >= s members.  For
// hash values that behave like uniform draws (murmur3 of distinct k-mers) T = mu/n * 2^32 with
// mu = s + 6 sqrt(s) + 48 admits mu hashes on average and fewer than s only 6 standard deviations below
// the mean -- and whether it did is CHECKED, never assumed: a row whose admitted count is < s (few
// distinct k-mers) or exceeds its buffer (heavy duplication below T) is redone by the exact streaming
// kernel above (retry list built on the device, no host round trip).  So:
//   A. sketch_thresh_walk_kernel<K, RARE>: one WARP per work item (<= 8 chunks of 32 x SEG
//      positions of one row, SeltGeom<K>; long sequences become many items, so there is no host-side
//      slicing and no merge pass).  Chunks arrive by double-buffered 1-D TMA bulk copies; lane l walks SEG
//      consecutive k-mers with the register ring of kmer_walk.cuh (one ring prologue per SEG k-mers
//      instead of per 20) and stores every hash into its private strip column, whose fill count advances
//      only for hashes <= T -- a store, a compare and an add, branch-free: no vote, no atomic, no barrier.
//      After the chunk the strips are compacted into the row's candidate list in global memory (one
//      global atomic per warp-chunk reserves the space; dense run of stores through the dead stage buffer).
//   B. sketch_thresh_select_kernel<U>: one CTA per row, counting sort of the ~mu candidates over 2048
//      value buckets + exact rank inside each bucket (ties counted) -> ascending bottom-s, stored to
//      every destination.
// Extra HBM traffic: mu words per row written and read once (cfg3: 2 x 1 GB next to 1.8 GB algorithmic).
// Positions per lane per chunk: 4 x an ODD number of word steps (lanes read their staged words an odd number
// of words apart: bank-conflict free) that is a multiple of NB = K / 4 where NB is odd, so that a full
// segment is whole groups of the NB-step loop body and never enters the bounds-checked tail; for even NB one
// checked step remains.
template <int K>
struct SeltGeom {
    static constexpr int NB = K / 4;
    static constexpr int STEPS = NB == 2 ? 17 : NB == 3 ? 21 : NB == 4 ? 17 : NB == 5 ? 15 : 21;  // NB >= 6: whole groups of 3 steps
    static constexpr int SEG = 4 * STEPS;      // 60 .. 84 k-mer positions
    static constexpr int CHUNK = 32 * SEG;     // per warp chunk
    static constexpr int STAGE = (15 + CHUNK + 32 + 48 + 15 + 255) / 256 * 256;  // head + chunk + k + over-read pad; also the dense flush buffer
    static_assert(STEPS % 2 == 1 && (NB % 2 == 0 || STEPS % NB == 0), "segment geometry");
};
constexpr int SELT_ITEM_CHUNKS = 8;
// rolled body (groups of 3 steps, then a ring rotation) from NB = 6 (k >= 24) on; k = 21 (NB = 5) keeps the unrolled 5-step
// body: 1.38 vs 1.43 ms (profiles/r02_k2_tuning.md)
#define SELT_ROLLED_DEFAULT(K_) ((K_) / 4 >= 6)
constexpr int SELT_SEL_THREADS = 256;

__host__ __device__ __forceinline__ uint32_t selt_threshold_m1(uint64_t n, uint32_t mu) {
    if ((uint64_t)mu >= n) return 0xffffffffu;  // every hash is a candidate
    const uint64_t t = ((uint64_t)mu << 32) / n;
    return t ? (uint32_t)(t - 1) : 0u;
}

__device__ __forceinline__ void strip_put(uint32_t saddr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory");
}
__device__ __forceinline__ void strip_advance_if_le(uint32_t &saddr, uint32_t h, uint32_t t) {
    asm("{\n\t.reg .pred p;\n\tsetp.le.u32 p, %1, %2;\n\t@p add.u32 %0, %0, 128;\n\t}" : "+r"(saddr) : "r"(h), "r"(t));
}

// branch-free: the hash is always stored at the lane's next strip slot and the slot is only kept when the
// hash is admitted (nvcc turned the `if` into a BSSY / BRA / BSYNC region per k-mer: 11 instructions and a
// fetch redirect instead of 4 straight-line ones).  c <= number of k-mers walked so far < rows of the strip.
// The slot is a running shared-space address: a store, a compare and a predicated add per k-mer (indexing
// my_strip[c * 32] cost a shift, an or and an add more, ncu source page).
#define PG_EMIT_STRIP(R_, H_) \
    { strip_put(sa, (H_)); strip_advance_if_le(sa, (H_), tm1); }
// RARE variant (expected admissions per warp step << 1, e.g. genomes: T/2^32 ~ s/n ~ 3e-4): one test of the
// minimum of the step's four hashes and a branch that is almost never taken, instead of four predicated
// compare/store/add triples.  Only valid for unchecked steps (all four hashes of the step exist).
#define PG_EMIT_STRIP_RARE(R_, H_)                                                       \
    if ((R_) == 3) {                                                                     \
        if (min(min(h[0], h[1]), min(h[2], h[3])) <= tm1) {                              \
            _Pragma("unroll") for (int rr = 0; rr < 4; ++rr)                             \
                if (h[rr] <= tm1) { strip_put(sa, h[rr]); sa += 128u; }                  \
        }                                                                                \
    }

template <int K, bool RARE>
__global__ void __launch_bounds__(32)
sketch_thresh_walk_kernel(const uint8_t *__restrict__ bases, const uint64_t *__restrict__ offsets, uint32_t uniform_len,
                          uint64_t row0, uint64_t n_rows, uint32_t items_per_row, uint32_t s, uint32_t mu, uint32_t cap,
                          uint32_t *__restrict__ gcand, uint32_t *__restrict__ gcnt, uint32_t lut_stride, uint32_t tm1_uniform) {
    constexpr int NB = K / 4;
    constexpr int TAIL = K % 4;
    constexpr uint32_t TAILMASK = TAIL == 1 ? 0xffu : TAIL == 2 ? 0xffffu : 0xffffffu;
    constexpr bool LUT = TAIL == 1;
    constexpr uint32_t k = K;
    constexpr bool ROLLED = SELT_ROLLED_DEFAULT(K);
    static_assert(NB >= 1 && K <= 32, "walk path: 4 <= k <= 32");
    constexpr int SELT_SEG = SeltGeom<K>::SEG, SELT_CHUNK = SeltGeom<K>::CHUNK, SELT_STAGE_BYTES = SeltGeom<K>::STAGE;

    extern __shared__ __align__(128) uint8_t smem[];  // 2 stage buffers | strip [SELT_SEG][32]
    __shared__ __align__(16) uint32_t s_lut[LUT ? 256 : 4];
    __shared__ __align__(8) uint64_t s_bar[3];
    const uint32_t lane = threadIdx.x;
    const uint32_t item = blockIdx.x;                   // 32-bit: a 64-bit divide costs ~120 instructions per CTA
    const uint64_t lrow = item / items_per_row;  // row within this launch group
    if (lrow >= n_rows) return;
    const uint64_t row = row0 + lrow;
    uint64_t beg, len;
    if (offsets) {
        beg = offsets[row];
        len = offsets[row + 1] - beg;
    } else {
        beg = row * (uint64_t)uniform_len;
        len = uniform_len;
    }
    const uint64_t n = len > k ? len - k : 0;
    if (n < s || n == 0) return;  // fill regime: other kernel
    const uint64_t p0 = (uint64_t)(item % items_per_row) * (uint64_t)(SELT_ITEM_CHUNKS * SELT_CHUNK);
    if (p0 >= n) return;
    const uint64_t p1 = min(n, p0 + (uint64_t)(SELT_ITEM_CHUNKS * SELT_CHUNK));
    const uint8_t *seq = bases + beg;
    const uint32_t tm1 = offsets ? selt_threshold_m1(n, mu) : tm1_uniform;  // fixed-length reads: computed once on the host
    uint32_t *my_cand = gcand + lrow * (uint64_t)cap;
    uint32_t *strip = reinterpret_cast<uint32_t *>(smem + 2 * SELT_STAGE_BYTES);
    uint32_t *my_strip = strip + lane;
    const uint32_t sa0 = smem_u32(my_strip);

    if (lane == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        mbar_init(&s_bar[2], 1);
        fence_mbar_init();
        if (LUT) {
            mbar_expect_tx(&s_bar[2], 1024u);
            bulk_g2s(s_lut, &g_kmix_byte, 1024u, &s_bar[2]);
        }
    }
    __syncwarp();
    const uint32_t lut_base = smem_u32(s_lut);

    // A chunk that is not the last of its row may over-read up to 15 bytes (they belong to the same
    // sequence): the whole stage is then one TMA copy.  Otherwise the 16-byte aligned body comes by
    // TMA and the tail by plain loads.
    auto tail_by_tma = [&](uint64_t c0, uint32_t ch) { return n - (c0 + ch) >= 16; };
    auto issue_stage = [&](uint64_t c0, uint32_t buf) {
        const uint32_t ch = (uint32_t)min((uint64_t)SELT_CHUNK, p1 - c0);
        const uint32_t nbytes = ch + k;
        const uint8_t *src = seq + c0;
        const uint32_t head = (uint32_t)((uintptr_t)src & 15u);
        const bool all_tma = tail_by_tma(c0, ch);
        const uint32_t body = all_tma ? (head + nbytes + 15u) & ~15u : (head + nbytes) & ~15u;
        uint8_t *sb8 = smem + buf * SELT_STAGE_BYTES;
        if (lane == 0) {
            mbar_expect_tx(&s_bar[buf], body);
            if (body) bulk_g2s(sb8, src - head, body, &s_bar[buf]);
        }
        if (!all_tma)
            for (uint32_t i = body + lane; i < head + nbytes + 32; i += 32)  // tail + over-read pad
                sb8[i] = i < head + nbytes ? __ldg(src - head + i) : (uint8_t)0;
    };
    issue_stage(p0, 0);
    if (LUT) mbar_wait(&s_bar[2], 0);
    uint32_t par0 = 0u, par1 = 0u, chunk_idx = 0;
    for (uint64_t c0 = p0; c0 < p1; c0 += SELT_CHUNK, ++chunk_idx) {
        const uint32_t ch = (uint32_t)min((uint64_t)SELT_CHUNK, p1 - c0);
        const uint32_t buf = chunk_idx & 1u;
        __syncwarp();  // every lane is done with the other buffer (chunk c-1) before it is refilled
        if (c0 + SELT_CHUNK < p1) issue_stage(c0 + SELT_CHUNK, buf ^ 1u);
        const uint32_t head = (uint32_t)((uintptr_t)(seq + c0) & 15u);
        const uint8_t *stage = smem + buf * SELT_STAGE_BYTES;
        if (buf == 0) { mbar_wait(&s_bar[0], par0); par0 ^= 1u; }
        else          { mbar_wait(&s_bar[1], par1); par1 ^= 1u; }
        if (!tail_by_tma(c0, ch)) __syncwarp();  // plain-store part of this stage

        uint32_t sa = sa0;  // shared address of the lane's next strip slot: (sa - sa0) / 128 hashes admitted in this chunk
        // A full chunk gives every lane SELT_SEG positions.  A shorter (last) chunk is spread over all lanes
        // instead of leaving the upper lanes idle while the lower ones walk full segments: an odd number
        // of word steps per lane keeps the lanes' staged words in different banks.
        uint32_t seg_len = SELT_SEG;
        if (ch != SELT_CHUNK) {
            uint32_t steps = (ch + 127u) >> 7;  // ceil(ch / 32 lanes / 4 positions per step)
            steps |= 1u;
            seg_len = 4u * steps;               // <= SELT_SEG because ch < SELT_CHUNK
        }
        const uint32_t seg = lane * seg_len;
        if (seg < ch) {
            const uint32_t nk = min(seg_len, ch - seg);
            const uint32_t b0 = head + seg;
            const uint32_t *sw = reinterpret_cast<const uint32_t *>(stage) + (b0 >> 2);
            const uint8_t *sb = stage + b0 + 4 * NB;
            const uint32_t sh = (b0 & 3u) * 8u;
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
            // whole groups of NB word steps without bounds tests, then < NB checked steps: the loop body is
            // NB steps of code (it stays in the instruction cache) instead of a fully unrolled segment
            uint32_t i = 0;
            if (ROLLED) {  // groups of 3 steps of code with the ring rotated after each group: the body fits the instruction cache
                const uint32_t n_full = nk & ~3u;
                const uint32_t n_grp = (nk / 12u) * 12u;
                if (RARE) {
#pragma unroll 1
                    while (i < n_grp) {
                        PG_KMER_STEP(0, false, PG_EMIT_STRIP_RARE)
                        PG_KMER_STEP(1, false, PG_EMIT_STRIP_RARE)
                        PG_KMER_STEP(2, false, PG_EMIT_STRIP_RARE)
                        PG_RING_ROTATE(3)
                    }
                } else {
#pragma unroll 1
                    while (i < n_grp) {
                        PG_KMER_STEP(0, false, PG_EMIT_STRIP)
                        PG_KMER_STEP(1, false, PG_EMIT_STRIP)
                        PG_KMER_STEP(2, false, PG_EMIT_STRIP)
                        PG_RING_ROTATE(3)
                    }
                }
#pragma unroll 1
                while (i < n_full) PG_KMER_STEP_ROLLED(false, PG_EMIT_STRIP)  // < 3 whole steps left: one step of code, ring shifted per step
                if (i < nk) PG_KMER_STEP_ROLLED(true, PG_EMIT_STRIP)
            } else {
                const uint32_t n_main = (nk / (4 * NB)) * (4 * NB);
                if (RARE) {
#pragma unroll 1
                    while (i < n_main) {
#pragma unroll
                        for (int u = 0; u < NB; ++u) PG_KMER_STEP(u, false, PG_EMIT_STRIP_RARE)
                    }
                } else {
#pragma unroll 1
                    while (i < n_main) {
#pragma unroll
                        for (int u = 0; u < NB; ++u) PG_KMER_STEP(u, false, PG_EMIT_STRIP)
                    }
                }
#pragma unroll
                for (int u = 0; u < NB; ++u) {
                    if (i < nk) PG_KMER_STEP(u, true, PG_EMIT_STRIP)
                }
            }
        }
        // flush: compact the strip columns into the row's candidate list (order is irrelevant: a multiset)
        const uint32_t c = (sa - sa0) >> 7;
        uint32_t incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d) incl += y;
        }
        const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
        if (tot) {
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(&gcnt[lrow], tot);
            base = __shfl_sync(0xffffffffu, base, 0);
            if ((uint64_t)base + tot <= cap) {  // otherwise the count alone tells stage B that the row overflowed
                if (tot <= SELT_STAGE_BYTES / 4) {
                    // usual case: the chunk's stage buffer is dead by now -- gather the strip columns into it (lane l's
                    // entries behind those of the lanes below it), then copy the dense list out with coalesced stores
                    uint32_t *dense = reinterpret_cast<uint32_t *>(smem + buf * SELT_STAGE_BYTES);
                    const uint32_t excl = incl - c;
                    __syncwarp();  // every lane is done reading the staged bytes
                    for (uint32_t j = 0; j < c; ++j) dense[excl + j] = my_strip[j * 32u];
                    __syncwarp();
                    for (uint32_t i = lane; i < tot; i += 32) my_cand[base + i] = dense[i];
                } else {  // many admissions (T close to 2^32): compact strip row by strip row with ballots
                    const uint32_t maxc = __reduce_max_sync(0xffffffffu, c);
                    const uint32_t below = (1u << lane) - 1u;
                    uint32_t off = base;
                    for (uint32_t j = 0; j < maxc; ++j) {
                        const bool v = j < c;
                        const uint32_t b = __ballot_sync(0xffffffffu, v);
                        if (v) my_cand[off + __popc(b & below)] = my_strip[j * 32u];
                        off += __popc(b);
                    }
                }
            }
        }
    }
}
#undef PG_EMIT_STRIP
#undef PG_EMIT_STRIP_RARE

// Stage B: exact bottom-s of the admitted candidates of one row (cnt <= cap by construction).  A counting sort
// over 2048 value buckets scaled to T (about one candidate per bucket) with an exact rank inside the bucket;
// ties keep distinct slots through their index.  Rows whose count is < s or > cap, or whose values crowd into
// one bucket (degenerate distribution: ranking would be quadratic), go onto the retry list for the exact
// streaming kernel.  Shared memory is only the bucket-grouped copy (cap words) and the 2048 counters, so ~10
// rows are in flight per SM; the candidates themselves are read from global memory twice (second time from L2).
template <int U, bool MUL>  // MUL: scaled buckets (all 2048 in use whatever T is) or plain shift; U: candidates loaded per thread and batch: chosen so that a typical row is a whole number of batches
__global__ void __launch_bounds__(SELT_SEL_THREADS)
sketch_thresh_select_kernel(const uint64_t *__restrict__ offsets, uint32_t uniform_len, uint64_t row0, uint64_t n_rows, uint32_t k,
                            uint32_t s, uint32_t mu, uint32_t cap, const uint32_t *__restrict__ gcand,
                            const uint32_t *__restrict__ gcnt, uint32_t *__restrict__ out, uint64_t row_stride,
                            uint32_t *__restrict__ count, int32_t *__restrict__ status, const SketchDst extra,
                            uint32_t *__restrict__ retry_rows, uint32_t *__restrict__ n_retry, uint32_t tm1_uniform) {
    extern __shared__ __align__(16) uint32_t smem_w[];  // tmp[cap] | cur[SEL_NBK] | flag
    const uint32_t o_tmp = 0, o_cur = (cap + 3u) & ~3u, o_flag = o_cur + SEL_NBK;
    __shared__ uint32_t s_wtot[SELT_SEL_THREADS / 32];
    const uint32_t tid = threadIdx.x;
    for (uint64_t lrow = blockIdx.x; lrow < n_rows; lrow += gridDim.x) {
        const uint64_t row = row0 + lrow;
        uint64_t len;
        if (offsets) len = offsets[row + 1] - offsets[row];
        else len = uniform_len;
        const uint64_t n = len > k ? len - k : 0;
        if (n < s || n == 0) continue;  // fill regime: other kernel
        const uint32_t cnt = gcnt[lrow];
        if (cnt < s || cnt > cap) {  // the estimate did not hold for this row: exact streaming kernel redoes it
            if (tid == 0) retry_rows[atomicAdd(n_retry, 1u)] = (uint32_t)row;
            continue;
        }
        const uint32_t *src = gcand + lrow * (uint64_t)cap;
        uint32_t *dst = out + row * row_stride;
        asm volatile("" : "+l"(dst));  // keep the row pointer in registers: nvcc otherwise redoes the 64-bit multiply per store
        const uint32_t tm1 = offsets ? selt_threshold_m1(n, mu) : tm1_uniform;
        // shift: bucket(e) = e >> (bits(T) - 11), between 1024 and 2048 buckets in use.  MUL (rows whose T sits just above a
        // power of two, ragged batches): the 16 leading bits of e times 2048 * 2^16 / (T16 + 1) -- monotone, < 2048 for
        // e <= T, (nearly) all 2048 buckets in use; a shift, a 32-bit multiply and a shift (__umulhi measured slower)
        const uint32_t bits = 32u - __clz(tm1 | 1u);
        const uint32_t bshift = MUL ? (bits > 16u ? bits - 16u : 0u) : (bits > 11u ? bits - 11u : 0u);
        const uint32_t bscale = MUL ? ((uint32_t)SEL_NBK << 16) / ((tm1 >> bshift) + 1u) : 0u;
        auto bucket = [&](uint32_t e) -> uint32_t { return MUL ? ((e >> bshift) * bscale) >> 16 : e >> bshift; };
        for (uint32_t i = tid; i < SEL_NBK; i += SELT_SEL_THREADS) smem_w[o_cur + i] = 0;
        if (tid == 0) smem_w[o_flag] = 0;
        __syncthreads();
        // histogram; loads in batches of U per thread so that a batch is one global round trip
        for (uint32_t base = 0; base < cnt; base += U * SELT_SEL_THREADS) {
            uint32_t v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t i = base + u * SELT_SEL_THREADS + tid;
                v[u] = i < cnt ? __ldg(src + i) : 0u;
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (base + u * SELT_SEL_THREADS + tid < cnt) atomicAdd(&smem_w[o_cur + bucket(v[u])], 1u);
        }
        __syncthreads();
        {   // exclusive scan over the buckets: 8 per thread, warp scan, warp totals
            constexpr int PER = SEL_NBK / SELT_SEL_THREADS;
            uint32_t cb[PER], sum = 0, mx = 0;
#pragma unroll
            for (int j = 0; j < PER; ++j) { cb[j] = smem_w[o_cur + tid * PER + j]; sum += cb[j]; mx = max(mx, cb[j]); }
            uint32_t incl = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
                if ((int)(tid & 31u) >= d) incl += y;
            }
            if ((tid & 31u) == 31u) s_wtot[tid >> 5] = incl;
            mx = __reduce_max_sync(0xffffffffu, mx);
            if ((tid & 31u) == 0 && mx > 48u) atomicMax(&smem_w[o_flag], mx);
            __syncthreads();
            uint32_t run = incl - sum;
            for (uint32_t w = 0; w < (tid >> 5); ++w) run += s_wtot[w];
#pragma unroll
            for (int j = 0; j < PER; ++j) { smem_w[o_cur + tid * PER + j] = run; run += cb[j]; }
        }
        __syncthreads();
        if (smem_w[o_flag] != 0) {  // crowded bucket: degenerate values, the exact streaming kernel takes the row
            __syncthreads();
            if (tid == 0) retry_rows[atomicAdd(n_retry, 1u)] = (uint32_t)row;
            continue;
        }
        // scatter into bucket order (second read of the candidates: L2); cur[b] ends as the END of bucket b
        for (uint32_t base = 0; base < cnt; base += U * SELT_SEL_THREADS) {
            uint32_t v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t i = base + u * SELT_SEL_THREADS + tid;
                v[u] = i < cnt ? __ldg(src + i) : 0u;
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (base + u * SELT_SEL_THREADS + tid < cnt) smem_w[o_tmp + smem_fetch_inc(&smem_w[o_cur + bucket(v[u])])] = v[u];
        }
        __syncthreads();
        {   // rank inside the bucket, through explicit shared-space addresses (kept in registers across the loop)
            const uint32_t s_tmp = smem_u32(smem_w + o_tmp), s_cur = smem_u32(smem_w + o_cur);
#pragma unroll 2
            for (uint32_t p = tid; p < cnt; p += SELT_SEL_THREADS) {
                const uint32_t e = lds_u32(s_tmp + 4u * p), b = bucket(e);
                const uint32_t lo = b ? lds_u32(s_cur + 4u * b - 4u) : 0u;
                if (lo >= s) continue;  // the whole bucket lies beyond the s-th smallest
                uint32_t a = s_tmp + 4u * lo;
                const uint32_t a_hi = s_tmp + 4u * lds_u32(s_cur + 4u * b);
                uint32_t r = lo, m = 0;  // r: strictly smaller values in front; m: copies of e in the bucket (itself included)
#pragma unroll 1
                do {  // the bucket holds e itself: never empty
                    const uint32_t x = lds_u32(a);
                    a += 4u;
                    count_lt_eq(x, e, r, m);
                } while (a != a_hi);
                // every copy of a tied value writes the whole run r .. r + m - 1 (same words): no tie-break by index needed
                if (r < s) stg_u32(dst + r, e);
                if (m > 1) {
#pragma unroll 1
                    for (uint32_t t = 1; t < m; ++t)
                        if (r + t < s) stg_u32(dst + r + t, e);
                }
            }
        }
        if (extra.n > 0) {  // fused all-gather: replicate the finished row into every rank's buffer
            __syncthreads();
#pragma unroll
            for (int pr = 0; pr < PG_MAX_PEERS; ++pr) {
                if (pr >= extra.n) continue;
                uint32_t *peer = extra.ptr[pr] + row * row_stride;
                if (peer == dst) continue;
                for (uint32_t i = tid; i < s; i += SELT_SEL_THREADS) peer[i] = dst[i];
            }
        }
        if (tid == 0) {
            if (status) status[row] = PG_ITEM_OK;
            if (count) count[row] = s;
        }
        __syncthreads();
    }
}

template <int K>
static int launch_select_walk(const uint8_t *d_bases, const uint64_t *d_offsets, uint32_t read_len, uint64_t n_reads, int s,
                              uint32_t P, uint32_t *d_out, uint64_t row_stride, uint32_t *d_count, int32_t *d_status,
                              cudaStream_t st, const SketchDst &ex, const uint64_t *d_slice_beg = nullptr,
                              const uint32_t *d_slice_n = nullptr, const uint32_t *d_row_list = nullptr,
                              const uint32_t *d_n_list = nullptr) {
    const uint32_t cap = (std::max<uint32_t>(P, (uint32_t)s + SELW_ROOM) + 3u) & ~3u;
    const size_t words = (size_t)cap + (((size_t)s + 3) & ~(size_t)3) + 4 + 2 * SELW_STAGE_WORDS + (SEL_NBK + 1) + 16;
    const size_t smem = words * 4;
    { const int rc_ = func_smem((const void *)sketch_select_walk_kernel<K>, smem); if (rc_ != PG_OK) return rc_; }
    int per_sm = 1;
    PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sketch_select_walk_kernel<K>, SELW_THREADS, smem));
    const uint64_t blocks = std::min<uint64_t>(n_reads, (uint64_t)sm_count() * std::max(per_sm, 1));
    StreamScratch tmp(st);
    unsigned long long *d_next = nullptr;
    PG_CUDA(tmp.alloc(&d_next, 1));
    PG_CUDA(cudaMemsetAsync(d_next, 0, 8, st));
    sketch_select_walk_kernel<K><<<(unsigned)blocks, SELW_THREADS, smem, st>>>(d_bases, d_offsets, read_len, n_reads, (uint32_t)s, P, cap,
                                                                              d_out, row_stride, d_count, d_status, ex, 4u, d_slice_beg,
                                                                              d_slice_n, d_next, d_row_list, d_n_list);
    PG_LAUNCH_CHECK("sketch_select_walk_kernel");
    return PG_OK;
}

// Few, long sequences (genomes): one CTA per sequence leaves the GPU idle.  Cut every
// select-regime row into slices of >= max(4 chunks, 8 s) k-mer positions (about 4 slices per
// resident CTA slot over the whole batch; rows are handed out dynamically), sketch the slices independently, merge per row.
// *sliced = false when slicing would not add parallelism (the caller then runs the direct path).
template <int K>
static int try_select_sliced(const uint8_t *d_bases, const uint64_t *d_offsets, uint32_t read_len, uint64_t n_reads, int s,
                             uint32_t P, uint32_t *d_out, uint64_t row_stride, uint32_t *d_count, int32_t *d_status,
                             cudaStream_t st, bool *sliced) {
    *sliced = false;
    const uint64_t slots = (uint64_t)sm_count() * 3;
    if (s < 2 || n_reads > 4 * slots) return PG_OK;  // s == 1 needs the positional panic rule; enough rows already
    std::vector<uint64_t> off(n_reads + 1);
    if (d_offsets) {
        PG_CUDA(cudaMemcpyAsync(off.data(), d_offsets, (n_reads + 1) * 8, cudaMemcpyDeviceToHost, st));
        PG_CUDA(cudaStreamSynchronize(st));
    } else {
        for (uint64_t r = 0; r <= n_reads; ++r) off[r] = r * (uint64_t)read_len;
    }
    uint64_t total = 0, rows_sel = 0;
    for (uint64_t r = 0; r < n_reads; ++r) {
        const uint64_t len = off[r + 1] - off[r], n = len > (uint64_t)K ? len - K : 0;
        if (n >= (uint64_t)s && n > 0) { total += n; ++rows_sel; }
    }
    if (rows_sel == 0 || rows_sel >= slots) return PG_OK;  // every resident CTA slot already has a row of its own
    uint64_t sl = std::max<uint64_t>({(uint64_t)4 * SELW_CHUNK, (uint64_t)8 * s, (total + 4 * slots - 1) / (4 * slots)});
    sl = (sl + SELW_CHUNK - 1) / SELW_CHUNK * SELW_CHUNK;
    std::vector<uint64_t> beg;
    std::vector<uint32_t> cnt, row0(n_reads + 1);
    for (uint64_t r = 0; r < n_reads; ++r) {
        row0[r] = (uint32_t)beg.size();
        const uint64_t len = off[r + 1] - off[r], n = len > (uint64_t)K ? len - K : 0;
        if (!(n >= (uint64_t)s && n > 0)) continue;
        const uint64_t nsl = std::max<uint64_t>(1, n / sl);  // the last slice takes the remainder (< 2 sl)
        if (n / nsl + sl > 0xffffffffull) return PG_OK;      // slice length must fit 32 bits
        for (uint64_t j = 0; j < nsl; ++j) {
            beg.push_back(off[r] + j * sl);
            cnt.push_back((uint32_t)(j + 1 < nsl ? sl : n - j * sl));
        }
    }
    row0[n_reads] = (uint32_t)beg.size();
    const uint64_t n_slices = beg.size();
    if (n_slices <= rows_sel) return PG_OK;  // nothing gets split
    StreamScratch tmp(st);
    uint64_t *d_beg = nullptr;
    uint32_t *d_cnt = nullptr, *d_row0 = nullptr, *d_part = nullptr;
    PG_CUDA(tmp.alloc(&d_beg, n_slices));
    PG_CUDA(tmp.alloc(&d_cnt, n_slices));
    PG_CUDA(tmp.alloc(&d_row0, n_reads + 1));
    PG_CUDA(tmp.alloc(&d_part, n_slices * (uint64_t)s));
    PG_CUDA(cudaMemcpyAsync(d_beg, beg.data(), n_slices * 8, cudaMemcpyHostToDevice, st));
    PG_CUDA(cudaMemcpyAsync(d_cnt, cnt.data(), n_slices * 4, cudaMemcpyHostToDevice, st));
    PG_CUDA(cudaMemcpyAsync(d_row0, row0.data(), (n_reads + 1) * 4, cudaMemcpyHostToDevice, st));
    PG_CUDA(cudaStreamSynchronize(st));  // the host vectors are pageable
    SketchDst none;
    none.n = 0;
    int rc = launch_select_walk<K>(d_bases, nullptr, 0, n_slices, s, P, d_part, (uint64_t)s, nullptr, nullptr, st, none, d_beg, d_cnt);
    if (rc == PG_OK) {
        const uint32_t cap = (std::max<uint32_t>(P, (uint32_t)s + 2 * SELM_CHUNK) + 3u) & ~3u;
        const size_t smem = ((size_t)cap + s + SEL_NBK + 64 + SEL_NBK + 1 + 8) * 4;
        { const int rc_ = func_smem((const void *)select_merge_kernel, smem); if (rc_ != PG_OK) return rc_; }
        const uint64_t blocks = std::min<uint64_t>(n_reads, (uint64_t)sm_count() * 2);
        select_merge_kernel<<<(unsigned)blocks, SELM_THREADS, smem, st>>>(d_part, d_row0, n_reads, (uint32_t)s, P, cap, d_out, row_stride,
                                                                         d_count, d_status);
        note_launch("select_merge_kernel");
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = cuda_fail(e, "select_merge_kernel", __FILE__, __LINE__);
    }
    *sliced = rc == PG_OK;
    return rc;
}

// K2t launcher.  *handled = false: not applicable (the caller takes the streaming path).
template <int K>
static int launch_select_thresh(const uint8_t *d_bases, const uint64_t *d_offsets, uint32_t read_len, uint64_t max_read_len,
                                uint64_t n_reads, int s, uint32_t P, uint32_t *d_out, uint64_t row_stride, uint32_t *d_count,
                                int32_t *d_status, cudaStream_t st, const SketchDst &ex, bool *handled) {
    *handled = false;
    const uint64_t len_max = d_offsets ? max_read_len : read_len;
    if (s < 2 || len_max <= (uint64_t)K || n_reads > 0xffffffffull) return PG_OK;  // s == 1 needs the positional panic rule
    const uint64_t nmax = len_max - K;
    const uint64_t item_len = (uint64_t)SELT_ITEM_CHUNKS * SeltGeom<K>::CHUNK;
    const uint64_t ipr = (nmax + item_len - 1) / item_len;
    if (ipr > 0xffffffffull) return PG_OK;
    // ragged batches map items as row x ipr (rows shorter than the longest leave empty items): bounded waste only
    if (d_offsets && ipr > 1 && n_reads * ipr > (4ull << 20)) return PG_OK;
    const uint32_t mu = (uint32_t)s + 6u * (uint32_t)ceil(sqrt((double)s)) + 48u;
    uint32_t cap = mu + 8u * (uint32_t)ceil(sqrt((double)mu)) + 96u;
    cap = (cap + 3u) & ~3u;
    const size_t smem_a = 2 * (size_t)SeltGeom<K>::STAGE + (size_t)SeltGeom<K>::SEG * 32 * 4;
    const size_t smem_b = ((((size_t)cap + 3) & ~(size_t)3) + SEL_NBK + 16) * 4;  // tmp | cur | flag
    if (smem_b > 220 * 1024) return PG_OK;
    // admission probability of the longest rows: below 1/512 a warp step (128 hashes) admits something a quarter of the time
    const uint32_t tm1_u = d_offsets ? 0u : selt_threshold_m1(nmax, mu);  // every row of a fixed-length batch has n == nmax
    const bool rare = (uint64_t)mu * 512 < nmax;
    const void *walk_fn = rare ? (const void *)sketch_thresh_walk_kernel<K, true> : (const void *)sketch_thresh_walk_kernel<K, false>;
    { const int rc_ = func_smem(walk_fn, smem_a); if (rc_ != PG_OK) return rc_; }
    // batch width of the select: fewest load slots for a typical row (mu + 2.5 sigma candidates), ties to the wider batch
    const uint32_t typ = mu + (uint32_t)(2.5 * sqrt((double)mu));
    int sel_u = 8;
    {
        uint32_t best = ~0u;
        for (int u : {3, 4, 5, 6, 8}) {
            const uint32_t slots = (typ + u * SELT_SEL_THREADS - 1) / (u * SELT_SEL_THREADS) * u;
            if (slots <= best) { best = slots; sel_u = u; }
        }
    }
    // bucket function: the plain shift when it uses >= 3/4 of the 2048 buckets (fixed-length batch: T known here)
    bool sel_mul = true;
    if (!d_offsets) {
        const uint32_t tb = 32u - (uint32_t)__builtin_clz(tm1_u | 1u);
        sel_mul = ((tm1_u >> (tb > 11u ? tb - 11u : 0u)) + 1u) < 1536u;
    }
#define PG_SEL_FN(U_) (sel_mul ? (const void *)sketch_thresh_select_kernel<U_, true> : (const void *)sketch_thresh_select_kernel<U_, false>)
    const void *sel_fn = sel_u == 3 ? PG_SEL_FN(3) : sel_u == 4 ? PG_SEL_FN(4) : sel_u == 5 ? PG_SEL_FN(5) : sel_u == 6 ? PG_SEL_FN(6) : PG_SEL_FN(8);
#undef PG_SEL_FN
    { const int rc_ = func_smem(sel_fn, smem_b); if (rc_ != PG_OK) return rc_; }
    int per_sm = 1;
    PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sel_fn, SELT_SEL_THREADS, smem_b));
    // candidate lists: cap words per row, rows in groups of <= 1.5 GiB of temporaries
    uint64_t rows_per_group = std::max<uint64_t>(1, std::min<uint64_t>((3ull << 28) / cap, 0x7fffffffull / ipr));
    if (const char *e = getenv("PG_K2T_GROUP_ROWS"))  // test knob: force several launch groups
        if (atoll(e) > 0) rows_per_group = std::min<uint64_t>(rows_per_group, (uint64_t)atoll(e));
    const uint64_t group = std::min(n_reads, rows_per_group);
    StreamScratch tmp(st);
    uint32_t *d_cand = nullptr, *d_cnt = nullptr, *d_retry = nullptr, *d_nretry = nullptr;
    PG_CUDA(tmp.alloc(&d_cand, group * cap));
    PG_CUDA(tmp.alloc(&d_cnt, group));
    PG_CUDA(tmp.alloc(&d_retry, n_reads));
    PG_CUDA(tmp.alloc(&d_nretry, 1));
    PG_CUDA(cudaMemsetAsync(d_nretry, 0, 4, st));
    for (uint64_t r0 = 0; r0 < n_reads; r0 += group) {
        const uint64_t rows = std::min(group, n_reads - r0);
        PG_CUDA(cudaMemsetAsync(d_cnt, 0, rows * 4, st));
#define PG_LAUNCH_WALK(RARE_)                                                                                              \
    sketch_thresh_walk_kernel<K, RARE_><<<(unsigned)(rows * ipr), 32, smem_a, st>>>(d_bases, d_offsets, read_len, r0, rows, \
                                                                                   (uint32_t)ipr, (uint32_t)s, mu, cap, d_cand, d_cnt, 4u, tm1_u)
        if (rare) PG_LAUNCH_WALK(true);
        else PG_LAUNCH_WALK(false);
#undef PG_LAUNCH_WALK
        PG_LAUNCH_CHECK("sketch_thresh_walk_kernel");
        const uint64_t blocks = std::min<uint64_t>(rows, (uint64_t)sm_count() * std::max(per_sm, 1));
#define PG_LAUNCH_SEL_(U_, M_)                                                                                                 \
    sketch_thresh_select_kernel<U_, M_><<<(unsigned)blocks, SELT_SEL_THREADS, smem_b, st>>>(d_offsets, read_len, r0, rows, (uint32_t)K, (uint32_t)s, \
                                                                                             mu, cap, d_cand, d_cnt, d_out, row_stride, d_count,     \
                                                                                             d_status, ex, d_retry, d_nretry, tm1_u)
#define PG_LAUNCH_SEL(U_) do { if (sel_mul) PG_LAUNCH_SEL_(U_, true); else PG_LAUNCH_SEL_(U_, false); } while (0)
        switch (sel_u) {
            case 3: PG_LAUNCH_SEL(3); break;
            case 4: PG_LAUNCH_SEL(4); break;
            case 5: PG_LAUNCH_SEL(5); break;
            case 6: PG_LAUNCH_SEL(6); break;
            default: PG_LAUNCH_SEL(8); break;
        }
#undef PG_LAUNCH_SEL
#undef PG_LAUNCH_SEL_
        PG_LAUNCH_CHECK("sketch_thresh_select_kernel");
    }
    // rows the estimate failed on (few distinct k-mers, heavy duplication): exact streaming kernel, device-side list
    int rc = launch_select_walk<K>(d_bases, d_offsets, read_len, n_reads, s, P, d_out, row_stride, d_count, d_status, st, ex, nullptr, nullptr,
                                   d_retry, d_nretry);
    if (rc != PG_OK) return rc;
    *handled = true;
    return PG_OK;
}

template <int K>
static int launch_select_auto(const uint8_t *d_bases, const uint64_t *d_offsets, uint32_t read_len, uint64_t max_read_len, uint64_t n_reads, int s,
                              uint32_t P, uint32_t *d_out, uint64_t row_stride, uint32_t *d_count, int32_t *d_status,
                              cudaStream_t st, const SketchDst &ex) {
    bool handled = false;
    int rc = launch_select_thresh<K>(d_bases, d_offsets, read_len, max_read_len, n_reads, s, P, d_out, row_stride, d_count, d_status, st, ex,
                                     &handled);
    if (rc != PG_OK || handled) return rc;
    if (ex.n == 0) {
        bool sliced = false;
        rc = try_select_sliced<K>(d_bases, d_offsets, read_len, n_reads, s, P, d_out, row_stride, d_count, d_status, st, &sliced);
        if (rc != PG_OK || sliced) return rc;
    }
    return launch_select_walk<K>(d_bases, d_offsets, read_len, n_reads, s, P, d_out, row_stride, d_count, d_status, st, ex);
}

}  // namespace

int launch_sketch_select(const uint8_t *d_bases, const uint64_t *d_offsets, uint32_t read_len,
                         uint64_t n_reads, int k, int s, uint32_t flags, uint32_t *d_out,
                         uint64_t row_stride, uint32_t *d_count, int32_t *d_status,
                         cudaStream_t st, const SketchDst *extra, uint64_t max_read_len) {
    if (n_reads == 0) return PG_OK;
    SketchDst ex;
    ex.n = 0;
    if (extra) ex = *extra;
    // rows wider than s: the header promises zeros in [count, row_stride) -- the select kernels write
    // exactly s words, so clear the tail columns first (fill-regime rows of a ragged batch zero their own)
    if (row_stride > (uint64_t)s)
        PG_CUDA(cudaMemset2DAsync(d_out + s, row_stride * 4, 0, (row_stride - (uint64_t)s) * 4, n_reads, st));
    // beyond the shared-memory kernels (sketch or k-mer too large for them): the global-memory path, no limit on either
    if (s > SEL_MAX_S || k > SEL_LOOKAHEAD)
        return launch_sketch_select_large(d_bases, d_offsets, read_len, n_reads, k, s, d_out, row_stride, d_count, d_status, st, ex);
    uint32_t P = 1;
    while (P < (uint32_t)std::max(s, 1)) P <<= 1;
    if (P < 2) P = 2;
    // K2t / K2w (register-ring walks) for the instantiated k
    if ((size_t)s * 8 + 56 * 1024 <= 227 * 1024) {  // shared memory of the walk kernel
        switch (k) {
#define PG_K2W_CASE(KK) \
    case KK: return launch_select_auto<KK>(d_bases, d_offsets, read_len, max_read_len, n_reads, s, P, d_out, row_stride, d_count, d_status, st, ex);
            PG_K2W_CASE(11) PG_K2W_CASE(13) PG_K2W_CASE(15) PG_K2W_CASE(16) PG_K2W_CASE(17) PG_K2W_CASE(19)
            PG_K2W_CASE(21) PG_K2W_CASE(23) PG_K2W_CASE(24) PG_K2W_CASE(25) PG_K2W_CASE(27) PG_K2W_CASE(29)
            PG_K2W_CASE(31) PG_K2W_CASE(32)
#undef PG_K2W_CASE
            default: break;
        }
    }
    uint32_t cap = (std::max<uint32_t>(P, (uint32_t)s + 4 * SEL_CHUNK) + 3u) & ~3u;
    const size_t words = (size_t)cap + (((size_t)s + 3) & ~(size_t)3) + 4 + (SEL_CHUNK + SEL_LOOKAHEAD) +
                         2 * SEL_STAGE_WORDS + (SEL_NBK + 1) + 8;
    const size_t smem = words * 4;
    { const int rc_ = func_smem((const void *)sketch_select_kernel, smem); if (rc_ != PG_OK) return rc_; }
    int per_sm = 1;
    PG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sketch_select_kernel, SEL_THREADS, smem));
    const uint64_t blocks = std::min<uint64_t>(n_reads, (uint64_t)sm_count() * std::max(per_sm, 1));  // one wave, grid-stride over rows
    sketch_select_kernel<<<(unsigned)blocks, SEL_THREADS, smem, st>>>(
        d_bases, d_offsets, read_len, n_reads, (uint32_t)k, (uint32_t)s, P, cap, flags, d_out,
        row_stride, d_count, d_status, ex);
    PG_LAUNCH_CHECK("sketch_select_kernel");
    return PG_OK;
}

}  // namespace pg
