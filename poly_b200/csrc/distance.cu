// distance.cu -- K3: (*Mash).Similarity / Distance,
// /root/reference/search/mash/mash.go:107-140, with the reference's literal semantics:
// larger/smaller by SketchSize (receiver wins ties), the range early-out on
// Sketches[size-1] / Sketches[0], the two-pointer walk, same/smaller.SketchSize.
//
// similarity_pairs_kernel : explicit pair list over sketches of arbitrary sizes, one
//                           warp per pair (merge-path partition of the walk when both
//                           sketches are ascending, literal serial walk otherwise).
// distance_block_kernel   : row block x all columns over equal-size sketches; a CTA
//                           owns a TILE x TILE block of pairs with both sketch tiles
//                           staged in shared memory.
#include <algorithm>

#include "common.cuh"

namespace pg {

namespace {

// literal walk, mash.go:121-132
template <typename GetS, typename GetL>
__device__ __forceinline__ uint32_t walk_literal(GetS small, uint32_t ss, GetL large, uint32_t sl) {
    uint32_t same = 0, si = 0, li = 0;
    while (si < ss && li < sl) {
        const uint32_t a = small(si), b = large(li);
        if (a == b) { ++same; ++si; ++li; }
        else if (a < b) ++si;
        else ++li;
    }
    return same;
}

// One warp per pair.  Lanes cooperatively test sortedness; sorted pairs are counted by
// binary-search intersection with multiset semantics (sum over values of
// min(cnt_small, cnt_large), identical to the walk on ascending inputs, SURVEY 8a a5);
// anything else falls back to the literal walk on lane 0.
__global__ void __launch_bounds__(256)
similarity_pairs_kernel(const uint32_t *__restrict__ sk, const uint64_t *__restrict__ off,
                        uint64_t n_sk, const uint32_t *__restrict__ pa,
                        const uint32_t *__restrict__ pb, uint64_t n_pairs,
                        int64_t *__restrict__ same_out, double *__restrict__ sim_out,
                        double *__restrict__ dist_out, int32_t *__restrict__ status) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t p = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; p < n_pairs;
         p += warps) {
        const uint32_t ia = pa[p], ib = pb[p];
        if (ia >= n_sk || ib >= n_sk) {
            if (lane == 0 && status) status[p] = PG_ITEM_PANIC;
            continue;
        }
        const uint32_t *A = sk + off[ia], *B = sk + off[ib];
        const uint64_t sa64 = off[ia + 1] - off[ia], sb64 = off[ib + 1] - off[ib];
        if (sa64 == 0 || sb64 == 0) {  // Sketches[SketchSize-1] with SketchSize 0
            if (lane == 0) {
                if (status) status[p] = PG_ITEM_PANIC;
                if (same_out) same_out[p] = 0;
            }
            continue;
        }
        const uint32_t sa = (uint32_t)sa64, sb = (uint32_t)sb64;
        const uint32_t *L = A, *S = B;  // mash.go:109-110: receiver is "larger"
        uint32_t sl = sa, ss = sb;
        if (sa < sb) { L = B; sl = sb; S = A; ss = sa; }  // mash.go:112-115
        uint32_t same = 0;
        const bool early = __ldg(L + sl - 1) < __ldg(S) || __ldg(S + ss - 1) < __ldg(L);  // :117
        if (!early) {
            // sortedness of both arrays (non-decreasing)
            bool ok = true;
            for (uint32_t i = lane + 1; i < sl; i += 32) ok &= __ldg(L + i - 1) <= __ldg(L + i);
            for (uint32_t i = lane + 1; i < ss; i += 32) ok &= __ldg(S + i - 1) <= __ldg(S + i);
            ok = __all_sync(0xffffffffu, ok);
            if (ok) {
                // element i of S (its t-th copy, t = i - first index of the value) matches
                // iff L holds more than t copies of the value
                uint32_t local = 0;
                for (uint32_t i = lane; i < ss; i += 32) {
                    const uint32_t v = __ldg(S + i);
                    // lower bounds of v in S and in L, upper bound in L
                    uint32_t lo = 0, hi = i;
                    while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if (__ldg(S + m) < v) lo = m + 1; else hi = m; }
                    const uint32_t t = i - lo;
                    uint32_t l0 = 0, l1 = sl;
                    while (l0 < l1) { const uint32_t m = (l0 + l1) >> 1; if (__ldg(L + m) < v) l0 = m + 1; else l1 = m; }
                    if (l0 + t < sl && __ldg(L + l0 + t) == v) ++local;
                }
                for (int d = 16; d > 0; d >>= 1) local += __shfl_xor_sync(0xffffffffu, local, d);
                same = local;
            } else {
                if (lane == 0)
                    same = walk_literal([S](uint32_t i) { return __ldg(S + i); }, ss,
                                        [L](uint32_t i) { return __ldg(L + i); }, sl);
                same = __shfl_sync(0xffffffffu, same, 0);
            }
        }
        if (lane == 0) {
            const double sim = (double)same / (double)ss;  // mash.go:134
            if (same_out) same_out[p] = (int64_t)same;
            if (sim_out) sim_out[p] = sim;
            if (dist_out) dist_out[p] = 1 - sim;  // mash.go:139
            if (status) status[p] = PG_ITEM_OK;
        }
    }
}

// Row block x all columns over n equal-size sketches.  One warp per (row, column)
// pair inside a CTA tile of BT x BT pairs; equal sizes -> receiver (row) is "larger",
// argument (column) is "smaller" (mash.go:109-115).
constexpr int BT = 8;  // sketches per tile side

__global__ void __launch_bounds__(256)
distance_block_kernel(const uint32_t *__restrict__ sk, uint64_t n, uint32_t s, uint64_t row_begin,
                      uint64_t row_end, const uint8_t *__restrict__ sorted_flag,
                      uint32_t *__restrict__ same_out, double *__restrict__ dist_out) {
    extern __shared__ __align__(16) uint32_t tile[];  // rows [BT][s] then cols [BT][s]
    uint32_t *srow = tile, *scol = tile + (size_t)BT * s;
    const uint64_t r0 = row_begin + (uint64_t)blockIdx.y * BT;
    const uint64_t c0 = (uint64_t)blockIdx.x * BT;
    const uint32_t nr = (uint32_t)min((uint64_t)BT, row_end - r0);
    const uint32_t nc = (uint32_t)min((uint64_t)BT, n - c0);
    // mash.go:117-119 needs only the first and last word of each sketch: if every pair of the
    // tile early-outs (always the case for zero-padded fill-regime sketches) skip the staging
    {
        bool work = false;
        if (threadIdx.x < nr * nc) {
            const uint32_t ri = threadIdx.x / nc, ci = threadIdx.x % nc;
            const uint32_t *L = sk + (r0 + ri) * s, *S = sk + (c0 + ci) * s;
            work = !(__ldg(L + s - 1) < __ldg(S) || __ldg(S + s - 1) < __ldg(L));
            if (!work) {
                const uint64_t o = (r0 + ri - row_begin) * n + (c0 + ci);
                if (same_out) same_out[o] = 0;
                if (dist_out) dist_out[o] = 1 - (double)0 / (double)s;
            }
        }
        if (!__syncthreads_or(work)) return;
    }
    for (uint32_t i = threadIdx.x; i < nr * s; i += blockDim.x) srow[i] = __ldg(sk + r0 * s + i);
    for (uint32_t i = threadIdx.x; i < nc * s; i += blockDim.x) scol[i] = __ldg(sk + c0 * s + i);
    __syncthreads();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u, nwarps = blockDim.x >> 5;
    for (uint32_t pr = warp; pr < nr * nc; pr += nwarps) {
        const uint32_t ri = pr / nc, ci = pr % nc;
        const uint32_t *L = srow + (size_t)ri * s;  // receiver
        const uint32_t *S = scol + (size_t)ci * s;  // argument
        uint32_t same = 0;
        const bool early = L[s - 1] < S[0] || S[s - 1] < L[0];  // mash.go:117
        if (!early) {
            if (sorted_flag[r0 + ri] && sorted_flag[c0 + ci]) {
                uint32_t local = 0;
                for (uint32_t i = lane; i < s; i += 32) {
                    const uint32_t v = S[i];
                    uint32_t lo = 0, hi = i;
                    while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if (S[m] < v) lo = m + 1; else hi = m; }
                    const uint32_t t = i - lo;
                    uint32_t l0 = 0, l1 = s;
                    while (l0 < l1) { const uint32_t m = (l0 + l1) >> 1; if (L[m] < v) l0 = m + 1; else l1 = m; }
                    if (l0 + t < s && L[l0 + t] == v) ++local;
                }
                for (int d = 16; d > 0; d >>= 1) local += __shfl_xor_sync(0xffffffffu, local, d);
                same = local;
            } else {
                if (lane == 0)
                    same = walk_literal([S](uint32_t i) { return S[i]; }, s,
                                        [L](uint32_t i) { return L[i]; }, s);
                same = __shfl_sync(0xffffffffu, same, 0);
            }
        }
        if (lane == 0) {
            const uint64_t o = (r0 + ri - row_begin) * n + (c0 + ci);
            if (same_out) same_out[o] = same;
            if (dist_out) dist_out[o] = 1 - (double)same / (double)s;
        }
    }
}

__global__ void sorted_flag_kernel(const uint32_t *__restrict__ sk, uint64_t n, uint32_t s,
                                   uint8_t *__restrict__ flag, uint32_t *__restrict__ n_unsorted) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
        const uint32_t *x = sk + r * s;
        bool ok = true;
        for (uint32_t i = lane + 1; i < s; i += 32) ok &= __ldg(x + i - 1) <= __ldg(x + i);
        ok = __all_sync(0xffffffffu, ok);
        if (lane == 0) {
            flag[r] = ok ? 1 : 0;
            if (!ok) atomicAdd(n_unsorted, 1u);
        }
    }
}

// dense row-block tile -> (i, j, same) triples of the non-zero off-diagonal entries
__global__ void __launch_bounds__(256)
compact_pairs_kernel(const uint32_t *__restrict__ tile, uint64_t rows, uint64_t n, uint64_t row0, uint32_t upper,
                     uint32_t *__restrict__ oi, uint32_t *__restrict__ oj, uint32_t *__restrict__ osame, uint64_t cap,
                     unsigned long long *__restrict__ counter) {
    const uint64_t total = rows * n;
    const uint32_t lane = threadIdx.x & 31u;
    // the loop bound is warp-uniform (the ballots below need every lane): a warp covers 128 consecutive words
    for (uint64_t w0 = ((uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)) * 4; w0 < total; w0 += (uint64_t)gridDim.x * blockDim.x * 4) {
        const uint64_t e0 = w0 + lane * 4;
        uint32_t v[4] = {0, 0, 0, 0};
        if (e0 + 3 < total && (n & 3) == 0) {
            const uint4 q = *reinterpret_cast<const uint4 *>(tile + e0);  // rows are 16-byte aligned when n % 4 == 0
            v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
            for (int t = 0; t < 4; ++t) if (e0 + t < total) v[t] = tile[e0 + t];
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const uint64_t e = e0 + t;
            const uint64_t i = row0 + (e < total ? e / n : 0), j = e < total ? e % n : 0;
            const bool keep = e < total && v[t] != 0 && j != i && (!upper || j > i);
            const uint32_t b = __ballot_sync(0xffffffffu, keep);
            if (!b) continue;
            unsigned long long base = 0;
            if (lane == (uint32_t)(__ffs(b) - 1)) base = atomicAdd(counter, (unsigned long long)__popc(b));
            base = __shfl_sync(0xffffffffu, base, __ffs(b) - 1);
            const unsigned long long slot = base + __popc(b & ((1u << lane) - 1u));
            if (keep && slot < cap) { oi[slot] = (uint32_t)i; oj[slot] = (uint32_t)j; osame[slot] = v[t]; }
        }
    }
}

}  // namespace

// Non-zero off-diagonal matching counts of rows [row_begin, row_end) as (i, j, same) triples: dense tiles of
// the row block (same kernels as the dense entry point) compacted on the device, so only the informative
// pairs ever leave the GPU.  *d_n_pairs counts every qualifying pair, also beyond pairs_cap.
int launch_distance_sparse(const uint32_t *d_sk, uint64_t n, int s, uint64_t row_begin, uint64_t row_end, uint32_t flags,
                           uint32_t *d_i, uint32_t *d_j, uint32_t *d_same, uint64_t cap, unsigned long long *d_n_pairs,
                           cudaStream_t st) {
    PG_CUDA(cudaMemsetAsync(d_n_pairs, 0, 8, st));
    if (row_end <= row_begin || n == 0) return PG_OK;
    if (n > 0xffffffffull) { set_error("too many sketches for 32-bit pair indices"); return PG_ERR_ARG; }
    DistancePlan plan;
    int rc = distance_plan_create(d_sk, n, s, st, &plan);
    // tiles of <= 8 GiB: every pass over the index costs one read of all its entries and the run tables of every
    // bucket, but a tile that outgrows the memory pool's cache is mapped and unmapped by the driver on every call
    // (measured: one 40 GB tile = 675 ms per call against 111 ms for five 8 GiB tiles)
    const uint64_t budget_words = 2ull << 30;
    const uint64_t rows_per = std::max<uint64_t>(8, std::min<uint64_t>(row_end - row_begin, (budget_words / n) & ~7ull));
    uint32_t *d_tile = nullptr;
    if (rc == PG_OK) {
        cudaError_t e = cudaMallocAsync(&d_tile, rows_per * n * 4, st);
        if (e != cudaSuccess) { cudaGetLastError(); set_error("cudaMallocAsync(%llu) for the pair tile failed", (unsigned long long)(rows_per * n * 4)); rc = PG_ERR_NOMEM; }
    }
    for (uint64_t rb = row_begin; rb < row_end && rc == PG_OK; rb += rows_per) {
        const uint64_t re = std::min(row_end, rb + rows_per);
        rc = distance_plan_rows(plan, rb, re, d_tile, nullptr, st);
        if (rc != PG_OK) break;
        const uint64_t quads = ((re - rb) * n + 3) / 4;
        compact_pairs_kernel<<<(unsigned)std::min<uint64_t>((quads + 255) / 256, (uint64_t)sm_count() * 16), 256, 0, st>>>(
            d_tile, re - rb, n, rb, flags & PG_PAIRS_UPPER, d_i, d_j, d_same, cap, d_n_pairs);
        note_launch("compact_pairs_kernel");
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = cuda_fail(e, "compact_pairs_kernel", __FILE__, __LINE__);
    }
    if (d_tile) cudaFreeAsync(d_tile, st);
    distance_plan_destroy(plan, st);
    return rc;
}

int launch_similarity_pairs(const uint32_t *d_sk, const uint64_t *d_off, uint64_t n_sk,
                            const uint32_t *d_a, const uint32_t *d_b, uint64_t n_pairs,
                            int64_t *d_same, double *d_sim, double *d_dist, int32_t *d_status,
                            cudaStream_t st) {
    if (n_pairs == 0) return PG_OK;
    const uint64_t blocks = std::min<uint64_t>((n_pairs + 7) / 8, (uint64_t)sm_count() * 16);
    similarity_pairs_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_sk, d_off, n_sk, d_a, d_b, n_pairs,
                                                              d_same, d_sim, d_dist, d_status);
    PG_LAUNCH_CHECK("similarity_pairs_kernel");
    return PG_OK;
}

int distance_plan_create(const uint32_t *d_sk, uint64_t n, int s, cudaStream_t st, DistancePlan *plan) {
    plan->d_sk = d_sk; plan->n = n; plan->s = s; plan->d_flag = nullptr; plan->join = JoinIndex();
    if (n == 0) return PG_OK;
    if (s <= 0) {
        set_error("distance over sketches of size %d: the reference panics (Sketches[-1])", s);
        return PG_ERR_PANIC;
    }
    PG_CUDA(cudaMallocAsync(&plan->d_flag, n + 8, st));
    uint32_t *d_unsorted = reinterpret_cast<uint32_t *>(plan->d_flag + ((n + 3) & ~3ull));
    PG_CUDA(cudaMemsetAsync(d_unsorted, 0, 4, st));
    sorted_flag_kernel<<<(unsigned)std::min<uint64_t>((n + 7) / 8, 4096), 256, 0, st>>>(d_sk, n, s, plan->d_flag, d_unsorted);
    PG_LAUNCH_CHECK("sorted_flag_kernel");
    // every sketch ascending (the select regime, L-k >= s): inverted-index join, output-sensitive
    uint32_t n_unsorted = 1;
    PG_CUDA(cudaMemcpyAsync(&n_unsorted, d_unsorted, 4, cudaMemcpyDeviceToHost, st));
    PG_CUDA(cudaStreamSynchronize(st));
    if (n_unsorted == 0) return join_build(d_sk, n, s, st, &plan->join);
    return PG_OK;
}

void distance_plan_destroy(DistancePlan &plan, cudaStream_t st) {
    join_free(plan.join, st);
    if (plan.d_flag) cudaFreeAsync(plan.d_flag, st);
    plan.d_flag = nullptr;
}

int distance_plan_rows(const DistancePlan &plan, uint64_t row_begin, uint64_t row_end, uint32_t *d_same, double *d_dist,
                       cudaStream_t st) {
    const uint64_t n = plan.n;
    const int s = plan.s;
    if (row_end <= row_begin || n == 0) return PG_OK;
    const uint64_t rows = row_end - row_begin;
    if (plan.join.ok) {
        uint32_t *same = d_same;
        if (!same) PG_CUDA(cudaMallocAsync(&same, rows * n * 4, st));  // distances only: counts are a temporary
        int rc = join_emit(plan.join, row_begin, row_end, same, d_dist, st);
        if (!d_same) cudaFreeAsync(same, st);
        return rc;
    }
    const size_t smem = (size_t)2 * BT * s * 4;
    if (smem > 200 * 1024) {
        set_error("sketch size %d too large for the all-pairs tile kernel", s);
        return PG_ERR_UNSUPPORTED;
    }
    { const int rc_ = func_smem((const void *)distance_block_kernel, smem); if (rc_ != PG_OK) return rc_; }
    const uint64_t gy_total = (rows + BT - 1) / BT;
    const uint64_t gx = (n + BT - 1) / BT;
    if (gx > 0x7fffffffull) { set_error("too many sketches"); return PG_ERR_ARG; }
    for (uint64_t y0 = 0; y0 < gy_total; y0 += 65535) {  // gridDim.y limit
        const uint64_t gy = std::min<uint64_t>(65535, gy_total - y0);
        const uint64_t rb = row_begin + y0 * BT;
        dim3 grid((unsigned)gx, (unsigned)gy);
        distance_block_kernel<<<grid, 256, smem, st>>>(
            plan.d_sk, n, (uint32_t)s, rb, row_end, plan.d_flag,
            d_same ? d_same + (rb - row_begin) * n : nullptr,
            d_dist ? d_dist + (rb - row_begin) * n : nullptr);
        PG_LAUNCH_CHECK("distance_block_kernel");
    }
    return PG_OK;
}

int launch_distance_block(const uint32_t *d_sk, uint64_t n, int s, uint64_t row_begin,
                          uint64_t row_end, uint32_t *d_same, double *d_dist, cudaStream_t st) {
    if (row_end <= row_begin || n == 0) return PG_OK;
    DistancePlan plan;
    int rc = distance_plan_create(d_sk, n, s, st, &plan);
    if (rc == PG_OK) rc = distance_plan_rows(plan, row_begin, row_end, d_same, d_dist, st);
    distance_plan_destroy(plan, st);
    return rc;
}

}  // namespace pg
