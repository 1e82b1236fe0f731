// sw_score.cu -- K4: Smith-Waterman (and Needleman-Wunsch, align.go:100-134,166) score of n short
// queries against one template,
// /root/reference/search/align/align.go:171-203 (fill + running max; the traceback at
// :205-231 is out of scope).  Linear gap (ADDED, align.go:193-194), arbitrary
// substitution table addressed through two byte->index LUTs
// (search/align/matrix/matrix.go:28-38, alphabet/alphabet.go:35-41).
//
// One thread per query.  The thread sweeps the template once, keeping the DP column
// over its query (<= MAXQ cells) in registers; the template's symbol indices are
// staged in shared memory and broadcast; the substitution table sits in shared memory
// (a nucleotide table is <= 32 words = one word per bank).  Three DPX
// add-max instructions per cell.  The max score does not depend on which string is
// the outer loop; the reported error (first failing cell in row-major order,
// align.go:188-191) does, and is resolved per orientation at the end.
#include <algorithm>
#include <cstring>
#include <limits>
#include <type_traits>
#include <vector>

#include "common.cuh"

namespace pg {

namespace {

constexpr int SW_THREADS = 128;
constexpr int SW_TCHUNK = 8192;  // template symbols staged per pass

template <typename T>
__device__ __forceinline__ T addmax(T a, T b, T c) {  // max(a + b, c)
    const T x = a + b;
    return x > c ? x : c;
}
template <>
__device__ __forceinline__ int addmax<int>(int a, int b, int c) {
    return __viaddmax_s32(a, b, c);
}

struct SwParams {
    const uint8_t *q;
    const uint64_t *qoff;
    uint64_t nq;
    const uint8_t *t;
    uint64_t tlen;
    int query_is_a;
    int n_q, n_t;  // alphabet sizes on the query / template side
    int global;    // 0: Smith-Waterman (local), 1: Needleman-Wunsch (global) score
};

// Short queries (<= ROWS cells): one thread per query, DP column in registers, no branches in
// the cell loop.  Rows at or beyond the query length read a score of -BIG, so (for gap <= 0)
// they can never exceed a valid cell and need no masking; a positive "gap" takes the MASK
// variant.  PROFILE: the per-thread query profile prof[t][i] = S(q_i, t) is expanded into
// shared memory ([n_t][ROWS][threads], conflict-free, immediate offsets) so a cell is
// 1 LDS + 3 add-max + 1 max; otherwise (large alphabets) the score comes from the shared
// table through a per-row offset.
template <typename T>
struct SwBig {
    static constexpr T value = (T)1 << (sizeof(T) * 8 - 3);  // 2^29 / 2^61: no overflow in diag + sc
};

template <typename T, int ROWS, bool PROFILE, bool MASK, bool GLOBAL>
__global__ void __launch_bounds__(SW_THREADS)
sw_score_kernel(SwParams p, const int16_t *__restrict__ lut_q, const int16_t *__restrict__ lut_t,
                const T *__restrict__ tab, T gap, int64_t *__restrict__ score,
                int32_t *__restrict__ err, int64_t *__restrict__ errpos) {
    extern __shared__ __align__(16) uint8_t sm[];
    // layout: [s_tidx: SW_TCHUNK bytes][s_lut_t: 256 int16][s_tab: (n_q+1)*n_t T][prof: n_t*ROWS*threads T]
    uint8_t *s_tidx = sm;
    int16_t *s_lut_t = reinterpret_cast<int16_t *>(sm + SW_TCHUNK);
    T *s_tab = reinterpret_cast<T *>(sm + SW_TCHUNK + 512);
    T *s_prof = s_tab + (p.n_q + 1) * p.n_t;
    __shared__ unsigned long long s_first_bad_t;

    const uint32_t tid = threadIdx.x;
    const T NEG = (T)0 - SwBig<T>::value;
    for (int i = tid; i < p.n_q * p.n_t; i += SW_THREADS) s_tab[i] = tab[i];
    for (int i = tid; i < p.n_t; i += SW_THREADS) s_tab[p.n_q * p.n_t + i] = NEG;  // row n_q: "beyond the query"
    for (int i = tid; i < 256; i += SW_THREADS) s_lut_t[i] = lut_t[i];
    if (tid == 0) s_first_bad_t = ~0ull;
    __syncthreads();

    const uint64_t qi = (uint64_t)blockIdx.x * SW_THREADS + tid;
    const bool active = qi < p.nq;
    uint64_t qbeg = 0;
    uint32_t qlen = 0;
    if (active) {
        qbeg = p.qoff[qi];
        qlen = (uint32_t)(p.qoff[qi + 1] - qbeg);
    }
    // per-row table offsets; invalid symbols score through row 0 and are reported at the end
    int qrow[ROWS];
    int64_t first_bad_q = -1;
#pragma unroll
    for (int i = 0; i < ROWS; ++i) {
        qrow[i] = p.n_q * p.n_t;
        if (i < (int)qlen) {
            const int ix = lut_q[__ldg(p.q + qbeg + i)];
            if (ix < 0) {
                if (first_bad_q < 0) first_bad_q = i;
                qrow[i] = 0;
            } else {
                qrow[i] = ix * p.n_t;
            }
        }
    }
    if (PROFILE) {
        for (int t = 0; t < p.n_t; ++t) {
#pragma unroll
            for (int i = 0; i < ROWS; ++i) s_prof[(t * ROWS + i) * SW_THREADS + tid] = s_tab[qrow[i] + t];
        }
    }
    T col[ROWS];
#pragma unroll
    for (int i = 0; i < ROWS; ++i) col[i] = GLOBAL ? (T)(i + 1) * gap : (T)0;  // NW: first column, align.go:115-117
    T best = 0;
    T edge = 0;  // NW: H[0][j-1], the first-row gap ramp (align.go:120-122)

    for (uint64_t t0 = 0; t0 < p.tlen; t0 += SW_TCHUNK) {
        const uint32_t tc = (uint32_t)min((uint64_t)SW_TCHUNK, p.tlen - t0);
        __syncthreads();
        for (uint32_t j = tid; j < tc; j += SW_THREADS) {
            const int ix = s_lut_t[__ldg(p.t + t0 + j)];
            if (ix < 0) atomicMin(&s_first_bad_t, (unsigned long long)(t0 + j));
            s_tidx[j] = ix < 0 ? 0 : (uint8_t)ix;
        }
        __syncthreads();
        if (active && qlen > 0) {
            for (uint32_t j = 0; j < tc; ++j) {
                const int tj = s_tidx[j];
                const T *pcol = s_prof + (size_t)tj * ROWS * SW_THREADS + tid;
                T diag = GLOBAL ? edge : (T)0, up = GLOBAL ? edge + gap : (T)0;
                if (GLOBAL) edge += gap;
#pragma unroll
                for (int i = 0; i < ROWS; ++i) {
                    const T old = col[i];                                    // H[i][j-1]
                    const T sc = PROFILE ? pcol[i * SW_THREADS] : s_tab[qrow[i] + tj];  // align.go:188 / :126
                    T v;
                    if (GLOBAL) {
                        v = addmax<T>(diag, sc, old + gap);                  // align.go:132-135 (no zero floor)
                        v = addmax<T>(up, gap, v);
                    } else {
                        v = addmax<T>(diag, sc, (T)0);                       // align.go:192,195
                        v = addmax<T>(old, gap, v);                          // left / up by orientation
                        v = addmax<T>(up, gap, v);
                        if (MASK) { if (i < (int)qlen) best = v > best ? v : best; }
                        else best = v > best ? v : best;                     // align.go:197-201
                    }
                    diag = old;
                    up = v;
                    col[i] = v;
                }
            }
        }
    }
    if (GLOBAL) {  // matrix[la][lb] (align.go:166); la == 0 or lb == 0: a pure gap ramp
        best = (T)p.tlen * gap;
#pragma unroll
        for (int i = 0; i < ROWS; ++i)
            if (i + 1 == (int)qlen) best = p.tlen ? col[i] : (T)qlen * gap;
    }
    __syncthreads();
    if (!active) return;
    const int64_t bad_t = s_first_bad_t == ~0ull ? -1 : (int64_t)s_first_bad_t;
    int32_t ec = 0;
    int64_t ep = -1;
    if (qlen > 0 && p.tlen > 0) {
        // first failing cell in row-major order, stringA outer (align.go:186-191);
        // Encode(a) is tried before Encode(b) (matrix.go:29-36)
        const int64_t bad_a = p.query_is_a ? first_bad_q : bad_t;
        const int64_t bad_b = p.query_is_a ? bad_t : first_bad_q;
        if (bad_a == 0) { ec = 1; ep = 0; }
        else if (bad_b >= 0) { ec = 2; ep = bad_b; }
        else if (bad_a > 0) { ec = 1; ep = bad_a; }
    }
    score[qi] = ec ? 0 : (int64_t)best;
    if (err) err[qi] = ec;
    if (errpos) errpos[qi] = ep;
}

// Two queries per thread, packed as 2 x int16 in one register (DPX __viaddmax_s16x2): the same four
// ALU-pipe instructions per DP step now advance TWO cells, doubling the issue-bound cell rate of the
// 32-bit kernel.  Used for Smith-Waterman (local) scores with gap <= 0 when every DP value provably fits
// 15 bits (host check) and the query profile fits shared memory.  Thread t owns queries 2t and 2t+1 of its
// block; the profile word prof[sym][row][thread] holds S(qA_row, sym) in the low and S(qB_row, sym) in the
// high half.  Rows at or beyond a query's length score -16384, which the zero floor of align.go:192-195
// turns into 0: such cells never exceed a real cell and never feed one (a cell only depends on smaller rows).
constexpr int SW16_NEG = -16384;

__device__ __forceinline__ uint32_t pack16(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }

template <int ROWS>
__global__ void __launch_bounds__(SW_THREADS)
sw_score_x2_kernel(SwParams p, const int16_t *__restrict__ lut_q, const int16_t *__restrict__ lut_t,
                   const int *__restrict__ tab, int gap, int64_t *__restrict__ score,
                   int32_t *__restrict__ err, int64_t *__restrict__ errpos) {
    extern __shared__ __align__(16) uint8_t sm[];
    // layout: [s_tidx: SW_TCHUNK bytes][s_lut_t: 256 int16][s_tab: n_q*n_t int][prof: n_t*ROWS*threads u32]
    uint8_t *s_tidx = sm;
    int16_t *s_lut_t = reinterpret_cast<int16_t *>(sm + SW_TCHUNK);
    int *s_tab = reinterpret_cast<int *>(sm + SW_TCHUNK + 512);
    uint32_t *s_prof = reinterpret_cast<uint32_t *>(s_tab + p.n_q * p.n_t);
    __shared__ unsigned long long s_first_bad_t;

    const uint32_t tid = threadIdx.x;
    for (int i = tid; i < p.n_q * p.n_t; i += SW_THREADS) s_tab[i] = tab[i];
    for (int i = tid; i < 256; i += SW_THREADS) s_lut_t[i] = lut_t[i];
    if (tid == 0) s_first_bad_t = ~0ull;
    __syncthreads();

    const uint64_t q0 = ((uint64_t)blockIdx.x * SW_THREADS + tid) * 2;
    uint64_t qbeg[2] = {0, 0};
    uint32_t qlen[2] = {0, 0};
    int64_t first_bad_q[2] = {-1, -1};
#pragma unroll
    for (int h = 0; h < 2; ++h)
        if (q0 + h < p.nq) {
            qbeg[h] = p.qoff[q0 + h];
            qlen[h] = (uint32_t)(p.qoff[q0 + h + 1] - qbeg[h]);
        }
    // expand the packed profile: row i of query h scores through table row lut_q[q_h[i]] (row 0 for a bad symbol,
    // reported at the end), -16384 beyond the query
    for (int i = 0; i < ROWS; ++i) {
        int row[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            row[h] = -1;
            if (i < (int)qlen[h]) {
                const int ix = lut_q[__ldg(p.q + qbeg[h] + i)];
                if (ix < 0) { if (first_bad_q[h] < 0) first_bad_q[h] = i; row[h] = 0; }
                else row[h] = ix * p.n_t;
            }
        }
        for (int t = 0; t < p.n_t; ++t)
            s_prof[(t * ROWS + i) * SW_THREADS + tid] = pack16(row[0] < 0 ? SW16_NEG : s_tab[row[0] + t], row[1] < 0 ? SW16_NEG : s_tab[row[1] + t]);
    }
    uint32_t col[ROWS];
#pragma unroll
    for (int i = 0; i < ROWS; ++i) col[i] = 0u;
    uint32_t best = 0u;
    const uint32_t gap2 = pack16(gap, gap);

    for (uint64_t t0 = 0; t0 < p.tlen; t0 += SW_TCHUNK) {
        const uint32_t tc = (uint32_t)min((uint64_t)SW_TCHUNK, p.tlen - t0);
        __syncthreads();
        for (uint32_t j = tid; j < tc; j += SW_THREADS) {
            const int ix = s_lut_t[__ldg(p.t + t0 + j)];
            if (ix < 0) atomicMin(&s_first_bad_t, (unsigned long long)(t0 + j));
            s_tidx[j] = ix < 0 ? 0 : (uint8_t)ix;
        }
        __syncthreads();
        if (qlen[0] | qlen[1]) {
            for (uint32_t j = 0; j < tc; ++j) {
                const uint32_t *pcol = s_prof + (size_t)s_tidx[j] * ROWS * SW_THREADS + tid;
                uint32_t diag = 0u, up = 0u;
#pragma unroll
                for (int i = 0; i < ROWS; ++i) {
                    const uint32_t old = col[i];                             // H[i][j-1] of both queries
                    uint32_t v = __viaddmax_s16x2(diag, pcol[i * SW_THREADS], 0u);  // align.go:192,195
                    v = __viaddmax_s16x2(old, gap2, v);
                    v = __viaddmax_s16x2(up, gap2, v);
                    best = __vmaxs2(best, v);                                // align.go:197-201
                    diag = old;
                    up = v;
                    col[i] = v;
                }
            }
        }
    }
    __syncthreads();
    const int64_t bad_t = s_first_bad_t == ~0ull ? -1 : (int64_t)s_first_bad_t;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        if (q0 + h >= p.nq) continue;
        int32_t ec = 0;
        int64_t ep = -1;
        if (qlen[h] > 0 && p.tlen > 0) {
            const int64_t bad_a = p.query_is_a ? first_bad_q[h] : bad_t;
            const int64_t bad_b = p.query_is_a ? bad_t : first_bad_q[h];
            if (bad_a == 0) { ec = 1; ep = 0; }
            else if (bad_b >= 0) { ec = 2; ep = bad_b; }
            else if (bad_a > 0) { ec = 1; ep = bad_a; }
        }
        const int b16 = (int)(int16_t)(h ? (best >> 16) : (best & 0xffffu));
        score[q0 + h] = ec ? 0 : (int64_t)b16;
        if (err) err[q0 + h] = ec;
        if (errpos) errpos[q0 + h] = ep;
    }
}

// Long queries: same recurrence, DP column in global scratch laid out [cell][query]
// so that a warp's accesses coalesce.
template <typename T>
__global__ void __launch_bounds__(SW_THREADS)
sw_score_long_kernel(SwParams p, uint64_t q_first, const int16_t *__restrict__ lut_q,
                     const int16_t *__restrict__ lut_t, const T *__restrict__ tab, T gap,
                     T *__restrict__ scratch, uint64_t n_batch, int64_t *__restrict__ score,
                     int32_t *__restrict__ err, int64_t *__restrict__ errpos) {
    const uint64_t b = (uint64_t)blockIdx.x * SW_THREADS + threadIdx.x;
    if (b >= n_batch) return;
    const uint64_t qi = q_first + b;
    const uint64_t qbeg = p.qoff[qi];
    const uint64_t qlen = p.qoff[qi + 1] - qbeg;
    int64_t first_bad_q = -1, bad_t = -1;
    for (uint64_t i = 0; i < qlen; ++i) {
        scratch[i * n_batch + b] = p.global ? (T)(i + 1) * gap : (T)0;
        if (first_bad_q < 0 && lut_q[__ldg(p.q + qbeg + i)] < 0) first_bad_q = (int64_t)i;
    }
    T best = 0, edge = 0;
    for (uint64_t j = 0; j < p.tlen; ++j) {
        const int tj = lut_t[__ldg(p.t + j)];
        if (tj < 0 && bad_t < 0) bad_t = (int64_t)j;
        T diag = p.global ? edge : (T)0, up = p.global ? edge + gap : (T)0;
        edge += gap;
        for (uint64_t i = 0; i < qlen; ++i) {
            const int qx = lut_q[__ldg(p.q + qbeg + i)];
            const T old = scratch[i * n_batch + b];
            const T sc = (qx < 0 || tj < 0) ? (T)0 : tab[qx * p.n_t + tj];
            T v;
            if (p.global) {
                v = addmax<T>(diag, sc, old + gap);
                v = addmax<T>(up, gap, v);
            } else {
                v = addmax<T>(diag, sc, (T)0);
                v = addmax<T>(old, gap, v);
                v = addmax<T>(up, gap, v);
                best = v > best ? v : best;
            }
            diag = old;
            up = v;
            scratch[i * n_batch + b] = v;
        }
    }
    if (p.global) best = qlen == 0 ? (T)p.tlen * gap : (p.tlen == 0 ? (T)qlen * gap : scratch[(qlen - 1) * n_batch + b]);
    int32_t ec = 0;
    int64_t ep = -1;
    if (qlen > 0 && p.tlen > 0) {
        const int64_t bad_a = p.query_is_a ? first_bad_q : bad_t;
        const int64_t bad_b = p.query_is_a ? bad_t : first_bad_q;
        if (bad_a == 0) { ec = 1; ep = 0; }
        else if (bad_b >= 0) { ec = 2; ep = bad_b; }
        else if (bad_a > 0) { ec = 1; ep = bad_a; }
    }
    score[qi] = ec ? 0 : (int64_t)best;
    if (err) err[qi] = ec;
    if (errpos) errpos[qi] = ep;
}

template <typename T>
int run_sw(const SwParams &p, uint64_t max_qlen, const int16_t *h_lut_q, const int16_t *h_lut_t,
           const std::vector<int64_t> &tab_qt, int64_t gap, int64_t *d_score, int32_t *d_err,
           int64_t *d_errpos, cudaStream_t st, bool x2_ok = false) {
    // small parameter block: LUTs + table (query symbol major)
    const size_t ntab = (size_t)p.n_q * p.n_t;
    std::vector<uint8_t> blob(512 * 2 + ntab * sizeof(T));
    memcpy(blob.data(), h_lut_q, 512);
    memcpy(blob.data() + 512, h_lut_t, 512);
    T *ht = reinterpret_cast<T *>(blob.data() + 1024);
    for (size_t i = 0; i < ntab; ++i) ht[i] = (T)tab_qt[i];
    uint8_t *d_blob = nullptr;
    PG_CUDA(cudaMallocAsync(&d_blob, blob.size(), st));
    PG_CUDA(cudaMemcpyAsync(d_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice, st));
    PG_CUDA(cudaStreamSynchronize(st));  // blob is a stack-lifetime host buffer
    const int16_t *d_lut_q = reinterpret_cast<const int16_t *>(d_blob);
    const int16_t *d_lut_t = d_lut_q + 256;
    const T *d_tab = reinterpret_cast<const T *>(d_blob + 1024);

    const size_t base_smem = SW_TCHUNK + 512 + (ntab + p.n_t) * sizeof(T);
    const unsigned blocks = (unsigned)((p.nq + SW_THREADS - 1) / SW_THREADS);
    int rc = PG_OK;
    const bool mask = gap > 0;
    bool launched = false;
    // smallest instantiated row count that covers the longest query
    auto try_rows = [&](auto rows_tag) -> bool {
        constexpr int ROWS = decltype(rows_tag)::value;
        if (launched || max_qlen > (uint64_t)ROWS) return false;
        const size_t prof = (size_t)p.n_t * ROWS * SW_THREADS * sizeof(T);
        const bool profile = base_smem + prof <= 100 * 1024;
        const size_t smem = base_smem + (profile ? prof : 0);
        if (smem > 200 * 1024) return false;
#define PG_SW_LAUNCH(PROF, MSK, GLB)                                                                     \
        do {                                                                                                 \
            cudaFuncSetAttribute(sw_score_kernel<T, ROWS, PROF, MSK, GLB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
            sw_score_kernel<T, ROWS, PROF, MSK, GLB><<<blocks, SW_THREADS, smem, st>>>(p, d_lut_q, d_lut_t, d_tab, (T)gap, d_score, d_err, d_errpos); \
        } while (0)
        if (p.global) { if (profile) PG_SW_LAUNCH(true, false, true); else PG_SW_LAUNCH(false, false, true); }
        else if (profile && !mask) PG_SW_LAUNCH(true, false, false);
        else if (profile && mask) PG_SW_LAUNCH(true, true, false);
        else if (!profile && !mask) PG_SW_LAUNCH(false, false, false);
        else PG_SW_LAUNCH(false, true, false);
#undef PG_SW_LAUNCH
        note_launch(p.global ? "nw_score_kernel" : "sw_score_kernel");
        launched = true;
        return true;
    };
    // packed 2 x int16 kernel: local alignment, gap <= 0, every DP value < 2^14 (checked by the caller: x2_ok)
    auto try_x2 = [&](auto rows_tag) -> bool {
        constexpr int ROWS = decltype(rows_tag)::value;
        if (launched || max_qlen > (uint64_t)ROWS) return false;
        const size_t smem = SW_TCHUNK + 512 + ntab * sizeof(int) + (size_t)p.n_t * ROWS * SW_THREADS * sizeof(uint32_t);
        if (smem > 100 * 1024) return false;
        cudaFuncSetAttribute(sw_score_x2_kernel<ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        sw_score_x2_kernel<ROWS><<<(unsigned)((p.nq + 2 * SW_THREADS - 1) / (2 * SW_THREADS)), SW_THREADS, smem, st>>>(
            p, d_lut_q, d_lut_t, reinterpret_cast<const int *>(d_tab), (int)gap, d_score, d_err, d_errpos);
        note_launch("sw_score_x2_kernel");
        launched = true;
        return true;
    };
    if (sizeof(T) == 4 && x2_ok) {
        try_x2(std::integral_constant<int, 8>{});
        try_x2(std::integral_constant<int, 16>{});
        try_x2(std::integral_constant<int, 24>{});
        try_x2(std::integral_constant<int, 28>{});
        try_x2(std::integral_constant<int, 32>{});
    }
    if (sizeof(T) == 4) {
        try_rows(std::integral_constant<int, 8>{});
        try_rows(std::integral_constant<int, 16>{});
        try_rows(std::integral_constant<int, 20>{});
        try_rows(std::integral_constant<int, 24>{});
        try_rows(std::integral_constant<int, 28>{});
        try_rows(std::integral_constant<int, 32>{});
        try_rows(std::integral_constant<int, 40>{});
        try_rows(std::integral_constant<int, 48>{});
        try_rows(std::integral_constant<int, 64>{});
    } else {
        try_rows(std::integral_constant<int, 32>{});
        try_rows(std::integral_constant<int, 64>{});
    }
    if (launched) {
    } else {
        // batches bounded by a 1 GiB scratch column store
        uint64_t per = std::max<uint64_t>(1, (1ull << 30) / (std::max<uint64_t>(max_qlen, 1) * sizeof(T)));
        per = std::min<uint64_t>(per, p.nq);
        T *d_scr = nullptr;
        PG_CUDA(cudaMallocAsync(&d_scr, per * std::max<uint64_t>(max_qlen, 1) * sizeof(T), st));
        for (uint64_t q0 = 0; q0 < p.nq; q0 += per) {
            const uint64_t nb = std::min<uint64_t>(per, p.nq - q0);
            sw_score_long_kernel<T><<<(unsigned)((nb + SW_THREADS - 1) / SW_THREADS), SW_THREADS, 0, st>>>(
                p, q0, d_lut_q, d_lut_t, d_tab, (T)gap, d_scr, nb, d_score, d_err, d_errpos);
            note_launch("sw_score_long_kernel");
        }
        cudaFreeAsync(d_scr, st);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = cuda_fail(e, "sw_score launch", __FILE__, __LINE__);
    cudaFreeAsync(d_blob, st);
    return rc;
}

}  // namespace

int launch_sw_score(const uint8_t *d_q, const uint64_t *d_qoff, uint64_t nq, uint64_t max_qlen,
                    const uint8_t *d_t, uint64_t tlen, int query_is_a, const int16_t *lut_a,
                    const int16_t *lut_b, const int64_t *table, int n_a, int n_b, int64_t gap,
                    int64_t *d_score, int32_t *d_err, int64_t *d_errpos, cudaStream_t st, int global) {
    if (nq == 0) return PG_OK;
    if (n_a <= 0 || n_b <= 0 || n_a > 255 || n_b > 255) {
        set_error("alphabet sizes must be in 1..255 (got %d, %d)", n_a, n_b);
        return PG_ERR_ARG;
    }
    SwParams p;
    p.q = d_q; p.qoff = d_qoff; p.nq = nq; p.t = d_t; p.tlen = tlen; p.query_is_a = query_is_a;
    p.global = global;
    p.n_q = query_is_a ? n_a : n_b;
    p.n_t = query_is_a ? n_b : n_a;
    const int16_t *lut_q = query_is_a ? lut_a : lut_b;
    const int16_t *lut_t = query_is_a ? lut_b : lut_a;
    // table with the query symbol as the row: tab_qt[q][t] = S(a, b) in either orientation
    std::vector<int64_t> tab_qt((size_t)p.n_q * p.n_t);
    int64_t amax = 0;
    for (int q = 0; q < p.n_q; ++q)
        for (int t = 0; t < p.n_t; ++t) {
            const int64_t v = query_is_a ? table[(size_t)q * n_b + t] : table[(size_t)t * n_b + q];
            tab_qt[(size_t)q * p.n_t + t] = v;
            amax = std::max<int64_t>(amax, v < 0 ? -v : v);
        }
    const int64_t agap = gap < 0 ? -gap : gap;
    // every DP value lies in [0, min(la,lb) * max S]; operands of one add stay below
    // that plus max(|S|,|gap|): use 32-bit DPX arithmetic when this provably fits
    // (NW: every value lies within (la + lb) * max(|S|, |gap|))
    const long double bound = global ? (long double)std::max(amax, agap) * (long double)(max_qlen + tlen + 2)
                                     : (long double)amax * (long double)std::min<uint64_t>(max_qlen, tlen) +
                                           (long double)std::max(amax, agap);
    if (bound < 2.0e9L) {
        // two queries per register (2 x int16) when a local alignment's values stay below 2^14 and gap <= 0
        const bool x2_ok = !global && gap <= 0 && bound < 16000.0L && agap < 16000 && nq >= 2;
        return run_sw<int>(p, max_qlen, lut_q, lut_t, tab_qt, gap, d_score, d_err, d_errpos, st, x2_ok);
    }
    return run_sw<long long>(p, max_qlen, lut_q, lut_t, tab_qt, gap, d_score, d_err, d_errpos, st);
}

}  // namespace pg
