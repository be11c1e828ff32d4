// spmm.cu -- Y = A X for a dense X of k columns (SpMM) on resident CSR and HLL matrices, sm_100a (B200).
//
// X is N x k and Y is M x k, both row-major with leading dimensions ldx, ldy >= k; element (i, c) at i*ld + c, every
// offset in 64 bits.  One product over all k columns streams row_ptr / col_idx / values (or the HLL slots) ONCE and
// gathers a contiguous row of X per nonzero, where k single-vector products stream the matrix k times (DESIGN.md
// section 3, "Multi-vector products": lane mapping, measurements, and the shapes where it loses at small k).
//
// Kernels:
//   * csr_spmm_kernel<KT,BATCH>  -- a group of KT lanes per row (KT in {1,2,4,8,16,32}, 32/KT rows per warp); lane c of a
//       group owns column c0 + c.  The lanes of a group load the same column index / value (one broadcast transaction),
//       gather KT contiguous doubles X[col*ldx + c0 .. c0+KT) and store a contiguous piece of Y's row.  Each lane sums its
//       (row, column) alone, in index order, mul and add rounded separately: column c is bit for bit the serial loop
//       (csr_row_kernel) on column c of X.  Rows above the plan's long_threshold are left to:
//   * csr_spmm_fragment_kernel + csr_spmm_combine_kernel -- the plan's long rows (A->long_rows / frag_first, fragments of
//       8192 nonzeros), one column tile of up to 32 columns per launch pair.  A fragment is cut into kSpmmSubRanges
//       fixed index-ordered sub-ranges, each summed serially, then added by a fixed binary tree; the combine adds the
//       fragments of a row in order.  The decomposition depends on the fragment only, never on the tile width, so the
//       bits of a column do not depend on k, ldx, ldy or where the column sits in X.  No atomics.
//   * hll_spmm_kernel<KT,BATCH>  -- the same lane mapping over the column-major HLL image: a warp covers 32/KT rows of a
//       hack, slot loads JA/AS[off + 32 j + r] are contiguous across those rows, j runs in order and the padding slots
//       (x 0.0) are included: column c is bit for bit spmv_hll_serial on column c (hll_row_kernel's order).
// Every kernel takes the storage type V of values, X and Y: double, or float for the copy of enable_f32 (the *_spmm_f32
// entry points).  Loads are widened to double, accumulators and fragment partials are double, and Y is rounded to V once.
#include <algorithm>

#include "common.cuh"
#include "handles.cuh"

namespace spmv {

constexpr int kSpmmThreads = 256;
constexpr int kSpmmTile = 32;        // columns per column tile (the widest group)
constexpr int kSpmmFragNnz = 8192;   // = kFragNnz of csr.cu: the fragments of the plan's long rows
constexpr int kSpmmSubRanges = 128;  // fixed sub-ranges of a fragment (64 nonzeros each), summed serially, then a tree
constexpr int kSpmmSubLen = kSpmmFragNnz / kSpmmSubRanges;
// Column / value loads in flight per lane before the first gather, per format.  Swept over {2, 4, 8} with
// tools/spmm_bench.py --batches on a B200 at 1000 W (profiles/r03a_spmm_batch_sweep.json): CSR 2 and 4 within 4 % of
// each other and 8 slower; HLL 8 fastest on lap2d and on uniform for k >= 8.  SPMV_B200_SPMM_BATCH in {2, 4, 8}
// overrides both (for such sweeps).  The fp32 products, swept the same way (profiles/r03e_spmm_f32_batch_sweep.json): CSR 2
// fastest on lap2d, on R-MAT and on uniform for k >= 8 (uniform k = 32: 9.03 ms against 11.20 at 4), within 7 % of 4
// elsewhere; HLL 8 fastest for k >= 2, as in fp64.
constexpr int kSpmmBatchCsr = 4;
constexpr int kSpmmBatchCsr32 = 2;
constexpr int kSpmmBatchHll = 8;

// Lanes per row for a tile of `cols` columns: the smallest power of two >= cols (cols <= 32).
static int spmm_group(int cols) {
    int kt = 1;
    while (kt < cols) kt <<= 1;
    return kt;
}

// HLL slot loads: with one lane per row a warp reads one contiguous 128 / 256 B slice, consumed at once -- no L1
// allocation.  With several lanes per row a sector is consumed by several warps, so it should stay in L1 in between
// (plain read-only loads).  The CSR kernel always allocates: each group walks its own row, as csr_row_kernel's lanes do.
template <int KT>
__device__ __forceinline__ int hll_load_col(const int *p) {
    if constexpr (KT == 1) return ldg_stream_s32(p);
    else return __ldg(p);
}
template <int KT, typename V>
__device__ __forceinline__ double hll_load_val(const V *p) {
    if constexpr (KT == 1) return ldg_stream_f64(p);
    else return (double)__ldg(p);
}

// grid.x: blocks of 256/KT rows; grid.y: column tiles of KT columns starting at c0 + 32*blockIdx.y (cols <= KT live lanes)
template <int KT, int BATCH, typename V>
__global__ void __launch_bounds__(kSpmmThreads)
csr_spmm_kernel(int M, const int *__restrict__ row_ptr, const int *__restrict__ col_idx, const V *__restrict__ values,
                int long_threshold, int c0, int cols, const V *__restrict__ X, long long ldx, V *__restrict__ Y,
                long long ldy, int accumulate) {
    const long long row = (long long)blockIdx.x * (kSpmmThreads / KT) + threadIdx.x / KT;
    const int c = (int)(threadIdx.x & (KT - 1));
    if (row >= M || c >= cols) return;
    const int lo = __ldg(row_ptr + row), hi = __ldg(row_ptr + row + 1);
    if (hi - lo > long_threshold) return;  // a long row of the plan: the fragment kernels own it
    const int col = c0 + kSpmmTile * (int)blockIdx.y + c;
    const V *__restrict__ xc = X + col;
    V *__restrict__ yp = Y + row * ldy + col;
    double acc = accumulate ? (double)*yp : 0.0;
    for (int k = lo; k < hi; k += BATCH) {
        int ci[BATCH];
        double v[BATCH], xv[BATCH];
#pragma unroll
        for (int u = 0; u < BATCH; ++u) ci[u] = k + u < hi ? __ldg(col_idx + k + u) : -1;
#pragma unroll
        for (int u = 0; u < BATCH; ++u) v[u] = k + u < hi ? (double)__ldg(values + k + u) : 0.0;
#pragma unroll
        for (int u = 0; u < BATCH; ++u) xv[u] = ci[u] >= 0 ? (double)__ldg(xc + (long long)ci[u] * ldx) : 0.0;
#pragma unroll
        for (int u = 0; u < BATCH; ++u)
            if (ci[u] >= 0) acc = __dadd_rn(acc, __dmul_rn(v[u], xv[u]));  // one lane, index order: the serial loop
    }
    *yp = (V)acc;
}

// One CTA per (fragment f, column tile of `cols` <= 32 columns at c0).  The (sub-range s, column c) pairs p = s * cols + c
// are dealt to the threads round-robin (p = t, t + 256, ...), so the lanes of a warp cover consecutive columns of one or
// a few sub-ranges (broadcast column / value loads, contiguous gathers) and a narrow tile still keeps 128 threads busy.
// Which thread sums a pair changes with cols; the sum itself does not.  partial[f * 32 + c] = tree over the sub-range
// sums of column c (in double whatever V is).
template <typename V>
__global__ void __launch_bounds__(kSpmmThreads)
csr_spmm_fragment_kernel(const int *__restrict__ long_rows, const int *__restrict__ frag_first, int num_long,
                         const int *__restrict__ row_ptr, const int *__restrict__ col_idx, const V *__restrict__ values,
                         int c0, int cols, const V *__restrict__ X, long long ldx, double *__restrict__ partial) {
    __shared__ double sub[kSpmmSubRanges][kSpmmTile];
    const int f = (int)blockIdx.x;
    int lo = 0, hi = num_long;  // last long row whose first fragment is <= f
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(frag_first + mid) <= f) lo = mid; else hi = mid;
    }
    const int row = __ldg(long_rows + lo);
    const long long begin = (long long)__ldg(row_ptr + row) + (long long)(f - __ldg(frag_first + lo)) * kSpmmFragNnz;
    const long long row_end = __ldg(row_ptr + row + 1);
    const long long end = begin + kSpmmFragNnz < row_end ? begin + kSpmmFragNnz : row_end;
    constexpr int kBatch = 4;
    for (int p = (int)threadIdx.x; p < kSpmmSubRanges * cols; p += kSpmmThreads) {
        const int s = p / cols, c = p - s * cols;
        const V *__restrict__ xc = X + c0 + c;
        const long long sb = begin + (long long)s * kSpmmSubLen;
        const long long se = sb + kSpmmSubLen < end ? sb + kSpmmSubLen : end;
        double acc = 0.0;
        {
            for (long long k = sb; k < se; k += kBatch) {
                int ci[kBatch];
                double v[kBatch], xv[kBatch];
#pragma unroll
                for (int u = 0; u < kBatch; ++u) ci[u] = k + u < se ? __ldg(col_idx + k + u) : -1;
#pragma unroll
                for (int u = 0; u < kBatch; ++u) v[u] = k + u < se ? (double)__ldg(values + k + u) : 0.0;
#pragma unroll
                for (int u = 0; u < kBatch; ++u) xv[u] = ci[u] >= 0 ? (double)__ldg(xc + (long long)ci[u] * ldx) : 0.0;
#pragma unroll
                for (int u = 0; u < kBatch; ++u)
                    if (ci[u] >= 0) acc = fma(v[u], xv[u], acc);
            }
        }
        sub[s][c] = acc;
    }
    // fixed binary tree over the sub-ranges: sub[s] += sub[s + h] for h = 64, 32, ..., 1
    for (int h = kSpmmSubRanges / 2; h > 0; h >>= 1) {
        __syncthreads();
        for (int i = (int)threadIdx.x; i < h * cols; i += kSpmmThreads) {
            const int s = i / cols, cc = i - s * cols;
            sub[s][cc] += sub[s + h][cc];
        }
    }
    __syncthreads();
    if (threadIdx.x < (unsigned)cols) partial[(long long)f * kSpmmTile + threadIdx.x] = sub[0][threadIdx.x];
}

// One thread per (long row, column of the tile): Y (or 0) plus the row's fragments, in order, rounded to V once.
template <typename V>
__global__ void csr_spmm_combine_kernel(const int *__restrict__ long_rows, const int *__restrict__ frag_first, int num_long,
                                        const double *__restrict__ partial, int c0, int cols, V *__restrict__ Y,
                                        long long ldy, int accumulate) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int i = (int)(t / kSpmmTile), c = (int)(t % kSpmmTile);
    if (i >= num_long || c >= cols) return;
    V *yp = Y + (long long)long_rows[i] * ldy + c0 + c;
    double acc = accumulate ? (double)*yp : 0.0;
    for (int f = frag_first[i]; f < frag_first[i + 1]; ++f) acc += partial[(long long)f * kSpmmTile + c];  // fixed order
    *yp = (V)acc;
}

// grid.x: blocks of 256/KT rows of the padded image (num_hacks * 32 rows); grid.y: column tiles as csr_spmm_kernel
template <int KT, int BATCH, typename V>
__global__ void __launch_bounds__(kSpmmThreads)
hll_spmm_kernel(int M, int num_hacks, const long long *__restrict__ hack_off, const int *__restrict__ JA,
                const V *__restrict__ AS, int c0, int cols, const V *__restrict__ X, long long ldx,
                V *__restrict__ Y, long long ldy) {
    const long long prow = (long long)blockIdx.x * (kSpmmThreads / KT) + threadIdx.x / KT;  // row of the padded image
    const int c = (int)(threadIdx.x & (KT - 1));
    const int hack = (int)(prow >> 5), r = (int)(prow & 31);
    if (hack >= num_hacks || c >= cols) return;
    const long long off = __ldg(hack_off + hack);
    const int width = (int)((__ldg(hack_off + hack + 1) - off) >> 5);
    const long long base = off + r;
    const int col = c0 + kSpmmTile * (int)blockIdx.y + c;
    const V *__restrict__ xc = X + col;
    double acc = 0.0;
    for (int j = 0; j < width; j += BATCH) {
        int ci[BATCH];
        double v[BATCH], xv[BATCH];
#pragma unroll
        for (int u = 0; u < BATCH; ++u) ci[u] = j + u < width ? hll_load_col<KT>(JA + base + (long long)(j + u) * 32) : -1;
#pragma unroll
        for (int u = 0; u < BATCH; ++u) v[u] = j + u < width ? hll_load_val<KT>(AS + base + (long long)(j + u) * 32) : 0.0;
#pragma unroll
        for (int u = 0; u < BATCH; ++u) xv[u] = ci[u] >= 0 ? (double)__ldg(xc + (long long)ci[u] * ldx) : 0.0;
#pragma unroll
        for (int u = 0; u < BATCH; ++u)
            if (ci[u] >= 0) acc = __dadd_rn(acc, __dmul_rn(v[u], xv[u]));  // padding slots included: 0.0 * x
    }
    if (prow < M) Y[prow * ldy + col] = (V)acc;
}

static int spmm_batch(int fallback) {
    const int b = env_int("SPMV_B200_SPMM_BATCH", fallback);
    return b == 2 || b == 4 || b == 8 ? b : fallback;
}

// Column tiles of a k-column product: k / 32 full tiles of 32 columns (one launch, grid.y = tiles), then one launch for
// the remaining k % 32 columns at c0 = 32 * (k / 32) with the smallest group that covers them.
template <class Launch>
static int spmm_tiles(int k, Launch launch) {
    const int full = k / kSpmmTile, rest = k % kSpmmTile;
    if (full > 0) SPMV_TRY(launch(kSpmmTile, 0, kSpmmTile, full));
    if (rest > 0) SPMV_TRY(launch(spmm_group(rest), full * kSpmmTile, rest, 1));
    return SPMV_B200_OK;
}

// kernel<KT, batch> for a run-time group width and batch
template <template <int, int> class K, class... Args>
static int spmm_dispatch(int kt, int batch, Args... args) {
    switch (kt) {
        case 1: return K<1, 4>::pick(batch, args...);
        case 2: return K<2, 4>::pick(batch, args...);
        case 4: return K<4, 4>::pick(batch, args...);
        case 8: return K<8, 4>::pick(batch, args...);
        case 16: return K<16, 4>::pick(batch, args...);
        case 32: return K<32, 4>::pick(batch, args...);
        default: return fail(SPMV_B200_ERR_INVALID, "spmm: bad group width %d", kt);
    }
}

template <int KT, int>
struct CsrSpmmLaunch {
    template <class... Args>
    static int pick(int batch, dim3 grid, cudaStream_t stream, Args... args) {
        if (batch == 2) csr_spmm_kernel<KT, 2><<<grid, kSpmmThreads, 0, stream>>>(args...);
        else if (batch == 8) csr_spmm_kernel<KT, 8><<<grid, kSpmmThreads, 0, stream>>>(args...);
        else csr_spmm_kernel<KT, 4><<<grid, kSpmmThreads, 0, stream>>>(args...);
        SPMV_TRY_CUDA(cudaGetLastError());
        return SPMV_B200_OK;
    }
};

template <int KT, int>
struct HllSpmmLaunch {
    template <class... Args>
    static int pick(int batch, dim3 grid, cudaStream_t stream, Args... args) {
        if (batch == 2) hll_spmm_kernel<KT, 2><<<grid, kSpmmThreads, 0, stream>>>(args...);
        else if (batch == 8) hll_spmm_kernel<KT, 8><<<grid, kSpmmThreads, 0, stream>>>(args...);
        else hll_spmm_kernel<KT, 4><<<grid, kSpmmThreads, 0, stream>>>(args...);
        SPMV_TRY_CUDA(cudaGetLastError());
        return SPMV_B200_OK;
    }
};

int check_spmm_args(const char *what, const void *h, int k, const void *X, long long ldx, const void *Y,
                           long long ldy) {
    if (k < 0) return fail(SPMV_B200_ERR_INVALID, "%s: negative k (%d)", what, k);
    if (ldx < k || ldy < k)
        return fail(SPMV_B200_ERR_INVALID, "%s: leading dimensions must be >= k (k=%d ldx=%lld ldy=%lld)", what, k, ldx, ldy);
    if (k > 0 && (!h || !X || !Y)) return fail(SPMV_B200_ERR_INVALID, "%s: NULL argument", what);
    return SPMV_B200_OK;
}

// The products behind the entry points (arguments checked, k > 0, M > 0): V = double on the fp64 values, V = float on
// the copy of enable_f32; every sum is formed in double either way.  The host-buffer products (hostpath.cu) run the same
// launches window by window: csr_spmm_rows on rows [r0, r1) (the long rows left out, as the kernel does everywhere) and
// csr_spmm_long for the long rows, hll_spmm_hacks on hacks [h0, h1).  X and Y point at row 0 of the matrix.
template <typename V>
int csr_spmm_rows(const spmv_b200_csr *A, const V *values, long long r0, long long r1, int k, const V *d_X, long long ldx,
                  V *d_Y, long long ldy, int accumulate, cudaStream_t stream) {
    const int batch = spmm_batch(sizeof(V) == 4 ? kSpmmBatchCsr32 : kSpmmBatchCsr);
    const int M = (int)(r1 - r0);
    const int acc = accumulate ? 1 : 0;
    if (M <= 0) return SPMV_B200_OK;
    return spmm_tiles(k, [&](int kt, int c0, int cols, int tiles) {
        const dim3 grid(blocks_for(M, kSpmmThreads / kt), (unsigned)tiles);
        return spmm_dispatch<CsrSpmmLaunch>(kt, batch, grid, stream, M, (const int *)(A->row_ptr + r0), (const int *)A->col_idx,
                                            values, A->long_threshold, c0, cols, d_X, ldx, d_Y + r0 * ldy, ldy, acc);
    });
}

template <typename V>
int csr_spmm_long(const spmv_b200_csr *A, const V *values, int k, const V *d_X, long long ldx, V *d_Y, long long ldy,
                  int accumulate, cudaStream_t stream) {
    if (A->num_long == 0) return SPMV_B200_OK;
    const int acc = accumulate ? 1 : 0;
    // one fragment + combine launch pair per column tile, through the handle's partials buffer
    if (!A->spmm_partial) SPMV_TRY_CUDA(cudaMalloc(&A->spmm_partial, (size_t)A->num_frag * kSpmmTile * sizeof(double)));
    for (int c0 = 0; c0 < k; c0 += kSpmmTile) {
        const int cols = std::min(kSpmmTile, k - c0);
        csr_spmm_fragment_kernel<V><<<A->num_frag, kSpmmThreads, 0, stream>>>(A->long_rows, A->frag_first, A->num_long,
                                                                               A->row_ptr, A->col_idx, values, c0, cols,
                                                                               d_X, ldx, A->spmm_partial);
        SPMV_TRY_CUDA(cudaGetLastError());
        csr_spmm_combine_kernel<V><<<blocks_for((long long)A->num_long * kSpmmTile, 128), 128, 0, stream>>>(
            A->long_rows, A->frag_first, A->num_long, A->spmm_partial, c0, cols, d_Y, ldy, acc);
        SPMV_TRY_CUDA(cudaGetLastError());
    }
    return SPMV_B200_OK;
}

template <typename V>
static int csr_spmm(const spmv_b200_csr *A, const V *values, int k, const V *d_X, long long ldx, V *d_Y, long long ldy,
                    int accumulate, cudaStream_t stream) {
    SPMV_TRY(csr_spmm_rows(A, values, 0, A->M, k, d_X, ldx, d_Y, ldy, accumulate, stream));
    return csr_spmm_long(A, values, k, d_X, ldx, d_Y, ldy, accumulate, stream);
}

template <typename V>
int hll_spmm_hacks(const spmv_b200_hll *H, const V *AS, int h0, int h1, int k, const V *d_X, long long ldx, V *d_Y,
                   long long ldy, cudaStream_t stream) {
    const int batch = spmm_batch(kSpmmBatchHll);
    const int hacks = h1 - h0;
    if (hacks <= 0) return SPMV_B200_OK;
    const int M = (int)(std::min<long long>(H->M, 32LL * h1) - 32LL * h0);
    const long long rows = (long long)hacks * 32;
    return spmm_tiles(k, [&](int kt, int c0, int cols, int tiles) {
        const dim3 grid(blocks_for(rows, kSpmmThreads / kt), (unsigned)tiles);
        return spmm_dispatch<HllSpmmLaunch>(kt, batch, grid, stream, M, hacks, (const long long *)(H->hack_off + h0),
                                            (const int *)H->JA, AS, c0, cols, d_X, ldx, d_Y + 32LL * h0 * ldy, ldy);
    });
}

template <typename V>
static int hll_spmm(const spmv_b200_hll *H, const V *AS, int k, const V *d_X, long long ldx, V *d_Y, long long ldy,
                    cudaStream_t stream) {
    return hll_spmm_hacks(H, AS, 0, H->num_hacks, k, d_X, ldx, d_Y, ldy, stream);
}

#define SPMV_SPMM_WINDOWS(V)                                                                                                \
    template int csr_spmm_rows<V>(const spmv_b200_csr *, const V *, long long, long long, int, const V *, long long, V *,   \
                                  long long, int, cudaStream_t);                                                            \
    template int csr_spmm_long<V>(const spmv_b200_csr *, const V *, int, const V *, long long, V *, long long, int,         \
                                  cudaStream_t);                                                                            \
    template int hll_spmm_hacks<V>(const spmv_b200_hll *, const V *, int, int, int, const V *, long long, V *, long long,   \
                                   cudaStream_t);
SPMV_SPMM_WINDOWS(double)
SPMV_SPMM_WINDOWS(float)
#undef SPMV_SPMM_WINDOWS

}  // namespace spmv

using namespace spmv;

extern "C" {

int spmv_b200_csr_spmm(const spmv_b200_csr *A, int k, const double *d_X, long long ldx, double *d_Y, long long ldy,
                       int accumulate, void *stream) {
    SPMV_TRY(check_spmm_args("csr_spmm", A, k, d_X, ldx, d_Y, ldy));
    if (k == 0 || A->M == 0) return SPMV_B200_OK;
    return csr_spmm(A, (const double *)A->values, k, d_X, ldx, d_Y, ldy, accumulate, as_stream(stream));
}

int spmv_b200_csr_spmm_f32(const spmv_b200_csr *A, int k, const float *d_X, long long ldx, float *d_Y, long long ldy,
                           int accumulate, void *stream) {
    SPMV_TRY(check_spmm_args("csr_spmm_f32", A, k, d_X, ldx, d_Y, ldy));
    if (A && !A->values32) return fail(SPMV_B200_ERR_INVALID, "csr_spmm_f32: call spmv_b200_csr_enable_f32 first");
    if (k == 0 || A->M == 0) return SPMV_B200_OK;
    return csr_spmm(A, (const float *)A->values32, k, d_X, ldx, d_Y, ldy, accumulate, as_stream(stream));
}

int spmv_b200_hll_spmm(const spmv_b200_hll *H, int k, const double *d_X, long long ldx, double *d_Y, long long ldy,
                       void *stream) {
    SPMV_TRY(check_spmm_args("hll_spmm", H, k, d_X, ldx, d_Y, ldy));
    if (k == 0 || H->M == 0 || H->num_hacks == 0) return SPMV_B200_OK;
    return hll_spmm(H, (const double *)H->AS, k, d_X, ldx, d_Y, ldy, as_stream(stream));
}

int spmv_b200_hll_spmm_f32(const spmv_b200_hll *H, int k, const float *d_X, long long ldx, float *d_Y, long long ldy,
                           void *stream) {
    SPMV_TRY(check_spmm_args("hll_spmm_f32", H, k, d_X, ldx, d_Y, ldy));
    if (H && !H->AS32) return fail(SPMV_B200_ERR_INVALID, "hll_spmm_f32: call spmv_b200_hll_enable_f32 first");
    if (k == 0 || H->M == 0 || H->num_hacks == 0) return SPMV_B200_OK;
    return hll_spmm(H, (const float *)H->AS32, k, d_X, ldx, d_Y, ldy, as_stream(stream));
}

}  // extern "C"
