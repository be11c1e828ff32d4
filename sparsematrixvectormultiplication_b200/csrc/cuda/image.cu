// image.cu -- the private image of a CSR handle: a second copy of a short-row matrix that ALGO_ROW_IMAGE and AUTO
// multiply, bit for bit like csr_row_kernel.  It is chosen at plan time (image_candidates, image_keep) or asked for by
// spmv_b200_csr_set_image (image_build), and held in one of two forms:
//  * column-major: hll.cu's layout with the padding slots marked and a column field of 2 bytes (col - row, when every
//    column lies within 2^14 of its row) or 4; fp64 values, or 1-byte codes into a table of at most kMaxDistinct values.
//  * patterns: one byte per row naming the row's pattern.  On stencils, structured-grid FEM and unit-weight banded
//    matrices whole rows repeat: a row's pattern -- its length, the col - row of each slot and the 64-bit pattern of each
//    value -- takes 9 distinct forms on lap2d (interior, 4 edges, 4 corners) and 27 on lap3d.  When the matrix holds at
//    most kMaxDistinct of them, the product streams the pattern id instead of a column field and a value field per slot:
//    CSR-VI (Kourtis et al.) applied to whole rows.  The dictionary (value[W][P], delta[W][P], len[P]; slot-major, so lanes
//    of different patterns read different banks) is staged in shared memory.  lap2d 4096^2: 16.8 MB of ids and 540 B of
//    dictionary, against 252 MB for the coded column-major form.
// This module decides which forms exist, which are built, under which limits, and which kernel runs the one held.
#include <algorithm>
#include <cstring>
#include <new>
#include <numeric>
#include <vector>

#include "common.cuh"
#include "handles.cuh"

namespace spmv {

constexpr int kMaxDistinct = 256;                // value patterns of the coded form, row patterns of the pattern form
constexpr int kPatternDictMaxBytes = 24 * 1024;  // P * W * 12: 8 CTAs of 256 threads stay resident per SM

// The tiled pattern kernel (csr_pattern_tile_kernel): a CTA of kTileThreads threads multiplies kTileRows rows from windows
// of x staged in shared memory, one window per cluster of the patterns' deltas
constexpr int kTileRows = 1024;     // 4 rows per thread, strided by kTileThreads: consecutive lanes read consecutive words
constexpr int kTileThreads = 256;
constexpr int kWindowGap = 32;      // sorted deltas less than this apart share a window
constexpr int kWindowMaxSpan = 256; // hi - lo of one window: a window stages kTileRows + span + 2 doubles at most
// Slot records and windows: with the kTileRows ids, 8 CTAs (+ 1 KB reserved each) fit an SM's 228 KB, as the kernel needs
// all 2048 threads of an SM to hide its load phase.  Measured on lap3d 384^3 (B200): 5 windows (44 KB, 5 CTAs per SM)
// took 498 us against 422 us for csr_pattern_kernel, while lap2d's 3 windows (25 KB, 8 CTAs) gained.
constexpr int kWindowSmemMax = 26 * 1024;
constexpr int kMaxWindows = 3;      // and at most W; a fourth window of a 1024-row tile exceeds kWindowSmemMax

struct PatternWindows {
    int count = 0;                           // windows a tile stages; 0: csr_pattern_kernel gathers x from global memory
    int lo[kMaxWindows] = {}, hi[kMaxWindows] = {};  // the deltas each window covers
    int base[kMaxWindows + 1] = {};          // its first double in shared memory, after the slot records; base[count]: end
};

struct ImageForm {
    bool patterns = false;     // csr_pattern_tile_kernel<W> or csr_pattern_kernel<W>; otherwise the column-major form, run by
    bool offset_free = false;  // hll_rowu_kernel<batch> (regular layouts) or hll_row_kernel<batch>
    int batch = 0;
    bool coded = false;        // on the value codes, else on the fp64 values
};

struct ColumnImage {
    int num_hacks = 0, max_width = 0;
    long long slots = 0;
    HllSegments segments;
    long long *hack_off = nullptr;  // device [num_hacks + 1]
    int *JA = nullptr;              // device [slots]: the column, bit 31 marks padding; or
    uint16_t *JA16 = nullptr;       // device [slots]: the narrow field, col - row in bits 0-14, bit 15 marks padding
    double *AS = nullptr;           // device [slots]: fp64 values (padding 0.0), and/or
    uint8_t *AC = nullptr;          // device [slots]: codes into table (padding 0); during the plan both may be held
    double *table = nullptr;        // device [max(num_values, 1)]: the distinct 64-bit value patterns, ascending as uint64
    int num_values = 0;
};

struct CsrPatterns {
    int count = 0;          // P patterns, in the order of their (length, deltas, value bits)
    int width = 0;          // W: the matrix's longest row
    uint8_t *id = nullptr;  // device [M]: the pattern of each row
    int *dict = nullptr;    // device: value[W][P] (fp64), delta[W][P] (int32), len[P] (int32); a slot at or past a
                            // pattern's length holds delta 0 and value 0.0
    PatternWindows windows; // planned from the dictionary at build time
};
static long long dict_bytes(const CsrPatterns &P) { return 12LL * P.width * P.count + 4LL * P.count; }

struct CsrImage {
    explicit CsrImage(const spmv_b200_csr *A) : M(A->M), N(A->N) {}
    int M, N;
    ImageForm form;                     // the form the products run
    std::vector<ImageForm> candidates;  // plan time: every form built, in the plan's order
    ColumnImage cols;
    CsrPatterns patterns;
};

// ---- the product of the pattern form ---------------------------------------------------------------------------------
// One thread per row, straight-line code: the row's id, its W deltas from shared memory, all W gathers, then the adds of
// the slots below the pattern's length in slot order, mul and add rounded separately -- csr_row_kernel's order and
// operands (the dictionary holds the stored doubles), so y is bit for bit csr_row_kernel's for every x, accumulate from
// any y included (NaN payloads aside where two NaNs meet in one sum, as on the coded image).  A slot at or past the
// length holds delta 0 and gathers x[min(row, N - 1)]: no load is predicated on loaded data, and every gather stays in
// bounds when M > N (a real slot's column row + delta is below N already).  ACCUM: y[row] is loaded after the gathers,
// for the reason given at hll_rowu_kernel.
template <int W, bool ACCUM>
__global__ void __launch_bounds__(256, 8)
csr_pattern_kernel(int row_begin, int row_end, const uint8_t *__restrict__ id, const int *__restrict__ dict, int P,
                   const double *__restrict__ x, double *__restrict__ y, int N) {
    extern __shared__ double pattern_dict[];
    int *words = reinterpret_cast<int *>(pattern_dict);
    for (int i = threadIdx.x; i < (3 * W + 1) * P; i += blockDim.x) words[i] = __ldg(dict + i);
    __syncthreads();
    const double *value = pattern_dict;
    const int *delta = words + 2 * W * P, *len = delta + W * P;
    const long long r = row_begin + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= row_end) return;
    const int row = (int)r;
    const int p = ldg_stream_u8(id + row);
    double xv[W];
#pragma unroll
    for (int s = 0; s < W; ++s) xv[s] = ldg_x(x, min(row + delta[s * P + p], N - 1));
    double acc = ACCUM ? y[row] : 0.0;
    const int n = len[p];
#pragma unroll
    for (int s = 0; s < W; ++s)
        if (s < n) acc = __dadd_rn(acc, __dmul_rn(value[s * P + p], xv[s]));
    y[row] = acc;
}

// ---- the tiled product of the pattern form ---------------------------------------------------------------------------
// csr_pattern_kernel waits on three dependent round trips per row (dictionary, id, gathers) with one row per thread in
// flight.  When the patterns' deltas fall into a few narrow clusters (PatternWindows: lap2d {-n}, {-1..1}, {+n}), a CTA
// instead issues every load of kTileRows rows at once -- each cluster's window of x as 16-byte cp.async, the ids and the
// dictionary -- waits once, and computes the rows from shared memory (under ACCUM after a load of y).  The adds are
// csr_pattern_kernel's (same values, same x words, same order), so y keeps its bits.
struct alignas(16) PatternSlot {  // one slot of one pattern, read with one 16-byte shared-memory load
    double value;
    int offset;       // x[row + delta] is tile[offset + row - r0]
    int real;         // the slot lies below the pattern's length
};

__device__ __forceinline__ void cp_async16(double *dst, const double *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

// bytes 0 zero-fills the word without reading src
__device__ __forceinline__ void cp_async8(double *dst, const double *src, int bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src), "r"(bytes)
                 : "memory");
}

// Window c of the tile at r0 starts at x[r0 + lo[c] - a], a = 0 or 1 so that its address is 16-byte aligned whatever the
// alignment of x (a caller may pass x + 1); 64-bit, as r0 + lo reaches past 2^31 on lap3d 512^3.  Words outside [0, N)
// are zero-filled: only padding slots and rows past row_end could point there, and neither adds them.
__device__ __forceinline__ long long window_start(const double *x, long long r0, int lo) {
    const long long g = r0 + lo;
    return g - (long long)((((unsigned long long)x >> 3) + (unsigned long long)g) & 1);
}

template <int W, bool ACCUM>
__global__ void __launch_bounds__(kTileThreads, 8)
csr_pattern_tile_kernel(int row_begin, int row_end, const uint8_t *__restrict__ id, const int *__restrict__ dict, int P,
                        const PatternWindows win, const double *__restrict__ x, double *__restrict__ y, int N) {
    extern __shared__ __align__(16) double tile[];
    PatternSlot *slot = reinterpret_cast<PatternSlot *>(tile);  // [W][P], then the windows from win.base[0]
    __shared__ uint8_t ids[kTileRows];
    const int t = threadIdx.x;
    const long long r0 = row_begin + (long long)blockIdx.x * kTileRows;
#pragma unroll
    for (int c = 0; c < kMaxWindows; ++c) {
        if (c >= win.count) break;
        const long long start = window_start(x, r0, win.lo[c]);
        double *dst = tile + win.base[c];
        const int vecs = (win.base[c + 1] - win.base[c]) / 2;
        for (int v = t; v < vecs; v += kTileThreads) {
            const long long e = start + 2 * v;
            if (e >= 0 && e + 2 <= N) {
                cp_async16(dst + 2 * v, x + e);
            } else {
                const bool in0 = e >= 0 && e < N, in1 = e + 1 >= 0 && e + 1 < N;
                cp_async8(dst + 2 * v, in0 ? x + e : x, in0 ? 8 : 0);
                cp_async8(dst + 2 * v + 1, in1 ? x + e + 1 : x, in1 ? 8 : 0);
            }
        }
    }
    // the ids go through shared memory: held in registers, ptxas sank their loads below the barrier
#pragma unroll
    for (int k = 0; k < kTileRows / kTileThreads; ++k) {
        const long long row = r0 + t + k * kTileThreads;
        ids[t + k * kTileThreads] = (uint8_t)(row < row_end ? ldg_stream_u8(id + row) : 0);
    }
    const double *value = reinterpret_cast<const double *>(dict);
    const int *delta = dict + 2 * W * P, *len = delta + W * P;
    for (int i = t; i < W * P; i += kTileThreads) {
        const int s = i / P, d = __ldg(delta + i);
        int offset = win.base[0];  // a padding slot's delta 0 may lie in no window: any word of the tile will do
#pragma unroll
        for (int c = 0; c < kMaxWindows; ++c)
            if (c < win.count && d >= win.lo[c] && d <= win.hi[c])
                offset = win.base[c] + (int)(r0 + d - window_start(x, r0, win.lo[c]));
        slot[i] = PatternSlot{__ldg(value + i), offset, s < __ldg(len + (i - s * P))};
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kTileRows / kTileThreads; ++k) {
        const int i = t + k * kTileThreads;
        if (r0 + i >= row_end) break;
        double acc = ACCUM ? y[r0 + i] : 0.0;  // not held across the barrier: 4 rows of it spilled at 32 registers
        int4 sl[W];  // a PatternSlot as one LDS.128: value in x (low) and y (high), offset in z, real in w
        double xv[W];
#pragma unroll
        for (int s = 0; s < W; ++s) sl[s] = reinterpret_cast<const int4 *>(slot)[s * P + ids[i]];
#pragma unroll
        for (int s = 0; s < W; ++s) xv[s] = tile[sl[s].z + i];
#pragma unroll
        for (int s = 0; s < W; ++s)
            if (sl[s].w) acc = __dadd_rn(acc, __dmul_rn(__hiloint2double(sl[s].y, sl[s].x), xv[s]));
        y[r0 + i] = acc;
    }
}

// The windows of the tiled kernel, planned from the host copy of the dictionary: the distinct deltas of the real slots,
// sorted, clustered where neighbours lie less than kWindowGap apart.  count stays 0 (csr_pattern_kernel runs) unless there
// are at most min(W, kMaxWindows) clusters, none spans more than kWindowMaxSpan, and records and windows fit
// kWindowSmemMax.
static PatternWindows plan_windows(int W, int P, const int *delta, const int *len) {
    std::vector<int> d;
    for (int p = 0; p < P; ++p)
        for (int s = 0; s < len[p]; ++s) d.push_back(delta[s * P + p]);
    std::sort(d.begin(), d.end());
    d.erase(std::unique(d.begin(), d.end()), d.end());
    PatternWindows w;
    int n = 0;
    for (size_t k = 0; k < d.size(); ++k) {
        if (k > 0 && (long long)d[k] - d[k - 1] < kWindowGap) {
            w.hi[n - 1] = d[k];
            continue;
        }
        if (n == std::min(W, kMaxWindows)) return PatternWindows();
        w.lo[n] = w.hi[n] = d[k];
        ++n;
    }
    long long end = 2LL * W * P;  // the slot records: 16 bytes each
    for (int c = 0; c < n; ++c) {
        const long long span = (long long)w.hi[c] - w.lo[c];
        if (span > kWindowMaxSpan) return PatternWindows();
        w.base[c] = (int)end;
        end += (kTileRows + span + 3) & ~1LL;  // kTileRows + span + 1 words from a 16-byte boundary, whole vectors
    }
    if (n == 0 || 8 * end > kWindowSmemMax) return PatternWindows();
    w.base[n] = (int)end;
    w.count = n;
    return w;
}

static int launch_patterns(const CsrPatterns &P, int row_begin, int row_end, int N, const double *x, double *y, int accumulate,
                           cudaStream_t stream) {
    if (row_end <= row_begin) return SPMV_B200_OK;
    const PatternWindows &win = P.windows;
    SPMV_TRY_CUDA((with_batch<12, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11>(P.width, [&](auto W) {
        if (win.count > 0) {
            const unsigned int g = blocks_for(row_end - row_begin, kTileRows);
            const size_t smem = 8 * (size_t)win.base[win.count];
            if (accumulate)
                csr_pattern_tile_kernel<W, true><<<g, kTileThreads, smem, stream>>>(row_begin, row_end, P.id, P.dict, P.count, win, x, y, N);
            else
                csr_pattern_tile_kernel<W, false><<<g, kTileThreads, smem, stream>>>(row_begin, row_end, P.id, P.dict, P.count, win, x, y, N);
            return cudaGetLastError();
        }
        const unsigned int g = blocks_for(row_end - row_begin, 256);
        const size_t smem = (size_t)dict_bytes(P);
        if (accumulate) csr_pattern_kernel<W, true><<<g, 256, smem, stream>>>(row_begin, row_end, P.id, P.dict, P.count, x, y, N);
        else csr_pattern_kernel<W, false><<<g, 256, smem, stream>>>(row_begin, row_end, P.id, P.dict, P.count, x, y, N);
        return cudaGetLastError();
    })));
    return SPMV_B200_OK;
}

// ---- the distinct-key set ----------------------------------------------------------------------------------------------
// The distinct keys among n elements: the value patterns of the coded form, the row patterns of the pattern form.  A warp
// merges its lanes' equal keys (__match_any_sync), and one lane per key probes an open-addressing set of kSetSlots
// entries with a plain load: a key already in the set -- every one after the first few on a stencil -- costs no atomic.
// An entry, once written, never changes, so a stale load can only read kSetEmpty, and the compare-and-swap then tells the
// truth.  state[0] counts the entries and passes kMaxDistinct as soon as one more appears (or a probe walks past
// kMaxDistinct occupied entries, which only more keys can fill); every warp then stops.  An entry equal to kSetEmpty sets
// state[1] instead.  The caller sorts the entries on the host, so that ids do not depend on the order of the inserts.
// Keys supplies key(i), the 64-bit hash of element i that the warp merges and the probe starts from; entry(key, i), what
// the set stores; and same(cur, entry, i): whether the stored entry cur stands for element i.
constexpr int kSetSlots = 1024;
constexpr unsigned long long kSetEmpty = ~0ULL;

template <class Keys>
__global__ void distinct_kernel(long long n, const Keys K, unsigned long long *set, int *state) {
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    int step = 0;
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < n; base += stride, ++step) {
        if ((step & 63) == 0) {  // warp-uniform
            int stop = lane == 0 ? *(volatile int *)state : 0;
            if (__shfl_sync(0xffffffffu, stop, 0) > kMaxDistinct) return;
        }
        const long long i = min(base + lane, n - 1);
        const unsigned long long key = K.key(i);
        const unsigned int same = __match_any_sync(0xffffffffu, key);
        if (lane != __ffs(same) - 1) continue;
        const unsigned long long mine = K.entry(key, i);
        if (mine == kSetEmpty) {
            state[1] = 1;
            continue;
        }
        unsigned int slot = (unsigned int)key & (kSetSlots - 1);
        bool placed = false;
        for (int probe = 0; probe <= kMaxDistinct && !placed; ++probe) {
            unsigned long long cur = set[slot];
            if (cur == kSetEmpty) {
                cur = atomicCAS(set + slot, kSetEmpty, mine);
                if (cur == kSetEmpty) {
                    atomicAdd(state, 1);
                    placed = true;
                    break;
                }
            }
            placed = K.same(cur, mine, i);
            slot = (slot + 1) & (kSetSlots - 1);
        }
        if (!placed) atomicMax(state, kMaxDistinct + 1);
    }
}

// Runs distinct_kernel over n elements into a new set (*set, device: kSetSlots entries, then state[2]; the caller frees
// it) and copies the set and the state back
template <class Keys>
static int find_distinct(long long n, const Keys &K, cudaStream_t stream, unsigned long long **set,
                         std::vector<unsigned long long> &entries, int state[2]) {
    SPMV_TRY_CUDA(cudaMalloc(set, kSetSlots * sizeof(unsigned long long) + 2 * sizeof(int)));
    int *d_state = reinterpret_cast<int *>(*set + kSetSlots);
    SPMV_TRY_CUDA(cudaMemsetAsync(*set, 0xff, kSetSlots * sizeof(unsigned long long), stream));
    SPMV_TRY_CUDA(cudaMemsetAsync(d_state, 0, 2 * sizeof(int), stream));
    if (n > 0) {
        distinct_kernel<<<std::min(blocks_for(n, 256), 4096u), 256, 0, stream>>>(n, K, *set, d_state);
        SPMV_TRY_CUDA(cudaGetLastError());
    }
    entries.resize(kSetSlots);
    SPMV_TRY_CUDA(cudaMemcpyAsync(entries.data(), *set, kSetSlots * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
    SPMV_TRY_CUDA(cudaMemcpyAsync(state, d_state, 2 * sizeof(int), cudaMemcpyDeviceToHost, stream));
    SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
    return SPMV_B200_OK;
}

// the nonzeros' 64-bit value patterns: +0.0 and -0.0, and NaNs of different payloads, are different patterns; the pattern
// kSetEmpty itself sets state[1].  mix64 is a bijection, so equal hashes are equal patterns.
struct ValueKeys {
    const double *values;
    __device__ unsigned long long entry(unsigned long long, long long i) const { return __double_as_longlong(values[i]); }
    __device__ unsigned long long key(long long i) const { return mix64(entry(0, i)); }
    __device__ bool same(unsigned long long cur, unsigned long long mine, long long) const { return cur == mine; }
};

// the rows' patterns: a row is hashed, and an entry holds the top 33 bits of the hash and a representative row (bits 0-30;
// a row index never reaches 2^31 - 1, so no entry equals kSetEmpty).  A probe that meets its own tag compares the full
// rows, so two different rows of equal hash are two patterns; the warp merge trusts the hash alone, which is why
// pattern_fill_kernel compares every row with its representative and fails the build on a row it cannot place.
constexpr unsigned long long kRowBits = 0x7fffffffULL;

struct RowKeys {
    const int *row_ptr, *col_idx;
    const double *values;

    __device__ unsigned long long key(long long i) const {
        const int r = (int)i, lo = row_ptr[r], hi = row_ptr[r + 1];
        unsigned long long h = mix64(0x9E3779B97F4A7C15ULL + (unsigned long long)(hi - lo));
        for (int k = lo; k < hi; ++k) {
            h = mix64(h ^ (unsigned int)(col_idx[k] - r));
            h = mix64(h ^ (unsigned long long)__double_as_longlong(values[k]));
        }
        return h;
    }
    __device__ unsigned long long entry(unsigned long long h, long long r) const { return (h >> 31 << 31) | (unsigned long long)r; }
    __device__ bool same(unsigned long long cur, unsigned long long mine, long long i) const {
        if ((cur >> 31) != (mine >> 31)) return false;
        const int a = (int)i, b = (int)(cur & kRowBits);
        const int la = row_ptr[a], lb = row_ptr[b], n = row_ptr[a + 1] - la;
        if (row_ptr[b + 1] - lb != n) return false;
        for (int k = 0; k < n; ++k)
            if (col_idx[la + k] - a != col_idx[lb + k] - b ||
                __double_as_longlong(values[la + k]) != __double_as_longlong(values[lb + k]))
                return false;
        return true;
    }
};

// ---- the build of the pattern form -------------------------------------------------------------------------------------
// the representatives' rows, for the host's sort: out[p] = {len, delta[0..W), value bits[0..W)} (zero past len)
__global__ void pattern_rows_kernel(int P, int W, const int *__restrict__ reps, RowKeys A, unsigned long long *out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const int r = reps[p], lo = A.row_ptr[r], n = A.row_ptr[r + 1] - lo;
    unsigned long long *o = out + (size_t)p * (1 + 2 * W);
    o[0] = (unsigned long long)n;
    for (int s = 0; s < W; ++s) {
        o[1 + s] = s < n ? (unsigned long long)(unsigned int)(A.col_idx[lo + s] - r) : 0;
        o[1 + W + s] = s < n ? (unsigned long long)__double_as_longlong(A.values[lo + s]) : 0;
    }
}

// id[r]: the pattern of row r, found by its hash and a full compare with the representative (*missing = 1 when none)
__global__ void pattern_fill_kernel(int M, RowKeys A, const unsigned long long *__restrict__ keys,
                                    const uint8_t *__restrict__ slot_id, uint8_t *__restrict__ id, int *missing) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= M) return;
    const unsigned long long h = A.key(r), mine = A.entry(h, r);
    unsigned int slot = (unsigned int)h & (kSetSlots - 1);
    for (int probe = 0; probe < kSetSlots; ++probe) {
        const unsigned long long cur = keys[slot];
        if (cur == kSetEmpty) break;
        if (A.same(cur, mine, r)) {
            id[r] = slot_id[slot];
            return;
        }
        slot = (slot + 1) & (kSetSlots - 1);
    }
    *missing = 1;
}

static void free_patterns(CsrPatterns &P) {
    cudaFree(P.id);
    cudaFree(P.dict);
    P = CsrPatterns();
}

// The pattern form of A (owned arrays and no long rows assumed by the caller).  SPMV_B200_ERR_INVALID, without a message
// (the plan tries every eligible matrix), when A does not qualify: no row or one above kRowKernelMaxLen, more than
// kMaxDistinct patterns, or a dictionary above kPatternDictMaxBytes.  P is left empty on failure.
static int build_patterns(const spmv_b200_csr *A, cudaStream_t stream, CsrPatterns &P) {
    const int M = A->M, W = A->max_row;
    if (M <= 0 || W < 1 || W > kRowKernelMaxLen) return SPMV_B200_ERR_INVALID;
    P.width = W;
    const RowKeys rows{A->row_ptr, A->col_idx, A->values};
    unsigned long long *keys = nullptr, *contents = nullptr;  // keys[kSetSlots], then state[2] (count, missing)
    int *reps_d = nullptr;
    uint8_t *slot_id_d = nullptr;
    auto body = [&]() -> int {
        std::vector<unsigned long long> slots;
        int count[2] = {0, 0};
        SPMV_TRY(find_distinct(M, rows, stream, &keys, slots, count));
        int *state = reinterpret_cast<int *>(keys + kSetSlots);
        if (count[0] > kMaxDistinct) return SPMV_B200_ERR_INVALID;
        std::vector<int> where, reps;  // occupied entries and their representative rows
        for (int s = 0; s < kSetSlots; ++s)
            if (slots[s] != kSetEmpty) {
                where.push_back(s);
                reps.push_back((int)(slots[s] & kRowBits));
            }
        const int n = P.count = (int)reps.size();
        if (dict_bytes(P) - 4LL * n > kPatternDictMaxBytes) return SPMV_B200_ERR_INVALID;
        // ids in the order of the patterns' contents, so that they do not depend on the order of the inserts
        const int rec = 1 + 2 * W;
        std::vector<unsigned long long> content((size_t)n * rec);
        SPMV_TRY_CUDA(cudaMalloc(&reps_d, (size_t)n * sizeof(int)));
        SPMV_TRY_CUDA(cudaMalloc(&contents, content.size() * sizeof(unsigned long long)));
        SPMV_TRY_CUDA(cudaMemcpyAsync(reps_d, reps.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, stream));
        pattern_rows_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(n, W, reps_d, rows, contents);
        SPMV_TRY_CUDA(cudaGetLastError());
        SPMV_TRY_CUDA(cudaMemcpyAsync(content.data(), contents, content.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
        std::vector<int> order((size_t)n);
        std::iota(order.begin(), order.end(), 0);
        std::sort(order.begin(), order.end(), [&](int a, int b) {
            return std::lexicographical_compare(content.begin() + (size_t)a * rec, content.begin() + (size_t)(a + 1) * rec,
                                                content.begin() + (size_t)b * rec, content.begin() + (size_t)(b + 1) * rec);
        });
        std::vector<uint8_t> slot_id(kSetSlots, 0);
        const size_t bytes = (size_t)dict_bytes(P);
        std::vector<int> dict(bytes / sizeof(int), 0);
        double *value = reinterpret_cast<double *>(dict.data());
        int *delta = dict.data() + 2 * W * n, *len = delta + W * n;
        for (int p = 0; p < n; ++p) {
            const unsigned long long *c = content.data() + (size_t)order[p] * rec;
            slot_id[where[order[p]]] = (uint8_t)p;
            len[p] = (int)c[0];
            for (int s = 0; s < W; ++s) {
                delta[s * n + p] = (int)(unsigned int)c[1 + s];
                std::memcpy(value + s * n + p, c + 1 + W + s, sizeof(double));
            }
        }
        P.windows = plan_windows(W, n, delta, len);
        SPMV_TRY_CUDA(cudaMalloc(&P.dict, bytes));
        SPMV_TRY_CUDA(cudaMalloc(&P.id, (size_t)M));
        SPMV_TRY_CUDA(cudaMalloc(&slot_id_d, kSetSlots));
        SPMV_TRY_CUDA(cudaMemcpyAsync(P.dict, dict.data(), bytes, cudaMemcpyHostToDevice, stream));
        SPMV_TRY_CUDA(cudaMemcpyAsync(slot_id_d, slot_id.data(), kSetSlots, cudaMemcpyHostToDevice, stream));
        pattern_fill_kernel<<<blocks_for(M, 256), 256, 0, stream>>>(M, rows, keys, slot_id_d, P.id, state + 1);
        SPMV_TRY_CUDA(cudaGetLastError());
        SPMV_TRY_CUDA(cudaMemcpyAsync(count, state, sizeof count, cudaMemcpyDeviceToHost, stream));
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));  // also keeps the host vectors alive until the copies are done
        if (count[1]) return SPMV_B200_ERR_INVALID;  // two different rows of one warp with equal 64-bit hashes
        return SPMV_B200_OK;
    };
    const int rc = body();
    cudaFree(keys);
    cudaFree(contents);
    cudaFree(reps_d);
    cudaFree(slot_id_d);
    if (rc != SPMV_B200_OK) free_patterns(P);
    return rc;
}

// ---- the build of the column-major form ------------------------------------------------------------------------------
enum ImageValues { kImageF64 = 1, kImageCodes = 2, kImageBoth = 3 };

static void free_columns(ColumnImage &C) {
    cudaFree(C.hack_off);
    cudaFree(C.JA);
    cudaFree(C.JA16);
    cudaFree(C.AS);
    cudaFree(C.AC);
    cudaFree(C.table);
    C = ColumnImage();
}

// The value table of the coded form: the distinct 64-bit value patterns ascending as uint64, so that the image does not
// depend on the order of the inserts; *ok = false when there are more than kMaxDistinct
static int value_table(const spmv_b200_csr *A, cudaStream_t stream, std::vector<unsigned long long> &table, bool *ok) {
    unsigned long long *set = nullptr;
    int state[2] = {0, 0};
    const int rc = find_distinct(A->nnz, ValueKeys{A->values}, stream, &set, table, state);
    cudaFree(set);
    SPMV_TRY(rc);
    *ok = state[0] <= kMaxDistinct;
    if (*ok) {
        table.erase(std::remove(table.begin(), table.end(), kSetEmpty), table.end());
        if (state[1]) table.push_back(kSetEmpty);
        std::sort(table.begin(), table.end());
        *ok = (int)table.size() <= kMaxDistinct;
    }
    return SPMV_B200_OK;
}

// The column-major form of A into C.  values: the value streams to fill -- fp64, the codes (SPMV_B200_ERR_INVALID on a
// matrix of more than kMaxDistinct value patterns), or both where they fit (plan time: both when they fit, else the codes
// alone, else fp64 alone).  max_slots / max_bytes >= 0: a form of more slots, or of more bytes of columns, values and
// table, is not built.  C is left empty unless the form is built.
static int build_columns(const spmv_b200_csr *A, long long max_slots, long long max_bytes, ImageValues values,
                         cudaStream_t stream, ColumnImage &C) {
    const int M = A->M, N = A->N;
    auto body = [&]() -> int {
        std::vector<long long> host_off;
        bool narrow = false, codes = false;
        SPMV_TRY(hll_layout(M, N, A->row_ptr, A->col_idx, stream, &C.hack_off, host_off, &C.max_width, &narrow));
        C.num_hacks = (int)host_off.size() - 1;
        C.slots = host_off[C.num_hacks];
        std::vector<unsigned long long> table;
        if (values & kImageCodes) SPMV_TRY(value_table(A, stream, table, &codes));
        if (values == kImageCodes && !codes)
            return fail(SPMV_B200_ERR_INVALID, "csr image: the values hold more than %d distinct 64-bit patterns", kMaxDistinct);
        if (max_slots >= 0 && C.slots > max_slots) return SPMV_B200_OK;
        // bytes per slot of each choice, largest first: both value streams (plan time), the codes alone, fp64 alone
        const long long index = narrow ? 2 : 4, table_bytes = codes ? 8LL * (long long)table.size() : 0;
        auto fit = [&](long long per_slot, long long extra) { return max_bytes < 0 || C.slots * per_slot + extra <= max_bytes; };
        bool f64 = values != kImageCodes;
        if (f64 && codes && !fit(index + 9, table_bytes)) f64 = false;  // plan time: the codes alone where both do not fit
        if (!codes && !fit(index + 8, 0)) return SPMV_B200_OK;
        if (codes && !fit(index + (f64 ? 9 : 1), table_bytes)) return SPMV_B200_OK;
        const size_t n = (size_t)std::max<long long>(C.slots, 32);
        if (narrow) SPMV_TRY_CUDA(cudaMalloc(&C.JA16, n * sizeof(uint16_t)));
        else SPMV_TRY_CUDA(cudaMalloc(&C.JA, n * sizeof(int)));
        if (f64) SPMV_TRY_CUDA(cudaMalloc(&C.AS, n * sizeof(double)));
        if (codes) {
            SPMV_TRY_CUDA(cudaMalloc(&C.AC, n * sizeof(uint8_t)));
            std::vector<double> tab(std::max<size_t>(table.size(), 1), 0.0);  // at least one entry: padding reads code 0
            std::memcpy(tab.data(), table.data(), table.size() * sizeof(double));
            C.num_values = (int)table.size();
            SPMV_TRY_CUDA(cudaMalloc(&C.table, tab.size() * sizeof(double)));
            SPMV_TRY_CUDA(cudaMemcpyAsync(C.table, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, stream));
            SPMV_TRY_CUDA(cudaStreamSynchronize(stream));  // tab is a local
        }
        SPMV_TRY(hll_fill(M, N, A->row_ptr, A->col_idx, A->values, C.num_hacks, C.hack_off, C.JA, C.JA16, C.AS, C.AC, C.table,
                          C.num_values, true, stream));
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
        C.segments = hll_find_segments(host_off, C.num_hacks);
        return SPMV_B200_OK;
    };
    const int rc = body();
    if (rc != SPMV_B200_OK || (!C.JA && !C.JA16)) free_columns(C);
    return rc;
}

// ---- the interface (handles.cuh) -----------------------------------------------------------------------------------------
void image_free(CsrImage *&img) {
    if (!img) return;
    free_columns(img->cols);
    free_patterns(img->patterns);
    delete img;
    img = nullptr;
}

static int launch_form(const CsrImage *img, const ImageForm &f, int row_begin, int row_end, const double *x, double *y,
                       int accumulate, cudaStream_t stream) {
    if (f.patterns) return launch_patterns(img->patterns, row_begin, row_end, img->N, x, y, accumulate, stream);
    const ColumnImage &C = img->cols;
    return hll_masked_launch(row_begin / 32, (row_end + 31) / 32, img->M, C.hack_off, C.segments, C.JA, C.JA16, C.slots,
                             f.coded ? nullptr : C.AS, f.coded ? C.AC : nullptr, C.table, std::max(C.num_values, 1), f.batch,
                             f.offset_free, accumulate, x, y, stream);
}

int image_launch(const CsrImage *img, int row_begin, int row_end, const double *x, double *y, int accumulate,
                 cudaStream_t stream) {
    return launch_form(img, img->form, row_begin, row_end, x, y, accumulate, stream);
}

bool image_any_rows(const CsrImage *img) { return img->form.patterns; }

int image_candidates(const spmv_b200_csr *A, cudaStream_t stream, CsrImage **out) {
    CsrImage *img = *out = new (std::nothrow) CsrImage(A);
    if (!img) return 0;
    size_t free_bytes = 0, total_bytes = 0;
    if (cudaMemGetInfo(&free_bytes, &total_bytes) == cudaSuccess) {
        const long long fit_bytes = (long long)(free_bytes / 4) - 8LL * ((long long)A->M / 32 + 2);
        if (fit_bytes >= 0) build_columns(A, A->nnz + A->nnz / 4, fit_bytes, kImageBoth, stream, img->cols);
        if ((long long)A->M * A->max_row <= A->nnz + A->nnz / 4 && (long long)A->M <= fit_bytes)
            build_patterns(A, stream, img->patterns);
    }
    cudaGetLastError();
    const ColumnImage &C = img->cols;
    for (int coded = 0; coded <= 1; ++coded) {
        if (coded ? !C.AC : !C.AS) continue;
        for (int batch = 2; batch <= 7; ++batch)
            if (C.segments.count == 0) img->candidates.push_back({false, false, batch, coded != 0});
            else if (batch >= 4) img->candidates.push_back({false, true, batch, coded != 0});
    }
    if (img->patterns.id) img->candidates.push_back({true, false, 0, false});
    if (img->candidates.empty()) image_free(*out);
    return *out ? (int)img->candidates.size() : 0;
}

int image_launch_candidate(const CsrImage *img, int i, const double *x, double *y, cudaStream_t stream) {
    return launch_form(img, img->candidates[i], 0, img->M, x, y, 0, stream);
}

void image_keep(CsrImage *img, int i) {
    img->form = img->candidates[i];
    ColumnImage &C = img->cols;
    if (img->form.patterns) return free_columns(C);
    free_patterns(img->patterns);
    if (img->form.coded) {
        cudaFree(C.AS);
        C.AS = nullptr;
        return;
    }
    cudaFree(C.AC);
    cudaFree(C.table);
    C.AC = nullptr;
    C.table = nullptr;
    C.num_values = 0;
}

int image_build(spmv_b200_csr *A, int mode, cudaStream_t stream) {
    if (!A->owns) return fail(SPMV_B200_ERR_INVALID, "csr_set_image: the matrix wraps arrays it does not own");
    if (A->max_row > kRowKernelMaxLen || A->num_long > 0)
        return fail(SPMV_B200_ERR_INVALID, "csr_set_image: rows of up to %d nonzeros and no long rows only (longest row: %d)",
                    kRowKernelMaxLen, A->max_row);
    const CsrImage *held = A->image;  // already the form asked for: a column-major image holds only the value stream it runs
    if (held && (mode == 3 ? held->form.patterns : mode == 2 ? held->cols.AC != nullptr : held->cols.AS != nullptr))
        return SPMV_B200_OK;
    CsrImage *img = new (std::nothrow) CsrImage(A);  // the held image stays until the new one is built
    if (!img) return fail(SPMV_B200_ERR_NOMEM, "csr image: out of host memory");
    int rc;
    if (mode == 3) {
        rc = build_patterns(A, stream, img->patterns);
        if (rc != SPMV_B200_OK)
            rc = fail(SPMV_B200_ERR_INVALID, "csr_set_image: the pattern form needs 1 to %d nonzeros per row, at most %d distinct "
                      "rows and a dictionary of at most %d bytes", kRowKernelMaxLen, kMaxDistinct, kPatternDictMaxBytes);
        img->form.patterns = true;
    } else {
        rc = build_columns(A, -1, -1, mode == 2 ? kImageCodes : kImageF64, stream, img->cols);
        // hll_rowu_kernel<clamp(max_width, 3, 7)> on a regular layout, else hll_row_kernel<clamp(mean width, 2, 7)>
        const ColumnImage &C = img->cols;
        const long long mean = C.num_hacks > 0 ? (C.slots / 32 + C.num_hacks - 1) / C.num_hacks : 4;
        img->form.offset_free = C.segments.count > 0;
        img->form.batch = img->form.offset_free ? std::max(3, std::min(7, C.max_width)) : (int)std::max(2LL, std::min(7LL, mean));
        img->form.coded = mode == 2;
    }
    if (rc != SPMV_B200_OK) {
        image_free(img);
        return rc;
    }
    image_free(A->image);
    A->image = img;
    return SPMV_B200_OK;
}

void image_info(const CsrImage *img, spmv_b200_csr_info_t *info) {
    info->image_bytes = info->image_device_bytes = 0;
    info->image_form = info->image_index_bytes = info->image_value_bytes = info->image_patterns = info->image_windows = 0;
    if (!img) return;
    if (img->form.patterns) {  // one byte per row plus the dictionary
        info->image_form = 256 + img->patterns.width;  // csr_pattern_kernel<W> or csr_pattern_tile_kernel<W>
        info->image_bytes = info->image_device_bytes = img->M + dict_bytes(img->patterns);
        info->image_patterns = img->patterns.count;
        info->image_windows = img->patterns.windows.count;
        return;
    }
    const ColumnImage &C = img->cols;
    info->image_bytes = 12 * C.slots;
    info->image_form = (img->form.offset_free ? 64 : 0) + img->form.batch;
    info->image_index_bytes = C.JA16 ? 2 : 4;
    info->image_value_bytes = (C.AS ? 8 : 0) + (C.AC ? 1 : 0);
    info->image_device_bytes = C.slots * (info->image_index_bytes + info->image_value_bytes) + (C.AC ? 8LL * C.num_values : 0);
}

}  // namespace spmv
