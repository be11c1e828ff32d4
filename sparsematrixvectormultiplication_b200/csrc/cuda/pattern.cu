// pattern.cu -- the pattern form of a CSR handle's private image: one byte per row naming the row's pattern.
//
// On stencils, structured-grid FEM and unit-weight banded matrices whole rows repeat: a row's pattern -- its length, the
// col - row of each slot and the 64-bit pattern of each value -- takes 9 distinct forms on lap2d (interior, 4 edges, 4
// corners) and 27 on lap3d.  When the matrix holds at most kMaxPatterns of them, the product streams one byte per row
// (the pattern id) instead of a column field and a value field per slot: CSR-VI (Kourtis et al.) applied to whole rows.
// The dictionary (value[W][P], delta[W][P], len[P]; slot-major, so lanes of different patterns read different banks)
// is staged in shared memory.  lap2d 4096^2: 16.8 MB of ids and 540 B of dictionary, against 252 MB for the coded image.
#include <algorithm>
#include <cstring>
#include <new>
#include <numeric>
#include <vector>

#include "common.cuh"
#include "handles.cuh"

namespace spmv {

// ---- the product -----------------------------------------------------------------------------------------------------
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

int csr_patterns_launch(const CsrPatterns *P, int row_begin, int row_end, int N, const double *x, double *y, int accumulate,
                        cudaStream_t stream) {
    if (row_end <= row_begin) return SPMV_B200_OK;
    const unsigned int g = blocks_for(row_end - row_begin, 256);
    const size_t smem = (size_t)csr_patterns_dict_bytes(P);
    SPMV_TRY_CUDA((with_batch<12, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11>(P->width, [&](auto W) {
        if (accumulate) csr_pattern_kernel<W, true><<<g, 256, smem, stream>>>(row_begin, row_end, P->id, P->dict, P->count, x, y, N);
        else csr_pattern_kernel<W, false><<<g, 256, smem, stream>>>(row_begin, row_end, P->id, P->dict, P->count, x, y, N);
        return cudaGetLastError();
    })));
    return SPMV_B200_OK;
}

// ---- the build -------------------------------------------------------------------------------------------------------
// The distinct row patterns, in the style of hll_value_dict_kernel: each row is hashed, a warp merges its lanes' equal
// hashes (__match_any_sync) and one lane per hash probes an open-addressing set of kPatternSlots entries.  An entry holds
// the top 33 bits of the hash and a representative row (bits 0-30; a row index never reaches 2^31 - 1, so no entry
// equals kPatternEmpty).  A probe that meets its own tag compares the full rows, so two different rows of equal hash are
// two patterns; the warp merge trusts the hash alone, which is why the fill pass compares every row with its
// representative and fails the build on a row it cannot place.  state[0] counts the patterns and passes kMaxPatterns as
// soon as a 257th appears (or a probe walks past kMaxPatterns occupied entries, which only more patterns can fill);
// every warp then stops.  An entry, once written, never changes, so a stale load can only read kPatternEmpty, and the
// compare-and-swap then tells the truth.
constexpr int kPatternSlots = 1024;
constexpr unsigned long long kPatternEmpty = ~0ULL;
constexpr unsigned long long kRowBits = 0x7fffffffULL;

struct RowsRef {
    const int *row_ptr, *col_idx;
    const double *values;
};

__device__ unsigned long long row_hash(const RowsRef &A, int r) {
    const int lo = A.row_ptr[r], hi = A.row_ptr[r + 1];
    unsigned long long h = mix64(0x9E3779B97F4A7C15ULL + (unsigned long long)(hi - lo));
    for (int k = lo; k < hi; ++k) {
        h = mix64(h ^ (unsigned int)(A.col_idx[k] - r));
        h = mix64(h ^ (unsigned long long)__double_as_longlong(A.values[k]));
    }
    return h;
}

__device__ bool rows_equal(const RowsRef &A, int a, int b) {
    const int la = A.row_ptr[a], lb = A.row_ptr[b], n = A.row_ptr[a + 1] - la;
    if (A.row_ptr[b + 1] - lb != n) return false;
    for (int k = 0; k < n; ++k)
        if (A.col_idx[la + k] - a != A.col_idx[lb + k] - b ||
            __double_as_longlong(A.values[la + k]) != __double_as_longlong(A.values[lb + k]))
            return false;
    return true;
}

__device__ __forceinline__ unsigned long long pattern_entry(unsigned long long h, int r) {
    return (h >> 31 << 31) | (unsigned long long)r;
}

__device__ __forceinline__ bool entry_matches(const RowsRef &A, unsigned long long cur, unsigned long long mine, int r) {
    return (cur >> 31) == (mine >> 31) && rows_equal(A, r, (int)(cur & kRowBits));
}

__global__ void pattern_dict_kernel(int M, RowsRef A, unsigned long long *keys, int *state) {
    const int lane = threadIdx.x & 31;
    const long long stride = (long long)gridDim.x * blockDim.x;
    int step = 0;
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < M; base += stride, ++step) {
        if ((step & 63) == 0) {  // warp-uniform
            int stop = lane == 0 ? *(volatile int *)state : 0;
            if (__shfl_sync(0xffffffffu, stop, 0) > kMaxPatterns) return;
        }
        const int r = (int)min(base + lane, (long long)M - 1);
        const unsigned long long h = row_hash(A, r);
        const unsigned int same = __match_any_sync(0xffffffffu, h);
        if (lane != __ffs(same) - 1) continue;
        const unsigned long long mine = pattern_entry(h, r);
        unsigned int slot = (unsigned int)h & (kPatternSlots - 1);
        bool placed = false;
        for (int probe = 0; probe <= kMaxPatterns && !placed; ++probe) {
            unsigned long long cur = keys[slot];
            if (cur == kPatternEmpty) {
                cur = atomicCAS(keys + slot, kPatternEmpty, mine);
                if (cur == kPatternEmpty) {
                    atomicAdd(state, 1);
                    placed = true;
                    break;
                }
            }
            placed = entry_matches(A, cur, mine, r);
            slot = (slot + 1) & (kPatternSlots - 1);
        }
        if (!placed) atomicMax(state, kMaxPatterns + 1);
    }
}

// the representatives' rows, for the host's sort: out[p] = {len, delta[0..W), value bits[0..W)} (zero past len)
__global__ void pattern_rows_kernel(int P, int W, const int *__restrict__ reps, RowsRef A, unsigned long long *out) {
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
__global__ void pattern_fill_kernel(int M, RowsRef A, const unsigned long long *__restrict__ keys,
                                    const uint8_t *__restrict__ slot_id, uint8_t *__restrict__ id, int *missing) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= M) return;
    const unsigned long long h = row_hash(A, (int)r), mine = pattern_entry(h, (int)r);
    unsigned int slot = (unsigned int)h & (kPatternSlots - 1);
    for (int probe = 0; probe < kPatternSlots; ++probe) {
        const unsigned long long cur = keys[slot];
        if (cur == kPatternEmpty) break;
        if (entry_matches(A, cur, mine, (int)r)) {
            id[r] = slot_id[slot];
            return;
        }
        slot = (slot + 1) & (kPatternSlots - 1);
    }
    *missing = 1;
}

void csr_patterns_free(CsrPatterns *P) {
    if (!P) return;
    cudaFree(P->id);
    cudaFree(P->dict);
    delete P;
}

int csr_patterns_build(const spmv_b200_csr *A, cudaStream_t stream, CsrPatterns **out) {
    *out = nullptr;
    const int M = A->M, W = A->max_row;
    if (M <= 0 || W < 1 || W > kRowKernelMaxLen) return SPMV_B200_ERR_INVALID;
    CsrPatterns *P = new (std::nothrow) CsrPatterns();
    if (!P) return fail(SPMV_B200_ERR_NOMEM, "csr patterns: out of host memory");
    P->width = W;
    const RowsRef rows{A->row_ptr, A->col_idx, A->values};
    unsigned long long *keys = nullptr, *contents = nullptr;  // keys[kPatternSlots], then state[2] (count, missing)
    int *reps_d = nullptr;
    uint8_t *slot_id_d = nullptr;
    auto body = [&]() -> int {
        SPMV_TRY_CUDA(cudaMalloc(&keys, kPatternSlots * sizeof(unsigned long long) + 2 * sizeof(int)));
        int *state = reinterpret_cast<int *>(keys + kPatternSlots);
        SPMV_TRY_CUDA(cudaMemsetAsync(keys, 0xff, kPatternSlots * sizeof(unsigned long long), stream));
        SPMV_TRY_CUDA(cudaMemsetAsync(state, 0, 2 * sizeof(int), stream));
        pattern_dict_kernel<<<std::min(blocks_for(M, 256), 4096u), 256, 0, stream>>>(M, rows, keys, state);
        SPMV_TRY_CUDA(cudaGetLastError());
        std::vector<unsigned long long> slots(kPatternSlots);
        int count[2] = {0, 0};
        SPMV_TRY_CUDA(cudaMemcpyAsync(slots.data(), keys, kPatternSlots * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
        SPMV_TRY_CUDA(cudaMemcpyAsync(count, state, sizeof count, cudaMemcpyDeviceToHost, stream));
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
        if (count[0] > kMaxPatterns) return SPMV_B200_ERR_INVALID;
        std::vector<int> where, reps;  // occupied entries and their representative rows
        for (int s = 0; s < kPatternSlots; ++s)
            if (slots[s] != kPatternEmpty) {
                where.push_back(s);
                reps.push_back((int)(slots[s] & kRowBits));
            }
        const int n = P->count = (int)reps.size();
        if (csr_patterns_dict_bytes(P) - 4LL * n > kPatternDictMaxBytes) return SPMV_B200_ERR_INVALID;
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
        std::vector<uint8_t> slot_id(kPatternSlots, 0);
        const size_t dict_bytes = (size_t)csr_patterns_dict_bytes(P);
        std::vector<int> dict(dict_bytes / sizeof(int), 0);
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
        SPMV_TRY_CUDA(cudaMalloc(&P->dict, dict_bytes));
        SPMV_TRY_CUDA(cudaMalloc(&P->id, (size_t)M));
        SPMV_TRY_CUDA(cudaMalloc(&slot_id_d, kPatternSlots));
        SPMV_TRY_CUDA(cudaMemcpyAsync(P->dict, dict.data(), dict_bytes, cudaMemcpyHostToDevice, stream));
        SPMV_TRY_CUDA(cudaMemcpyAsync(slot_id_d, slot_id.data(), kPatternSlots, cudaMemcpyHostToDevice, stream));
        pattern_fill_kernel<<<blocks_for(M, 256), 256, 0, stream>>>(M, rows, keys, slot_id_d, P->id, state + 1);
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
    if (rc != SPMV_B200_OK) {
        csr_patterns_free(P);
        return rc;
    }
    *out = P;
    return SPMV_B200_OK;
}

}  // namespace spmv
