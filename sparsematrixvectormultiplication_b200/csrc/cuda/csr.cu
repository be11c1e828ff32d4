// csr.cu -- CSR y = A*x for sm_100a (B200): kernels, plans and the C-ABI entry points.
//
// Replaces the reference's spmv_csr_{naive,warp,warp_shared_memory}_kernel
// (reference cuda_src/csr_matrix_cuda.cu:122-241, launched from main_cuda.cu:166,238,317).
//
// SpMV is an HBM-bound gather (0.15 flop/B): no tensor cores.  Kernels in this file (DESIGN.md section 3):
//   * csr_row_kernel<BATCH,V>     -- one THREAD per row, L1-resident stream, serial order (bit-identical to the reference's
//       loop).  The automatic choice when no row exceeds 12 nonzeros (stencils); BATCH is timed at plan time.
//   * csr_row_fused_kernel / csr_row_async_kernel -- the same with the fused tail of the iterated product (scale,
//       |w|^2 partials, NVLink peer stores, mailbox / asynchronous exchange).
//   * csr_vector_kernel<VEC,V>    -- VEC lanes per row, batched gathers, shuffle reduction; needs no plan, works on raw
//       device arrays (drop-in for the reference's warp kernel launch).  Automatic choice for longer, even rows.
//   * csr_binned_kernel<V> + csr_long_fragment_kernel + csr_long_combine_kernel -- rows sorted by length class, 1..32
//       lanes per row in one launch; rows above 2048 nonzeros split into 8192-nonzero fragments combined in a fixed
//       order (deterministic, no atomics).  Automatic choice for skewed rows.
// V = storage type (double, or float with double arithmetic).  The TMA-pipelined stream kernels live in stream.cu.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include <utility>
#include <vector>

#include "common.cuh"
#include "handles.cuh"

namespace spmv {

constexpr int kAutoStreamMaxAvg = 12;  // ALGO_AUTO: stream kernel up to this many nonzeros per row on average
constexpr int kFragNnz = 8192;              // nonzeros per long-row fragment (one CTA)
constexpr int kFragThreads = 256;
constexpr int kVecBatch = 4;                // independent column -> gather chains per lane of the vector kernel
constexpr long long kAutotuneMinNnz = 1 << 22;  // plan-time timing of the row-kernel batch only pays on large matrices
constexpr int kRowBatch = 4;                // the same with ONE lane per row (bin 0 of the binned kernel)
constexpr int kVec4Default = 1;              // vector / binned kernels: aligned groups of four nonzeros per lane (SPMV_B200_VEC4)
constexpr int kFusedCtasPerSm = 8;          // grid of the fused row kernels per SM (SPMV_B200_FUSED_CTAS_PER_SM)
constexpr int kMatrixPersistDefault = 0;    // head of row_ptr / JA held in the persisting carve-out across products (SPMV_B200_MATRIX_PERSIST)
constexpr int kL2PersistDefault = 0;        // persisting-L2 window on x for the gather-bound kernels (SPMV_B200_L2_PERSIST)

__device__ __forceinline__ void ldg_stream_f64x4(const float *p, double (&v)[4]) {  // fp32 storage: one 128-bit load
    float4 f;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(f.x), "=f"(f.y), "=f"(f.z), "=f"(f.w) : "l"(p));
    v[0] = f.x;
    v[1] = f.y;
    v[2] = f.z;
    v[3] = f.w;
}

// Matrix stream loads of the vector kernels.  Several lanes per row: consecutive lanes read consecutive elements, every
// sector is consumed by one instruction -> no L1 allocation.  ONE lane per row: lane i walks its own row, a warp's
// loads are strided by the row length and a sector is consumed over several iterations -> it must live in L1 in
// between (plain read-only loads; measured on lap2d 4096^2: 5.1 TB/s without allocation, 6.0 TB/s with).
template <int VEC>
__device__ __forceinline__ int load_col(const int *p) {
    if constexpr (VEC == 1) return __ldg(p);
    else return ldg_stream_s32(p);
}
template <int VEC, typename V>
__device__ __forceinline__ double load_val(const V *p) {
    if constexpr (VEC == 1) return (double)__ldg(p);
    else return ldg_stream_f64(p);
}

// ================================================================================================
// kernels
// ================================================================================================

// One CTA per fragment of a long row; partial[f] = sum over the fragment (fixed tree).  Every thread of the CTA calls it.
template <typename V>
__device__ __forceinline__ void long_fragment(int f, const int *__restrict__ long_rows, const int *__restrict__ frag_first,
                                              int num_long, const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                                              const V *__restrict__ values, const V *__restrict__ x,
                                              double *__restrict__ partial) {
    __shared__ double warp_sum[kFragThreads / 32];
    int lo = 0, hi = num_long;  // last long row whose first fragment is <= f
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(frag_first + mid) <= f) lo = mid; else hi = mid;
    }
    const int row = __ldg(long_rows + lo);
    const long long begin = (long long)__ldg(row_ptr + row) + (long long)(f - __ldg(frag_first + lo)) * kFragNnz;
    const long long row_end = __ldg(row_ptr + row + 1);
    const long long end = begin + kFragNnz < row_end ? begin + kFragNnz : row_end;
    // batches of kVecBatch: all column / value loads, then all gathers, then the fmas (one round trip per batch)
    double acc = 0.0;
    for (long long k = begin + threadIdx.x; k < end; k += (long long)kVecBatch * kFragThreads) {
        int c[kVecBatch];
        double v[kVecBatch], xv[kVecBatch];
#pragma unroll
        for (int u = 0; u < kVecBatch; ++u) c[u] = k + u * kFragThreads < end ? ldg_stream_s32(col_idx + k + u * kFragThreads) : -1;
#pragma unroll
        for (int u = 0; u < kVecBatch; ++u) v[u] = k + u * kFragThreads < end ? ldg_stream_f64(values + k + u * kFragThreads) : 0.0;
#pragma unroll
        for (int u = 0; u < kVecBatch; ++u) xv[u] = c[u] >= 0 ? ldg_x(x, c[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < kVecBatch; ++u)
            if (c[u] >= 0) acc = fma(v[u], xv[u], acc);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double total = 0.0;
#pragma unroll
        for (int w = 0; w < kFragThreads / 32; ++w) total += warp_sum[w];
        partial[f] = total;
    }
}

template <typename V>
__global__ void __launch_bounds__(kFragThreads)
csr_long_fragment_kernel(const int *__restrict__ long_rows, const int *__restrict__ frag_first, int num_long,
                         const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                         const V *__restrict__ values, const V *__restrict__ x,
                         double *__restrict__ partial) {
    long_fragment<V>((int)blockIdx.x, long_rows, frag_first, num_long, row_ptr, col_idx, values, x, partial);
}

template <typename V>
__global__ void csr_long_combine_kernel(const int *__restrict__ long_rows, const int *__restrict__ frag_first,
                                        int num_long, const double *__restrict__ partial, V *__restrict__ y,
                                        int accumulate) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num_long) return;
    const int row = long_rows[i];
    double acc = accumulate ? (double)y[row] : 0.0;
    for (int f = frag_first[i]; f < frag_first[i + 1]; ++f) acc += partial[f];  // fixed order
    y[row] = (V)acc;
}

// Plain vector-per-row kernel: VEC lanes per row, lane-strided loop, xor-shuffle reduction.
template <int VEC, typename V, int BATCH = kVecBatch>
__global__ void __launch_bounds__(256)
csr_vector_kernel(int row_begin, int row_end, const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                  const V *__restrict__ values, const V *__restrict__ x, V *__restrict__ y,
                  int accumulate) {
    const long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = row_begin + gt / VEC;
    const int lane = threadIdx.x & (VEC - 1);
    const bool live = row < row_end;
    int lo = 0, hi = 0;
    if (live) {
        lo = __ldg(row_ptr + row);
        hi = __ldg(row_ptr + row + 1);
    }
    // kVecBatch column/value loads are issued before the first gather and the gathers before the first fma: the
    // column -> x dependency costs one round trip per batch instead of one per element
    double acc = (VEC == 1 && accumulate && live) ? (double)y[row] : 0.0;  // one lane per row: y += A x in the serial loop's order
    constexpr int kBatch = VEC == 1 ? kRowBatch : BATCH;
    for (int k = lo + lane; k < hi; k += kBatch * VEC) {
        int c[kBatch];
        double v[kBatch], xv[kBatch];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) c[u] = k + u * VEC < hi ? load_col<VEC>(col_idx + k + u * VEC) : -1;
#pragma unroll
        for (int u = 0; u < kBatch; ++u) v[u] = k + u * VEC < hi ? load_val<VEC, V>(values + k + u * VEC) : 0.0;
#pragma unroll
        for (int u = 0; u < kBatch; ++u) xv[u] = c[u] >= 0 ? ldg_x(x, c[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < kBatch; ++u)
            if (c[u] >= 0) {
                if constexpr (VEC == 1) acc = __dadd_rn(acc, __dmul_rn(v[u], xv[u]));  // one lane, index order: the serial loop
                else acc = fma(v[u], xv[u], acc);
            }
    }
#pragma unroll
    for (int off = VEC >> 1; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (live && lane == 0) y[row] = (V)((accumulate && VEC > 1) ? (double)y[row] + acc : acc);
}

// The same with 128-bit column / 256-bit value loads: every lane owns whole ALIGNED groups of four consecutive nonzeros
// (group g = the elements [4g, 4g+4) of the arrays; the first and last group of a row are masked to the row).  One
// LDG.128 + one LDG.256 + four gathers per four nonzeros instead of eight scalar loads + four gathers: on uniform 32/row
// the scalar kernel sat at 86-90 % L1TEX (LSU instruction issue) while the HLL slice kernel, which already loads like
// this, was 15 % faster on the same data (gather_bench, profiles/r02a_gather_bench.md).  GROUPS groups per lane are in
// flight per step.  safe_nnz: elements that vector loads may touch (the arrays of owned matrices are padded to a
// multiple of four; a wrapped array is only read up to nnz & ~3 this way, the ragged end goes element by element).
template <typename V>
__device__ __forceinline__ void load_group(const int *__restrict__ col_idx, const V *__restrict__ values, int g, int lo, int hi,
                                           int safe_nnz, int (&c)[4], double (&v)[4]) {
    if (g + 4 <= safe_nnz) {
        const int4 cc = ldg_stream_s32x4(col_idx + g);
        ldg_stream_f64x4(values + g, v);
        c[0] = cc.x; c[1] = cc.y; c[2] = cc.z; c[3] = cc.w;
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (g + e < lo || g + e >= hi) c[e] = -1;
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const bool on = g + e >= lo && g + e < hi;
            c[e] = on ? ldg_stream_s32(col_idx + g + e) : -1;
            v[e] = on ? ldg_stream_f64(values + g + e) : 0.0;
        }
    }
}

template <int VEC, int GROUPS, typename V>
__global__ void __launch_bounds__(256)
csr_vector4_kernel(int row_begin, int row_end, const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                   const V *__restrict__ values, const V *__restrict__ x, V *__restrict__ y, int accumulate, int safe_nnz) {
    const long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = row_begin + gt / VEC;
    const int lane = threadIdx.x & (VEC - 1);
    const bool live = row < row_end;
    int lo = 0, hi = 0;
    if (live) {
        lo = __ldg(row_ptr + row);
        hi = __ldg(row_ptr + row + 1);
    }
    double acc = 0.0;
    for (int g = (lo & ~3) + 4 * lane; g < hi; g += 4 * VEC * GROUPS) {
        int c[GROUPS][4];
        double v[GROUPS][4], xv[GROUPS][4];
#pragma unroll
        for (int u = 0; u < GROUPS; ++u) {
            if (g + 4 * VEC * u < hi) {
                load_group(col_idx, values, g + 4 * VEC * u, lo, hi, safe_nnz, c[u], v[u]);
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) c[u][e] = -1;
            }
        }
#pragma unroll
        for (int u = 0; u < GROUPS; ++u)
#pragma unroll
            for (int e = 0; e < 4; ++e) xv[u][e] = c[u][e] >= 0 ? ldg_x(x, c[u][e]) : 0.0;
#pragma unroll
        for (int u = 0; u < GROUPS; ++u)
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (c[u][e] >= 0) acc = fma(v[u][e], xv[u][e], acc);
    }
#pragma unroll
    for (int off = VEC >> 1; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (live && lane == 0) y[row] = (V)(accumulate ? (double)y[row] + acc : acc);
}

// The row loop of every thread-per-row CSR kernel: acc plus the products of row [lo, hi), BATCH column/value loads issued
// before the first gather.  One lane, index order, mul and add rounded separately: every row is bit-identical to the
// reference's serial loop (src/csr_matrix.c:134-138).
template <int BATCH, typename V>
__device__ __forceinline__ double row_sum(int lo, int hi, const int *__restrict__ col_idx, const V *__restrict__ values,
                                          const V *__restrict__ x, double acc) {
    for (int k = lo; k < hi; k += BATCH) {
        int c[BATCH];
        double v[BATCH], xv[BATCH];
#pragma unroll
        for (int u = 0; u < BATCH; ++u) c[u] = k + u < hi ? __ldg(col_idx + k + u) : -1;
#pragma unroll
        for (int u = 0; u < BATCH; ++u) v[u] = k + u < hi ? (double)__ldg(values + k + u) : 0.0;
#pragma unroll
        for (int u = 0; u < BATCH; ++u) xv[u] = c[u] >= 0 ? (double)__ldg(x + c[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < BATCH; ++u)
            if (c[u] >= 0) acc = __dadd_rn(acc, __dmul_rn(v[u], xv[u]));
    }
    return acc;
}

// One THREAD per row (stencil-like matrices, every row short).  Lane i walks row i: a warp's loads are strided by the
// row length, so a sector is consumed over several iterations and must live in L1 in between -- plain read-only
// loads that allocate, no shared memory (all 256 KB are L1), 8 CTAs x 256 threads per SM.  It is the reference's own
// thread-per-row idea (cuda_src/csr_matrix_cuda.cu:122-146), which at 6.0 TB/s on lap2d 4096^2 is the kernel to beat on
// this chip.
template <int BATCH, typename V>
__global__ void __launch_bounds__(256, 8)
csr_row_kernel(int row_begin, int row_end, const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
               const V *__restrict__ values, const V *__restrict__ x, V *__restrict__ y, int accumulate) {
    const long long row = row_begin + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= row_end) return;
    const int lo = __ldg(row_ptr + row), hi = __ldg(row_ptr + row + 1);
    y[row] = (V)row_sum<BATCH>(lo, hi, col_idx, values, x, accumulate ? (double)y[row] : 0.0);
}

// csr_row_kernel in a second form (round 2e; candidates of the fp32 path): ROWS rows per thread, CTAS CTAs per SM, and --
// the part that pays -- predicates that are INDEX ARITHMETIC only.  csr_row_kernel marks a slot past the end of its row
// with column -1 and predicates the gather and the add on the LOADED column; ptxas then issues 9-12 of a step's 17 loads,
// stalls on the first gather, and only then requests the rest (cuobjdump, tools/rowm_survey.py).  Here such a slot
// gathers x[0] (always a valid address: the loop only runs when the matrix has a nonzero) and is skipped by `k < hi`, so
// ptxas may issue every load of a step ahead of the first multiply.  Measured on lap2d 4096^2 with fp32 storage
// (profiles/r02e_rowm_probe_second_pass.log): <5 loads, 1 row, 8 CTAs> 152.3 us against 155.0 us for the best
// csr_row_kernel batch; its HLL twin 145.8 against 166.5 us.  It is a scheduling lottery, not a law: on lap3d 256^3 the
// old form wins (183 against 197 us), and with fp64 storage it wins everywhere -- hence candidates timed at plan time.
// ROWS > 1 (a thread owns rows t, t + 256, ... of its CTA's 256*ROWS rows; register budget 65536 / (256 CTAS)) was the
// hypothesis this kernel was written for -- "the fp32 kernels are latency bound, so put more rows in flight per SM than
// the 2048 threads an SM can hold" -- and the measurement REFUTED it: every multi-row form is 4-40 % slower than the
// one-row forms, fp32 and fp64, CSR and HLL (profiles/r02e_rowm_probe_first_pass.log).  Three such forms stay in the
// table so that the record can be re-measured.  Every row is summed by one lane in index order, mul and add rounded
// separately, skipped slots skipped: the same bits as csr_row_kernel (tests/test_gpu_parity.py walks all forms).
// Also tried on this kernel and removed (profiles/r02e_rowm_probe_third_pass.log): one lane per warp prefetching into L2
// the row_ptr line of the warp N CTAs further on, so that the first of that warp's three round trips ends in L2 -- CSR
// fp32 lap2d 152 us at N = 148, 162-166 us from N = 592 up, against 152-156 without; and the extra parameter alone moved
// ptxas from 15 to 12 of 18 loads ahead of the first multiply.
template <int BATCH, int ROWS, int CTAS, typename V>
__global__ void __launch_bounds__(256, CTAS)
csr_rowm_kernel(int row_begin, int row_end, const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                const V *__restrict__ values, const V *__restrict__ x, V *__restrict__ y, int accumulate) {
    const long long first = row_begin + (long long)blockIdx.x * (256 * ROWS) + threadIdx.x;
    int lo[ROWS], hi[ROWS];
    double acc[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
        const long long row = first + (long long)r * 256;
        const bool live = row < row_end;
        lo[r] = live ? __ldg(row_ptr + row) : 0;
        hi[r] = live ? __ldg(row_ptr + row + 1) : 0;
    }
    int longest = 0;
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
        const long long row = first + (long long)r * 256;
        acc[r] = accumulate && row < row_end ? (double)y[row] : 0.0;
        longest = max(longest, hi[r] - lo[r]);
    }
    for (int s = 0; s < longest; s += BATCH) {
        int c[ROWS][BATCH];
        V v[ROWS][BATCH], xv[ROWS][BATCH];
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
            for (int u = 0; u < BATCH; ++u) c[r][u] = lo[r] + s + u < hi[r] ? __ldg(col_idx + lo[r] + s + u) : 0;
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
            for (int u = 0; u < BATCH; ++u) v[r][u] = lo[r] + s + u < hi[r] ? __ldg(values + lo[r] + s + u) : (V)0;
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
            for (int u = 0; u < BATCH; ++u) xv[r][u] = __ldg(x + c[r][u]);
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
            for (int u = 0; u < BATCH; ++u)
                if (lo[r] + s + u < hi[r]) acc[r] = __dadd_rn(acc[r], __dmul_rn((double)v[r][u], (double)xv[r][u]));
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
        const long long row = first + (long long)r * 256;
        if (row < row_end) y[row] = (V)acc[r];
    }
}

// (ROWS, BATCH, CTAS per SM) forms of csr_rowm_kernel offered to the plan-time tuner of the fp32 path (tools/rowm_survey.py
// prints registers, spills and the load schedule of each; tools/rowm_probe.py times them).
struct RowmVariant {
    int rows, batch, ctas;
};
#define SPMV_ROWM_VARIANTS(X) \
    X(1, 4, 8) X(1, 5, 8) X(1, 6, 8) X(1, 7, 8) X(1, 5, 6) X(2, 3, 5) X(2, 4, 5) X(3, 3, 5)
#define ROWM_ENTRY(R, B, C) {R, B, C},
static const RowmVariant kRowmVariants[] = {SPMV_ROWM_VARIANTS(ROWM_ENTRY)};
#undef ROWM_ENTRY
constexpr int kNumRowmVariants = (int)(sizeof kRowmVariants / sizeof kRowmVariants[0]);

// csr_row_kernel with the tail of the two-launch iterated product (spmv_b200_csr_spmv_fused_flat): one thread per row,
// one CTA per 256 rows, NO chunk walk and no waiting -- the body of the plain kernel, then: multiply by 1/|w_prev| (read
// from memory, computed once by the exchange kernel), store, mirror boundary rows into the peers, one partial sum of
// squares per CTA.  (Round 2: the same epilogue on a chunk walk, grid-stride or C chunks per CTA, stayed 5-25 % behind the
// plain kernel whatever the batch -- profiles/r02k_diag_flatpick.log; this form is the plain kernel plus ~15 instructions.)
template <int BATCH>
__global__ void __launch_bounds__(256, 8)
csr_row_flat_kernel(int M, const int *__restrict__ row_ptr, const int *__restrict__ col_idx, const double *__restrict__ values,
                    const double *__restrict__ x, double *__restrict__ y, const __grid_constant__ Epilogue ep) {
    __shared__ double warp_sq[8];
    const long long row = (long long)blockIdx.x * 256 + threadIdx.x;
    const bool live = row < M;
    double acc = 0.0;
    if (live) {
        const int lo = __ldg(row_ptr + row), hi = __ldg(row_ptr + row + 1);
        acc = row_sum<BATCH>(lo, hi, col_idx, values, x, 0.0);
        if (ep.inv_norm != nullptr) acc *= __ldg(ep.inv_norm);
        y[row] = acc;
        if (fused_chunk_is_boundary(ep, (long long)blockIdx.x * 256)) fused_peer_store(ep, row, acc);
    }
    if (ep.partials == nullptr) return;
    double sq = acc * acc;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, off);
    if ((threadIdx.x & 31) == 0) warp_sq[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double total = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) total += warp_sq[w];
        ep.partials[blockIdx.x] = total;
    }
}

// The thread-per-row kernel with the fused tail of the iterated product (Epilogue, handles.cuh): every row is divided by
// |w_prev|, squared into a per-thread sum, stored, and mirrored into the peers that reference it; per-CTA partial sums
// in a fixed order; with a mailbox the launch first waits for the peers' previous launch and its last CTA publishes
// |w|^2 (common.cuh).  A fixed grid walks the rows in 256-row chunks (grid-stride), so the number of partials -- and the
// order of the sum of squares -- does not depend on the matrix size.
template <int BATCH>
__global__ void __launch_bounds__(256, 8)
csr_row_fused_kernel(int M, const int *__restrict__ row_ptr, const int *__restrict__ col_idx, const double *__restrict__ values,
                     const double *__restrict__ x, double *__restrict__ y, const __grid_constant__ Epilogue ep) {
    __shared__ double warp_sq[8];
    __shared__ double mail_total;
    bool scaled;
    const double inv_norm = fused_inv_norm(ep, scaled, &mail_total);
    double sq = 0.0;
    const int chunks = (M + 255) >> 8;
    for (int q = blockIdx.x; q < chunks; q += gridDim.x) {
        // boundary chunks first (ChunkOrder); peer stores: a CTA-uniform test on the chunk (uniform datapath), the per-row
        // range test only inside -- done per row for every row it cost 30 us per peer per 56 M rows
        const long long chunk_lo = (long long)ordered_chunk(ep.order, q) * 256;
        const bool boundary = ep.order.boundary_chunks > 0 ? q < ep.order.boundary_chunks : fused_chunk_is_boundary(ep, chunk_lo);
        const long long row = chunk_lo + threadIdx.x;
        if (row >= M) continue;
        const int lo = __ldg(row_ptr + row), hi = __ldg(row_ptr + row + 1);
        double acc = row_sum<BATCH>(lo, hi, col_idx, values, x, 0.0);
        if (scaled) acc *= inv_norm;
        sq = fma(acc, acc, sq);
        y[row] = acc;
        if (boundary) fused_peer_store(ep, row, acc);
    }
    fused_finish(ep, sq, warp_sq);
}

// Asynchronous fused product (spmv_b200_csr_spmv_fused_async, spmv_b200.h): the fused row kernel with (1) the chunks
// that hold rows a neighbour references moved to the front of the walk and a per-neighbour halo tag raised as soon as
// they are stored, (2) the scale factor taken from the sums of launch k-2, (3) waits only on things that finished a
// launch ago.  Chunk = 256 consecutive rows; q-th chunk of the walk -> row chunk through the boundary intervals.
struct AsyncArgs {  // one by-value kernel parameter, read through the constant bank (never address-taken: a copy on the
    spmv_b200_peers_t peers;   // local-memory stack would put two extra loads per row on the LSU)
    spmv_b200_async_t as;
    ChunkOrder order;
};

template <int BATCH>
__global__ void __launch_bounds__(256, 8)
csr_row_async_kernel(int M, const int *__restrict__ row_ptr, const int *__restrict__ col_idx, const double *__restrict__ values,
                     const double *__restrict__ x, double *__restrict__ y, double *__restrict__ partials,
                     const __grid_constant__ AsyncArgs args) {
#define peers args.peers
#define as args.as
#define order args.order
    __shared__ double warp_sq[8];
    __shared__ double s_scale;
    __shared__ unsigned int s_arrived;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long k = as.iteration;
    // ---- start: sums of launch k-2 (slot (k-2)%4, tag k-1) and halo tags >= k from the ranks I read from ----
    if (warp == 0) {
        double mine = 0.0;
        const long long t0 = clock64();
        if (k >= 2 && lane < as.world) {
            const unsigned long long *slot = as.box[as.rank] + 2 * ((int)((k - 2) & 3) * as.world + lane);
            while (ld_acquire_sys(slot + 1) != k - 1) {
                if (clock64() - t0 > kMailSpinCycles) {
                    *as.status = 1;
                    break;
                }
                __nanosleep(40);
            }
            mine = __longlong_as_double((long long)ld_acquire_sys(slot));
        }
        if (k >= 1 && lane < as.num_recv) {
            const unsigned long long *halo = as.box[as.rank] + 2 * 4 * as.world + as.recv_from[lane];
            while (ld_acquire_sys(halo) < k) {
                if (clock64() - t0 > kMailSpinCycles) {
                    *as.status = 2;
                    break;
                }
                __nanosleep(40);
            }
        }
        double total = 0.0;
        for (int r = 0; r < as.world; ++r) total += __shfl_sync(0xffffffffu, mine, r);
        if (lane == 0) s_scale = k >= 2 ? 1.0 / sqrt(total) : 1.0;
    }
    __syncthreads();
    const double scale = s_scale;
    const int chunks = (M + 255) >> 8;
    // boundary chunks of this CTA: q = blockIdx.x, blockIdx.x + gridDim.x, ... < boundary_chunks -- the first ones of its walk
    const int my_boundary = order.boundary_chunks > (int)blockIdx.x
                                ? (order.boundary_chunks - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    int walked = 0;
    double sq = 0.0;
    for (int q = blockIdx.x; q < chunks; q += gridDim.x) {
        int chunk = q;  // q-th chunk of the walk -> row chunk: the boundary intervals first, then the rest in order
        if (q < order.boundary_chunks) {
            int left = q;
            for (int i = 0; i < order.count; ++i) {
                const int len = order.hi[i] - order.lo[i];
                if (left < len) {
                    chunk = order.lo[i] + left;
                    break;
                }
                left -= len;
            }
        } else {
            chunk = q - order.boundary_chunks;
            for (int i = 0; i < order.count; ++i)
                if (chunk >= order.lo[i]) chunk += order.hi[i] - order.lo[i];
        }
        const long long row = (long long)chunk * 256 + threadIdx.x;
        if (row < M) {
            const int lo = __ldg(row_ptr + row), hi = __ldg(row_ptr + row + 1);
            double acc = row_sum<BATCH>(lo, hi, col_idx, values, x, 0.0);
            acc *= scale;
            sq = fma(acc, acc, sq);
            y[row] = acc;
            if (order.boundary_chunks == 0 || q < order.boundary_chunks)
                for (int p = 0; p < peers.count; ++p)
                    if (row >= peers.lo[p] && row < peers.hi[p]) peers.dst[p][row] = acc;
        }
        if (++walked == my_boundary) {  // CTA-uniform: the last chunk of this CTA that feeds a neighbour is stored
            // Ordering of the peer stores before the halo tag: CTA barrier, then a DEVICE-scope fence + device-scope
            // atomic by thread 0 (release pattern towards the CTA that completes the count), then that CTA's
            // system-scope fence + st.release.sys of the tag.  Every edge is morally strong at its own scope, so the peer
            // stores precede the tag in causality order and the neighbour's ld.acquire.sys of the tag orders its reads
            // after them.  A system-scope fence HERE costs ~0.1 us per CTA, serialised, while the SMs are busy (measured:
            // 0.313 vs 0.272 ms per iteration on 2 GPUs at 320^3) -- only the one CTA that raises the tags pays it.
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                s_arrived = atomicAdd(as.bcounter, (unsigned int)my_boundary);
            }
            __syncthreads();
            if (s_arrived + (unsigned int)my_boundary == (unsigned int)order.boundary_chunks && warp == 0) {
                __threadfence_system();  // every boundary row of this rank is in the neighbours' buffers: raise their tags
                if (lane < peers.count) st_release_sys(as.box[as.send_to[lane]] + 2 * 4 * as.world + as.rank, k + 1);
                if (lane == 0) *as.bcounter = 0;
            }
        }
    }
    // ---- end: per-CTA partial, last CTA publishes the rank's sum for launch k in slot k%4 with tag k+1 ----
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, off);
    if (lane == 0) warp_sq[warp] = sq;
    __syncthreads();  // the peers only ever read the boundary rows (fenced above) and the sums (released below)
    if (warp == 0) {
        unsigned int arrived = 0;
        if (lane == 0) {
            double total = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) total += warp_sq[w];
            partials[blockIdx.x] = total;
            if (order.boundary_chunks == 0) __threadfence_system(); else __threadfence();
            arrived = atomicAdd(as.counter, 1u);
        }
        arrived = __shfl_sync(0xffffffffu, arrived, 0);
        if (arrived == gridDim.x - 1) {
            __threadfence();
            if (order.boundary_chunks == 0 && lane < peers.count)  // experiment / degenerate ranges: tags at the end
                st_release_sys(as.box[as.send_to[lane]] + 2 * 4 * as.world + as.rank, k + 1);
            const double part = warp_sum_partials(partials, (int)gridDim.x, lane);
            if (lane < as.world) {
                unsigned long long *slot = as.box[lane] + 2 * ((int)(k & 3) * as.world + as.rank);
                st_relaxed_sys(slot, (unsigned long long)__double_as_longlong(part));
                st_release_sys(slot + 1, k + 1);
            }
            if (lane == 0) *as.counter = 0;
        }
    }
}

#undef peers
#undef as
#undef order

// ---- row-binned vector kernel (skewed matrices) ------------------------------------------------------
// Rows are binned by length at plan time; bin b < 6 gives every row 2^b lanes (about a quarter of its length, so
// each lane owns one batch of kVecBatch gathers), the rows of one bin are processed in ascending row order, and all
// bins run in ONE launch (a CTA finds its bin from block_start[]).  No shared memory: the whole L1 stays available
// to the gathers of x -- on this chip the number of gathers in flight is bounded by L1 lines, and gather-heavy
// kernels lose more to a smaller L1 than they gain from staging (profiles/r01d_kernel_selection.md).
constexpr int kBinLongThreshold = 2048;  // rows above this are split into kFragNnz fragments (csr_long_* kernels)

__host__ __device__ __forceinline__ int bin_of(int len) {
    if (len <= 8) return 0;
    if (len <= 12) return 1;
    if (len <= 24) return 2;
    if (len <= 48) return 3;
    if (len <= 96) return 4;
    return len <= kBinLongThreshold ? 5 : 6;
}

struct BinLaunch {
    int offset[kBins + 1];
    int block_start[kBins];
    int frag_blocks;            // CTAs [0, frag_blocks) of the launch own one fragment of a long row each (heaviest work first)
    int safe_nnz;               // >= 0: multi-lane classes use aligned groups of four (elements vector loads may touch)
    int num_long;
    const int *frag_first;
    double *frag_partial;
};

template <int VEC, typename V>
__device__ __forceinline__ void binned_rows(int local_block, int first, int count, const int *__restrict__ bin_rows,
                                            const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                                            const V *__restrict__ values, const V *__restrict__ x,
                                            V *__restrict__ y, int accumulate) {
    const int idx = (local_block * 256 + (int)threadIdx.x) / VEC;
    const int lane = threadIdx.x & (VEC - 1);
    const bool live = idx < count;
    int row = 0, lo = 0, hi = 0;
    if (live) {
        row = __ldg(bin_rows + first + idx);
        lo = __ldg(row_ptr + row);
        hi = __ldg(row_ptr + row + 1);
    }
    double acc = (VEC == 1 && accumulate && live) ? (double)y[row] : 0.0;
    constexpr int kBatch = VEC == 1 ? kRowBatch : kVecBatch;
    for (int k = lo + lane; k < hi; k += kBatch * VEC) {
        int c[kBatch];
        double v[kBatch], xv[kBatch];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) c[u] = k + u * VEC < hi ? load_col<VEC>(col_idx + k + u * VEC) : -1;
#pragma unroll
        for (int u = 0; u < kBatch; ++u) v[u] = k + u * VEC < hi ? load_val<VEC, V>(values + k + u * VEC) : 0.0;
#pragma unroll
        for (int u = 0; u < kBatch; ++u) xv[u] = c[u] >= 0 ? ldg_x(x, c[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < kBatch; ++u)
            if (c[u] >= 0) {
                if constexpr (VEC == 1) acc = __dadd_rn(acc, __dmul_rn(v[u], xv[u]));  // one lane, index order: the serial loop
                else acc = fma(v[u], xv[u], acc);
            }
    }
#pragma unroll
    for (int off = VEC >> 1; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (live && lane == 0) y[row] = (V)((accumulate && VEC > 1) ? (double)y[row] + acc : acc);
}

// the same rows with aligned groups of four (load_group): one LDG.128 + one LDG.256 per four nonzeros
template <int VEC, typename V>
__device__ __forceinline__ void binned_rows4(int local_block, int first, int count, const int *__restrict__ bin_rows,
                                             const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                                             const V *__restrict__ values, const V *__restrict__ x,
                                             V *__restrict__ y, int accumulate, int safe_nnz) {
    const int idx = (local_block * 256 + (int)threadIdx.x) / VEC;
    const int lane = threadIdx.x & (VEC - 1);
    const bool live = idx < count;
    int row = 0, lo = 0, hi = 0;
    if (live) {
        row = __ldg(bin_rows + first + idx);
        lo = __ldg(row_ptr + row);
        hi = __ldg(row_ptr + row + 1);
    }
    double acc = 0.0;
    for (int g = (lo & ~3) + 4 * lane; g < hi; g += 4 * VEC) {
        int c[4];
        double v[4], xv[4];
        load_group(col_idx, values, g, lo, hi, safe_nnz, c, v);
#pragma unroll
        for (int e = 0; e < 4; ++e) xv[e] = c[e] >= 0 ? ldg_x(x, c[e]) : 0.0;
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (c[e] >= 0) acc = fma(v[e], xv[e], acc);
    }
#pragma unroll
    for (int off = VEC >> 1; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (live && lane == 0) y[row] = (V)(accumulate ? (double)y[row] + acc : acc);
}

template <typename V>
__global__ void __launch_bounds__(256)
csr_binned_kernel(const __grid_constant__ BinLaunch plan, const int *__restrict__ bin_rows, const int *__restrict__ row_ptr,
                  const int *__restrict__ col_idx, const V *__restrict__ values, const V *__restrict__ x,
                  V *__restrict__ y, int accumulate) {
    if ((int)blockIdx.x < plan.frag_blocks) {  // CTA-uniform: a fragment of one of the longest rows (combined afterwards)
        long_fragment<V>((int)blockIdx.x, bin_rows + plan.offset[kBins - 1], plan.frag_first, plan.num_long, row_ptr, col_idx,
                         values, x, plan.frag_partial);
        return;
    }
    const int block = (int)blockIdx.x - plan.frag_blocks;
    int bin = 0;
    while (bin < kBins - 2 && block >= plan.block_start[bin + 1]) ++bin;  // CTA-uniform
    const int local_block = block - plan.block_start[bin];
    const int first = plan.offset[bin], count = plan.offset[bin + 1] - first;
    if (plan.safe_nnz >= 0 && bin > 0) {  // CTA-uniform: aligned-group loads for the multi-lane classes
        switch (bin) {
            case 1: binned_rows4<2, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate, plan.safe_nnz); break;
            case 2: binned_rows4<4, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate, plan.safe_nnz); break;
            case 3: binned_rows4<8, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate, plan.safe_nnz); break;
            case 4: binned_rows4<16, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate, plan.safe_nnz); break;
            default: binned_rows4<32, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate, plan.safe_nnz); break;
        }
        return;
    }
    switch (bin) {
        case 0: binned_rows<1, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate); break;
        case 1: binned_rows<2, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate); break;
        case 2: binned_rows<4, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate); break;
        case 3: binned_rows<8, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate); break;
        case 4: binned_rows<16, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate); break;
        default: binned_rows<32, V>(local_block, first, count, bin_rows, row_ptr, col_idx, values, x, y, accumulate); break;
    }
}

__global__ void bin_key_kernel(int M, const int *__restrict__ row_ptr, unsigned char *__restrict__ keys,
                               int *__restrict__ ids, int *__restrict__ counts) {
    __shared__ int local[kBins];
    if (threadIdx.x < kBins) local[threadIdx.x] = 0;
    __syncthreads();
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < M) {
        const int b = bin_of(row_ptr[r + 1] - row_ptr[r]);
        keys[r] = (unsigned char)b;
        ids[r] = (int)r;
        atomicAdd(&local[b], 1);
    }
    __syncthreads();
    if (threadIdx.x < kBins && local[threadIdx.x]) atomicAdd(&counts[threadIdx.x], local[threadIdx.x]);  // integer: order independent
}

struct RemapTable {
    int nparts;
    long long starts[SPMV_B200_MAX_RANKS + 1];
    long long stride;
};

__global__ void remap_columns_kernel(long long nnz, int *__restrict__ col_idx, const __grid_constant__ RemapTable t) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nnz) return;
    const long long c = col_idx[k];
    int p = 0;
    while (p + 1 < t.nparts && c >= t.starts[p + 1]) ++p;
    col_idx[k] = (int)(p * t.stride + (c - t.starts[p]));
}

// out[0] = 1 + last row below `mid` that references a column outside [col_lo, col_hi) (0 if none);
// out[1] = first such row at or above `mid` (M if none).  Integer max / min: order independent.
__global__ void interior_rows_kernel(int M, int mid, const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                                     long long col_lo, long long col_hi, int *__restrict__ out) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= M) return;
    const int lo = row_ptr[r], hi = row_ptr[r + 1];
    bool outside = false;
    if (hi > lo) outside = col_idx[lo] < col_lo || col_idx[hi - 1] >= col_hi;  // rows are column-sorted
    if (!outside) return;
    if (r < mid) atomicMax(out, (int)r + 1);
    else atomicMin(out + 1, (int)r);
}

// The exchange of the two-launch iterated product (spmv_b200_mail_exchange).  (1) the partials of the flat product kernel,
// added in a fixed order: CTA g adds chunk g (thread t its contiguous block left to right, then a fixed tree); with more
// than one CTA the chunk sum replaces the chunk's first element and the LAST CTA to arrive (ticket in mail.counter, one
// device-scope fence per CTA -- at most 64 of them) adds the chunk sums in chunk order and carries on alone: one SM read
// 8 KB of partials per microsecond, which put 8 / 17 / 30 us on the critical path of every iteration at 8 / 4 / 2 GPUs;
// (2) {sum, tag k+1} into slot [k&1][rank] of every rank's mailbox -- the product kernel has completed (stream order), a
// system-scope fence and a release store order its peer stores before the tag; (3) wait for the tags of all ranks in the own
// mailbox, add their sums in rank order, leave {|w_k|^2, 1/|w_k|} in sumsq_out[0..1] for the next product launch.
__global__ void __launch_bounds__(1024)
mail_exchange_kernel(double *__restrict__ partials, int count, int chunk, const __grid_constant__ spmv_b200_mail_t mail,
                     double *__restrict__ sumsq_out) {
    __shared__ double part[1024];
    __shared__ int is_last;
    const int c_lo = (int)blockIdx.x * chunk, c_hi = min(count, c_lo + chunk);
    // thread t adds ITS contiguous block of the chunk (a multiple of 4 elements) left to right; the loads of a block are
    // independent 256-bit loads, all in flight at once
    const int per = ((((c_hi - c_lo) + 1023) >> 10) + 3) & ~3;
    const int lo = c_lo + (int)threadIdx.x * per, hi = min(c_hi, lo + per);
    double s = 0.0;
    if ((reinterpret_cast<uintptr_t>(partials) & 31) == 0) {
        constexpr int kGroup = 8;  // 8 x 4 doubles per round
        for (int base = lo; base < hi; base += 4 * kGroup) {
            double v[kGroup][4];
#pragma unroll
            for (int g = 0; g < kGroup; ++g) {
                const int at = base + 4 * g;
                if (at + 4 <= hi) {
                    asm volatile("ld.global.cg.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v[g][0]), "=d"(v[g][1]), "=d"(v[g][2]), "=d"(v[g][3]) : "l"(partials + at));
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e) v[g][e] = at + e < hi ? __ldcg(partials + at + e) : 0.0;
                }
            }
#pragma unroll
            for (int g = 0; g < kGroup; ++g)
#pragma unroll
                for (int e = 0; e < 4; ++e) s += v[g][e];
        }
    } else {
        for (int i = lo; i < hi; ++i) s += __ldcg(partials + i);
    }
    part[threadIdx.x] = s;
    __syncthreads();
    for (int half = 512; half > 0; half >>= 1) {
        if ((int)threadIdx.x < half) part[threadIdx.x] += part[threadIdx.x + half];
        __syncthreads();
    }
    const int lane = threadIdx.x;
    double mine = part[0];
    if (gridDim.x > 1) {
        if (threadIdx.x == 0) {
            partials[c_lo] = mine;  // only this CTA read the chunk
            __threadfence();
            is_last = atomicAdd(mail.counter, 1u) == gridDim.x - 1;
        }
        __syncthreads();
        if (!is_last || threadIdx.x >= 32) return;
        __threadfence();
        const int chunks = (int)gridDim.x;  // <= 64
        const double a = lane < chunks ? __ldcg(partials + (long long)lane * chunk) : 0.0;
        const double b = lane + 32 < chunks ? __ldcg(partials + (long long)(lane + 32) * chunk) : 0.0;
        mine = 0.0;
        for (int g = 0; g < min(chunks, 32); ++g) mine += __shfl_sync(0xffffffffu, a, g);
        for (int g = 32; g < chunks; ++g) mine += __shfl_sync(0xffffffffu, b, g - 32);
        if (lane == 0) *mail.counter = 0;  // every CTA has drawn its ticket: ready for the next launch
    } else if (threadIdx.x >= 32) {
        return;
    }
    if (mail.world == 1) {  // nobody to talk to
        if (lane == 0) {
            sumsq_out[0] = mine;
            sumsq_out[1] = 1.0 / sqrt(mine);
        }
        return;
    }
    __threadfence_system();
    if (lane < mail.world) {
        unsigned long long *slot = mail.box[lane] + 2 * ((int)(mail.iteration & 1) * mail.world + mail.rank);
        st_relaxed_sys(slot, (unsigned long long)__double_as_longlong(mine));
        st_release_sys(slot + 1, mail.iteration + 1);
    }
    double got = 0.0;
    if (lane < mail.world) {
        const unsigned long long *slot = mail.box[mail.rank] + 2 * ((int)(mail.iteration & 1) * mail.world + lane);
        const long long t0 = clock64();
        while (ld_acquire_sys(slot + 1) != mail.iteration + 1) {
            if (clock64() - t0 > kMailSpinCycles) {
                *mail.status = 1;
                break;
            }
            __nanosleep(40);
        }
        got = __longlong_as_double((long long)ld_acquire_sys(slot));
    }
    double total = 0.0;
    for (int r = 0; r < mail.world; ++r) total += __shfl_sync(0xffffffffu, got, r);
    if (lane == 0) {
        sumsq_out[0] = total;
        sumsq_out[1] = 1.0 / sqrt(total);  // the next product launch multiplies by this: no square root or division per thread
    }
}

__global__ void to_f32_kernel(const double *__restrict__ in, float *__restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)in[i];  // round to nearest even
}

// ---- plan construction kernels ------------------------------------------------------------------
// boundary[r] = 1 when row r opens a tile: first row, a new window of D stream words (every
// nonzero streams 12 bytes = 3 words, every row 4 bytes = 1 word of row_ptr, so 3*row_ptr[r] + r
// counts the 4-byte words that precede row r), or a neighbour of / a long row.  All tiles therefore
// carry (nearly) the same number of bytes, whatever the row lengths.
__global__ void plan_flag_kernel(int M, const int *__restrict__ row_ptr, int tile_items, int long_threshold,
                                 unsigned char *__restrict__ boundary, unsigned char *__restrict__ is_long,
                                 int *__restrict__ max_row) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int len = 0;
    if (r < M) len = row_ptr[r + 1] - row_ptr[r];
    const int warp_max = __reduce_max_sync(0xffffffffu, len);
    if ((threadIdx.x & 31) == 0 && warp_max > 0) atomicMax(max_row, warp_max);  // integer max: order independent
    if (r >= M) return;
    const int a = row_ptr[r], b = row_ptr[r + 1];
    const bool long_here = b - a > long_threshold;
    bool open = r == 0 || long_here;
    if (r > 0) {
        const int before = row_ptr[r - 1];
        open = open || (a - before > long_threshold);
        open = open || (3LL * a + r) / tile_items != (3LL * before + r - 1) / tile_items;
    }
    boundary[r] = open ? 1 : 0;
    is_long[r] = long_here ? 1 : 0;
}

__global__ void plan_tiles_kernel(int num_tiles, int M, const int *__restrict__ tile_rows,
                                  const int *__restrict__ row_ptr, int2 *__restrict__ tiles) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > num_tiles) return;
    const int row = t < num_tiles ? tile_rows[t] : M;
    tiles[t] = make_int2(row, row_ptr[row]);
}

__global__ void plan_fragcount_kernel(int num_long, const int *__restrict__ long_rows,
                                      const int *__restrict__ row_ptr, int *__restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > num_long) return;
    int c = 0;
    if (i < num_long) {
        const int row = long_rows[i];
        c = (row_ptr[row + 1] - row_ptr[row] + kFragNnz - 1) / kFragNnz;
    }
    counts[i] = c;  // counts[num_long] = 0 so that the exclusive scan ends with the total
}

}  // namespace spmv

// ================================================================================================
// handle
// ================================================================================================

namespace spmv {

static void free_bins(spmv_b200_csr *A) {
    cudaFree(A->bins.rows);
    cudaFree(A->bins.frag_first);
    cudaFree(A->bins.frag_partial);
    A->bins = BinPlan();
}

static void free_plan(spmv_b200_csr *A) {
    free_bins(A);
    cudaFree(A->tiles);
    cudaFree(A->long_rows);
    cudaFree(A->frag_first);
    cudaFree(A->frag_partial);
    cudaFree(A->spmm_partial);
    A->tiles = nullptr;
    A->long_rows = nullptr;
    A->frag_first = nullptr;
    A->frag_partial = nullptr;
    A->spmm_partial = nullptr;
    A->num_tiles = A->num_long = A->num_frag = 0;
    image_free(A->image);
}

template <typename V>
static int launch_rows(int row_begin, int row_end, const int *row_ptr, const int *col_idx, const V *values,
                       const V *x, V *y, int batch, int accumulate, cudaStream_t stream);
static int safe_vector_nnz(const spmv_b200_csr *A);
static const int kFlatCandidates[] = {2, 3, 4, 5, 6, 7};
static int flat_grid(long long M);
static int launch_fused_flat(const spmv_b200_csr *A, const double *x, double *y, const Epilogue &ep, cudaStream_t stream,
                             int batch);
static int launch_fused(const spmv_b200_csr *A, const double *x, double *y, const Epilogue &ep, cudaStream_t stream, int batch);
static int fused_row_grid(const spmv_b200_csr *A);

static int build_plan(spmv_b200_csr *A, cudaStream_t stream) {
    free_plan(A);
    host_pipe_free(A->pipe);  // the row windows of the host entry point follow the tiles
    A->pipe = nullptr;
    host_pipe_free(A->spmm_pipe);  // its multi-vector windows know which hold long rows
    A->spmm_pipe = nullptr;
    const int M = A->M;
    if (M == 0) return SPMV_B200_OK;
    unsigned char *boundary = nullptr, *is_long = nullptr;
    int *tile_rows = nullptr, *counts = nullptr, *d_selected = nullptr;
    void *temp = nullptr;
    int rc = SPMV_B200_OK;
    auto cleanup = [&]() {
        cudaFree(boundary);
        cudaFree(is_long);
        cudaFree(tile_rows);
        cudaFree(counts);
        cudaFree(d_selected);
        cudaFree(temp);
    };
#define PLAN_TRY(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t e__ = (expr);                                                                       \
        if (e__ != cudaSuccess) {                                                                       \
            rc = fail(e__ == cudaErrorMemoryAllocation ? SPMV_B200_ERR_NOMEM : SPMV_B200_ERR_CUDA,      \
                      "%s: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__);            \
            cleanup();                                                                                  \
            free_plan(A);                                                                               \
            return rc;                                                                                  \
        }                                                                                               \
    } while (0)

    // upper bounds that do not need a counting pass
    const long long max_long = A->nnz / ((long long)A->long_threshold + 1) + 1;
    const long long max_tiles = (3 * A->nnz + M) / A->tile_items + 2 + 2 * max_long;
    PLAN_TRY(cudaMalloc(&boundary, (size_t)M));
    PLAN_TRY(cudaMalloc(&is_long, (size_t)M));
    PLAN_TRY(cudaMalloc(&tile_rows, (size_t)std::min<long long>(max_tiles, M) * sizeof(int)));
    PLAN_TRY(cudaMalloc(&A->long_rows, (size_t)std::min<long long>(max_long, M) * sizeof(int)));
    PLAN_TRY(cudaMalloc(&d_selected, 3 * sizeof(int)));
    PLAN_TRY(cudaMemsetAsync(d_selected, 0, 3 * sizeof(int), stream));
    plan_flag_kernel<<<blocks_for(M, 256), 256, 0, stream>>>(M, A->row_ptr, A->tile_items, A->long_threshold,
                                                             boundary, is_long, d_selected + 2);
    PLAN_TRY(cudaGetLastError());

    thrust::counting_iterator<int> row_ids(0);
    size_t temp_a = 0, temp_b = 0;
    PLAN_TRY(cub::DeviceSelect::Flagged(nullptr, temp_a, row_ids, boundary, tile_rows, d_selected, M, stream));
    PLAN_TRY(cub::DeviceSelect::Flagged(nullptr, temp_b, row_ids, is_long, A->long_rows, d_selected + 1, M, stream));
    size_t temp_bytes = std::max(temp_a, temp_b);
    PLAN_TRY(cudaMalloc(&temp, temp_bytes ? temp_bytes : 1));
    PLAN_TRY(cub::DeviceSelect::Flagged(temp, temp_bytes, row_ids, boundary, tile_rows, d_selected, M, stream));
    PLAN_TRY(cub::DeviceSelect::Flagged(temp, temp_bytes, row_ids, is_long, A->long_rows, d_selected + 1, M, stream));
    int selected[3] = {0, 0, 0};
    PLAN_TRY(cudaMemcpyAsync(selected, d_selected, sizeof selected, cudaMemcpyDeviceToHost, stream));
    PLAN_TRY(cudaStreamSynchronize(stream));
    A->num_tiles = selected[0];
    A->num_long = selected[1];
    A->max_row = selected[2];

    PLAN_TRY(cudaMalloc(&A->tiles, (size_t)(A->num_tiles + 1) * sizeof(int2)));
    plan_tiles_kernel<<<blocks_for(A->num_tiles + 1, 256), 256, 0, stream>>>(A->num_tiles, M, tile_rows, A->row_ptr,
                                                                            A->tiles);
    PLAN_TRY(cudaGetLastError());

    if (A->num_long > 0) {
        PLAN_TRY(cudaMalloc(&counts, (size_t)(A->num_long + 1) * sizeof(int)));
        PLAN_TRY(cudaMalloc(&A->frag_first, (size_t)(A->num_long + 1) * sizeof(int)));
        plan_fragcount_kernel<<<blocks_for(A->num_long + 1, 256), 256, 0, stream>>>(A->num_long, A->long_rows,
                                                                                   A->row_ptr, counts);
        PLAN_TRY(cudaGetLastError());
        size_t temp_c = 0;
        PLAN_TRY(cub::DeviceScan::ExclusiveSum(nullptr, temp_c, counts, A->frag_first, A->num_long + 1, stream));
        if (temp_c > temp_bytes) {
            cudaFree(temp);
            temp = nullptr;
            PLAN_TRY(cudaMalloc(&temp, temp_c));
            temp_bytes = temp_c;
        }
        PLAN_TRY(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, counts, A->frag_first, A->num_long + 1, stream));
        PLAN_TRY(cudaMemcpyAsync(&A->num_frag, A->frag_first + A->num_long, sizeof(int), cudaMemcpyDeviceToHost, stream));
        PLAN_TRY(cudaStreamSynchronize(stream));
        PLAN_TRY(cudaMalloc(&A->frag_partial, (size_t)std::max(A->num_frag, 1) * sizeof(double)));
    } else {
        cudaFree(A->long_rows);
        A->long_rows = nullptr;
    }
    PLAN_TRY(cudaStreamSynchronize(stream));
#undef PLAN_TRY
    cleanup();
    // batch of the thread-per-row kernel: about the mean row length; on large matrices the candidates are timed
    // (a few products on scratch vectors) -- the best batch depends on how rows, lines and L1 capacity interact
    const int forced_batch = env_int("SPMV_B200_ROW_BATCH", 0);
    A->row_batch = std::max(2, std::min(6, (int)((A->nnz + M - 1) / std::max(M, 1))));
    A->short_rows_stream = false;
    A->fused_batch = 0;
    SPMV_TRY(stream_prepare_csr(A));
    if (forced_batch >= 1 && forced_batch <= 8) {
        A->row_batch = forced_batch;
    } else if (A->max_row <= kRowKernelMaxLen && A->nnz >= kAutotuneMinNnz && env_int("SPMV_B200_AUTOTUNE", 1)) {
        // candidates: (0) the TMA stream kernel, the row kernel with batch 2..7 and, on a matrix that owns its arrays, every
        // form of the private image it qualifies for (image.cu).  All give the same bits on such rows.  The image is held
        // only when one of its forms wins, and then in that form alone.
        CsrImage *image = nullptr;
        const int forms = A->owns && A->num_long == 0 ? image_candidates(A, stream, &image) : 0;
        int ids[7], n = 0, fallback = 0;
        ids[n++] = 0;
        for (int batch = 2; batch <= 7; ++batch) {
            if (batch == A->row_batch) fallback = n;
            ids[n++] = batch;
        }
        const int plain = n, total = plain + forms;
        std::vector<float> ms((size_t)total);
        const int pick = tune_candidates(M, A->N, total, fallback, stream, [&](int i, double *x, double *y) {
            if (i >= plain) return image_launch_candidate(image, i - plain, x, y, stream);
            if (ids[i] == 0) return stream_launch_csr(A, x, y, 0, nullptr, stream);
            return launch_rows(0, M, A->row_ptr, A->col_idx, A->values, x, y, ids[i], 0, stream);
        }, ms.data());
        int best = fallback;  // the plain choice stays for ALGO_ROW and the other entry points even when the image wins
        for (int i = 0; i < plain; ++i)
            if (ms[i] >= 0.0f && (ms[best] < 0.0f || ms[i] < ms[best])) best = i;
        if (ids[best] == 0) A->short_rows_stream = true;
        else A->row_batch = ids[best];
        // SPMV_B200_IMAGE_CANDIDATE=i >= 0 keeps image candidate i (image_candidates' order) instead of the fastest, and no
        // image when i >= forms: the timing picks a form per machine and run, so tests walk every form the plan offers
        const int forced_image = env_int("SPMV_B200_IMAGE_CANDIDATE", -1);
        const int keep = forced_image < 0 ? pick - plain : forced_image < forms ? forced_image : -1;
        if (keep >= 0) image_keep(image, keep);
        else image_free(image);
        A->image = image;
        // the fused iterated product (scale + |w|^2 partials in the tail): fused stream kernel (0) or fused row kernel
        if (A->num_long == 0) {
            double *partials = nullptr;
            const int count = std::max(std::max(A->stream_grid, fused_row_grid(A)), 1);
            if (cudaMalloc(&partials, (size_t)count * sizeof(double)) == cudaSuccess) {
                Epilogue ep;
                ep.partials = partials;
                ep.partials_total = count;
                A->fused_batch = tune_batch(M, A->N, 0, stream, [&](int batch, double *x, double *y) {
                    return launch_fused(A, x, y, ep, stream, batch);
                }, 0);
            }
            cudaGetLastError();
            cudaFree(partials);
            // the FLAT form (two-launch iterated product): its batch
            double *flat_partials = nullptr;
            if (cudaMalloc(&flat_partials, (size_t)flat_grid(M) * sizeof(double)) == cudaSuccess) {
                Epilogue fe;
                fe.partials = flat_partials;
                fe.partials_total = flat_grid(M);
                fe.inv_norm = flat_partials;  // any finite double will do for the timing
                const int n = (int)(sizeof kFlatCandidates / sizeof kFlatCandidates[0]);
                const int best = tune_candidates(M, A->N, n, 1, stream, [&](int i, double *x, double *y) {
                    return launch_fused_flat(A, x, y, fe, stream, kFlatCandidates[i]);
                });
                A->flat_batch = kFlatCandidates[best];
            }
            cudaGetLastError();
            cudaFree(flat_partials);
        }
    }
    return SPMV_B200_OK;
}

// elements of col_idx / values that 128/256-bit loads may touch: owned arrays are padded to a multiple of four
static int safe_vector_nnz(const spmv_b200_csr *A) {
    return (int)(A->owns ? ((A->nnz + 3) & ~3LL) : (A->nnz & ~3LL));
}

// lanes per row: about a quarter of the mean row length, so that every lane owns one full batch of kVecBatch gathers
static int pick_vector_width(long long nnz, int M) {
    const int forced = env_int("SPMV_B200_VECTOR_WIDTH", 0);
    if (forced == 1 || forced == 2 || forced == 4 || forced == 8 || forced == 16 || forced == 32) return forced;
    const double avg = M > 0 ? (double)nnz / M : 0.0;
    if (avg <= 8.0) return 1;
    if (avg <= 12.0) return 2;
    if (avg <= 24.0) return 4;
    if (avg <= 48.0) return 8;
    if (avg <= 96.0) return 16;
    return 32;
}

template <typename V>
static int launch_rows(int row_begin, int row_end, const int *row_ptr, const int *col_idx, const V *values,
                       const V *x, V *y, int batch, int accumulate, cudaStream_t stream) {
    const long long rows = (long long)row_end - row_begin;
    if (rows <= 0) return SPMV_B200_OK;
    const XPolicy keep = matrix_policy(row_ptr + row_begin, (size_t)(rows + 1) * sizeof(int));
    // batch >= 16: csr_rowm_kernel, form kRowmVariants[batch - 16].  SPMV_B200_ROW_MULTI=k (k >= 1) sends EVERY row-kernel
    // launch through form k - 1 (parity runs: tests/test_gpu_parity.py walks all forms, fp64 bit for bit)
    const int forced_multi = env_int("SPMV_B200_ROW_MULTI", 0);
    const int variant = forced_multi >= 1 ? std::min(forced_multi, kNumRowmVariants) - 1 : batch - 16;
    if (variant >= 0) {
        if (variant >= kNumRowmVariants) return fail(SPMV_B200_ERR_INVALID, "row kernel: unknown multi-row form %d", variant);
        const unsigned int gm = blocks_for(rows, 256 * kRowmVariants[variant].rows);
        int at = 0;
#define ROWM_CASE(R, B, C)                                                                                                    \
    if (at++ == variant)                                                                                                      \
        SPMV_TRY_CUDA(launch_x(csr_rowm_kernel<B, R, C, V>, gm, 256, 0, stream, keep, row_begin, row_end, row_ptr, col_idx, values, x, \
                               y, accumulate));
        SPMV_ROWM_VARIANTS(ROWM_CASE)
#undef ROWM_CASE
        SPMV_TRY_CUDA(cudaGetLastError());
        return SPMV_B200_OK;
    }
    const unsigned int g = blocks_for(rows, 256);
    SPMV_TRY_CUDA((with_batch<4, 1, 2, 3, 5, 6, 7, 8>(batch, [&](auto B) {
        return launch_x(csr_row_kernel<B, V>, g, 256, 0, stream, keep, row_begin, row_end, row_ptr, col_idx, values, x, y, accumulate);
    })));
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

template <typename V>
static int launch_vector(int row_begin, int row_end, const int *row_ptr, const int *col_idx, const V *values,
                         const V *x, V *y, int vec, int accumulate, cudaStream_t stream, size_t x_bytes = 0, int safe_nnz = -1) {
    const long long rows = (long long)row_end - row_begin;
    if (rows <= 0) return SPMV_B200_OK;
    if (vec == 1) return launch_rows(row_begin, row_end, row_ptr, col_idx, values, x, y, env_int("SPMV_B200_ROW_BATCH", 4), accumulate, stream);
    // aligned-group kernel (128/256-bit stream loads) for matrices with a plan.  SPMV_B200_VEC4: 0 = scalar kernel,
    // 1 = one group of four per lane and step (default), 2 = two groups in flight per lane.  Lanes per row = an eighth
    // of the mean row length, i.e. a lane walks two groups: measured on uniform 32/row (tools/r02_diag.py, 3 rounds):
    // 4 lanes x 1 group 1.24 ms, 8 x 1 1.27, 4 x 2 1.36, scalar 8 lanes x 4 1.21 cold / 1.37 sustained, HLL slice 1.23.
    const int vec4 = env_int("SPMV_B200_VEC4", kVec4Default);
    if (safe_nnz >= 0 && vec4 != 0 && vec >= 2) {
        const XPolicy policy4 = x_policy(x, x_bytes);
        const int groups = vec4 == 1 ? 1 : 2;
        const int lanes = env_int("SPMV_B200_VECTOR_WIDTH", 0) > 0 ? std::max(1, vec / groups) : std::max(2, vec / 2);
        const unsigned int grid4 = blocks_for(rows * lanes, 256);
#define VEC4_CASE(W, G)                                                                                                     \
    case W:                                                                                                                 \
        SPMV_TRY_CUDA(launch_x(csr_vector4_kernel<W, G, V>, grid4, 256, 0, stream, policy4, row_begin, row_end, row_ptr, col_idx, \
                               values, x, y, accumulate, safe_nnz));                                                        \
        break;
        if (groups == 1) {
            switch (lanes) {
                VEC4_CASE(1, 1) VEC4_CASE(2, 1) VEC4_CASE(4, 1) VEC4_CASE(8, 1) VEC4_CASE(16, 1) VEC4_CASE(32, 1)
                default: return fail(SPMV_B200_ERR_INVALID, "bad lane count %d", lanes);
            }
        } else {
            switch (lanes) {
                VEC4_CASE(1, 2) VEC4_CASE(2, 2) VEC4_CASE(4, 2) VEC4_CASE(8, 2) VEC4_CASE(16, 2)
                default: return fail(SPMV_B200_ERR_INVALID, "bad lane count %d", lanes);
            }
        }
#undef VEC4_CASE
        return SPMV_B200_OK;
    }
    const unsigned int grid = blocks_for(rows * vec, 256);
    // (8 lanes x 4 gathers per lane is the measured optimum on 32 nonzeros per row: 1208 us; 8 x 8: 1246, 4 x 8: 1415,
    //  16 x 4: 1369 -- profiles/r01d_kernel_selection.md)
    const XPolicy policy = x_policy(x, x_bytes);
#define VEC_CASE(W)                                                                                                 \
    case W:                                                                                                         \
        SPMV_TRY_CUDA(launch_x(csr_vector_kernel<W, V>, grid, 256, 0, stream, policy, row_begin, row_end, row_ptr, col_idx, \
                               values, x, y, accumulate));                                                          \
        break;
    switch (vec) {
        VEC_CASE(1) VEC_CASE(2) VEC_CASE(4) VEC_CASE(8) VEC_CASE(16) VEC_CASE(32)
        default:
            return fail(SPMV_B200_ERR_INVALID, "threads_per_row must be 0,1,2,4,8,16 or 32 (got %d)", vec);
    }
#undef VEC_CASE
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

// tiles [tile_begin, tile_end) of the plan; the long rows (if any) ride with the call that covers the last tile
static int launch_tiles(const spmv_b200_csr *A, const double *x, double *y, int accumulate, bool pipelined,
                        cudaStream_t stream, int tile_begin = 0, int tile_end = -1) {
    if (A->num_tiles == 0) return SPMV_B200_OK;
    if (tile_end < 0) tile_end = A->num_tiles;
    if (tile_end <= tile_begin) return SPMV_B200_OK;
    (void)pipelined;  // the first-generation tile kernel (products parked in shared memory, one CTA per tile) was retired in
                      // round 2: it lost to the stream kernel on every shape measured (lap2d 0.34 vs 0.24 ms, uniform 1.87 vs
                      // 1.31 ms vector, R-MAT 1.87 vs 1.60 ms binned); SPMV_B200_ALGO_TILE now runs the stream kernel
    SPMV_TRY(stream_launch_csr(A, x, y, accumulate, nullptr, stream, tile_begin, tile_end - tile_begin));
    if (A->num_long > 0 && tile_end == A->num_tiles) {
        csr_long_fragment_kernel<double><<<A->num_frag, kFragThreads, 0, stream>>>(A->long_rows, A->frag_first, A->num_long,
                                                                          A->row_ptr, A->col_idx, A->values, x,
                                                                          A->frag_partial);
        SPMV_TRY_CUDA(cudaGetLastError());
        csr_long_combine_kernel<double><<<blocks_for(A->num_long, 128), 128, 0, stream>>>(A->long_rows, A->frag_first,
                                                                                 A->num_long, A->frag_partial, y,
                                                                                 accumulate);
        SPMV_TRY_CUDA(cudaGetLastError());
    }
    return SPMV_B200_OK;
}

// Bin plan: stable sort of the row ids by bin (radix sort on 3-bit keys), bin offsets, fragments of the longest rows.
static int build_bins(spmv_b200_csr *A, cudaStream_t stream) {
    free_bins(A);
    const int M = A->M;
    BinPlan &B = A->bins;
    unsigned char *keys = nullptr, *keys_sorted = nullptr;
    int *ids = nullptr, *d_counts = nullptr, *frag_counts = nullptr;
    void *temp = nullptr;
    auto body = [&]() -> int {
        SPMV_TRY_CUDA(cudaMalloc(&keys, (size_t)M));
        SPMV_TRY_CUDA(cudaMalloc(&keys_sorted, (size_t)M));
        SPMV_TRY_CUDA(cudaMalloc(&ids, (size_t)M * sizeof(int)));
        SPMV_TRY_CUDA(cudaMalloc(&B.rows, (size_t)M * sizeof(int)));
        SPMV_TRY_CUDA(cudaMalloc(&d_counts, kBins * sizeof(int)));
        SPMV_TRY_CUDA(cudaMemsetAsync(d_counts, 0, kBins * sizeof(int), stream));
        bin_key_kernel<<<blocks_for(M, 256), 256, 0, stream>>>(M, A->row_ptr, keys, ids, d_counts);
        SPMV_TRY_CUDA(cudaGetLastError());
        size_t temp_bytes = 0;
        SPMV_TRY_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys, keys_sorted, ids, B.rows, M, 0, 3, stream));
        SPMV_TRY_CUDA(cudaMalloc(&temp, temp_bytes ? temp_bytes : 1));
        SPMV_TRY_CUDA(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, keys_sorted, ids, B.rows, M, 0, 3, stream));
        int counts[kBins];
        SPMV_TRY_CUDA(cudaMemcpyAsync(counts, d_counts, sizeof counts, cudaMemcpyDeviceToHost, stream));
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
        B.offset[0] = 0;
        for (int b = 0; b < kBins; ++b) B.offset[b + 1] = B.offset[b] + counts[b];
        long long blocks = 0;
        for (int b = 0; b < kBins - 1; ++b) {
            B.block_start[b] = (int)blocks;
            blocks += ((long long)counts[b] * (1 << b) + 255) / 256;
        }
        if (blocks > 0x7fffffffLL) return fail(SPMV_B200_ERR_INVALID, "bin plan: too many CTAs");
        B.block_start[kBins - 1] = (int)blocks;
        B.num_long = counts[kBins - 1];
        if (B.num_long > 0) {
            const int *long_rows = B.rows + B.offset[kBins - 1];
            SPMV_TRY_CUDA(cudaMalloc(&frag_counts, (size_t)(B.num_long + 1) * sizeof(int)));
            SPMV_TRY_CUDA(cudaMalloc(&B.frag_first, (size_t)(B.num_long + 1) * sizeof(int)));
            plan_fragcount_kernel<<<blocks_for(B.num_long + 1, 256), 256, 0, stream>>>(B.num_long, long_rows, A->row_ptr, frag_counts);
            SPMV_TRY_CUDA(cudaGetLastError());
            size_t scan_bytes = 0;
            SPMV_TRY_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, frag_counts, B.frag_first, B.num_long + 1, stream));
            if (scan_bytes > temp_bytes) {
                cudaFree(temp);
                temp = nullptr;
                SPMV_TRY_CUDA(cudaMalloc(&temp, scan_bytes));
                temp_bytes = scan_bytes;
            }
            SPMV_TRY_CUDA(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, frag_counts, B.frag_first, B.num_long + 1, stream));
            SPMV_TRY_CUDA(cudaMemcpyAsync(&B.num_frag, B.frag_first + B.num_long, sizeof(int), cudaMemcpyDeviceToHost, stream));
            SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
            SPMV_TRY_CUDA(cudaMalloc(&B.frag_partial, (size_t)std::max(B.num_frag, 1) * sizeof(double)));
        }
        B.built = true;
        return SPMV_B200_OK;
    };
    const int rc = body();
    cudaFree(keys);
    cudaFree(keys_sorted);
    cudaFree(ids);
    cudaFree(d_counts);
    cudaFree(frag_counts);
    cudaFree(temp);
    if (rc != SPMV_B200_OK) free_bins(A);
    return rc;
}

template <typename V>
static int launch_binned(const spmv_b200_csr *A, const V *values, const V *x, V *y, int accumulate, cudaStream_t stream) {
    if (A->M == 0) return SPMV_B200_OK;
    if (!A->bins.built) SPMV_TRY(build_bins(const_cast<spmv_b200_csr *>(A), stream));  // lazily, once per plan
    const BinPlan &B = A->bins;
    BinLaunch L;
    for (int b = 0; b <= kBins; ++b) L.offset[b] = B.offset[b];
    for (int b = 0; b < kBins; ++b) L.block_start[b] = B.block_start[b];
    // the fragments of the longest rows ride in the same launch, as its first CTAs (round 1 ran them as a second
    // launch behind the binned one: 0.29 ms serialised on R-MAT scale 24)
    // SPMV_B200_BINNED_SPLIT=1: the fragments as a launch of their own behind the binned one (round-1 shape, kept for A/B)
    const bool split = env_int("SPMV_B200_BINNED_SPLIT", 0) != 0;
    L.frag_blocks = (B.num_long > 0 && !split) ? B.num_frag : 0;
    L.safe_nnz = env_int("SPMV_B200_VEC4", kVec4Default) != 0 ? safe_vector_nnz(A) : -1;
    L.num_long = B.num_long;
    L.frag_first = B.frag_first;
    L.frag_partial = B.frag_partial;
    const long long blocks = (long long)B.block_start[kBins - 1] + L.frag_blocks;
    if (blocks > 0x7fffffffLL) return fail(SPMV_B200_ERR_INVALID, "bin plan: too many CTAs");
    if (blocks > 0) {
        SPMV_TRY_CUDA(launch_x(csr_binned_kernel<V>, (unsigned int)blocks, 256, 0, stream, x_policy(x, (size_t)A->N * sizeof(V)),
                               L, B.rows, A->row_ptr, A->col_idx, values, x, y, accumulate));
    }
    if (B.num_long > 0 && split) {
        csr_long_fragment_kernel<V><<<B.num_frag, kFragThreads, 0, stream>>>(B.rows + B.offset[kBins - 1], B.frag_first, B.num_long,
                                                                            A->row_ptr, A->col_idx, values, x, B.frag_partial);
        SPMV_TRY_CUDA(cudaGetLastError());
    }
    if (B.num_long > 0) {
        const int *long_rows = B.rows + B.offset[kBins - 1];
        csr_long_combine_kernel<V><<<blocks_for(B.num_long, 128), 128, 0, stream>>>(long_rows, B.frag_first, B.num_long,
                                                                                   B.frag_partial, y, accumulate);
        SPMV_TRY_CUDA(cudaGetLastError());
    }
    return SPMV_B200_OK;
}

// Which kernel a request resolves to.  AUTO: short rows (stencils) -> the TMA stream kernel, which runs at the HBM
// roofline; longer rows mean many gathers of x per streamed byte, bounded by the L1TEX/L2 sector rate and by
// the latency of gathers that miss L2 -- those need the occupancy of the direct-load kernels: vector-per-row when no
// row is long, the row-binned tile kernel (+ long-row split) when the lengths are skewed
// (profiles/r01c_ncu_full_summary.md).  threads_per_row == 1 is a request for the reference's summation order,
// which the stream kernel honours.
CsrPath csr_resolve(const spmv_b200_csr *A, int algo) {
    switch (algo) {
        case SPMV_B200_ALGO_STREAM: return kPathStream;
        case SPMV_B200_ALGO_TILE: return kPathTile;
        case SPMV_B200_ALGO_VECTOR: return kPathVector;
        case SPMV_B200_ALGO_BINNED: return kPathBinned;
        case SPMV_B200_ALGO_ROW: return kPathRow;
        case SPMV_B200_ALGO_ROW_IMAGE: return kPathImage;
        default:
            // every row short: one thread per row (serial order, so forced_tpr == 1 is honoured as well) -- on the
            // private image when the handle holds one
            if (A->max_row <= kRowKernelMaxLen) return A->image ? kPathImage : A->short_rows_stream ? kPathStream : kPathRow;
            if (A->forced_tpr == 1 || A->nnz <= (long long)kAutoStreamMaxAvg * A->M) return kPathStream;
            {   // longer rows: one lane count for all rows (vector kernel) only while the lengths are even; a longest row
                // far above the mean (or above the long-row threshold) means skew -> lanes per row by length class
                const long long mean = A->M > 0 ? (A->nnz + A->M - 1) / A->M : 0;
                const bool skewed = A->num_long > 0 || A->max_row > 4 * std::max<long long>(mean, 8);
                return skewed ? kPathBinned : kPathVector;
            }
    }
}

int csr_launch_window(const spmv_b200_csr *A, CsrPath path, int unit_begin, int unit_end, const double *x, double *y,
                      int accumulate, cudaStream_t stream) {
    if (path == kPathBinned) return launch_binned<double>(A, A->values, x, y, accumulate, stream);  // whole matrix: rows are permuted
    if (path == kPathRow)
        return launch_rows(unit_begin, unit_end, A->row_ptr, A->col_idx, A->values, x, y, A->row_batch, accumulate, stream);
    if (path == kPathImage) return image_launch(A->image, unit_begin, unit_end, x, y, accumulate, stream);
    if (path == kPathVector)
        return launch_vector(unit_begin, unit_end, A->row_ptr, A->col_idx, A->values, x, y, pick_vector_width(A->nnz, A->M),
                             accumulate, stream, (size_t)A->N * sizeof(double), safe_vector_nnz(A));
    return launch_tiles(A, x, y, accumulate, path == kPathStream, stream, unit_begin, unit_end);
}

// grid of the fused row kernel: a fixed number of CTAs of 256 threads per SM (8 are resident), whatever the matrix size
int fused_ctas_per_sm() { return std::max(1, std::min(env_int("SPMV_B200_FUSED_CTAS_PER_SM", kFusedCtasPerSm), 256)); }

static int fused_row_grid(const spmv_b200_csr *A) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (int)std::max<long long>(1, std::min<long long>((long long)fused_ctas_per_sm() * sms, ((long long)A->M + 255) / 256));
}

static int launch_fused(const spmv_b200_csr *A, const double *x, double *y, const Epilogue &ep, cudaStream_t stream,
                        int batch) {
    if (batch < 0) batch = env_int("SPMV_B200_FUSED_BATCH", A->fused_batch);
    if (batch == 0) return stream_launch_csr(A, x, y, 0, &ep, stream);
    const int g = fused_row_grid(A);
    with_batch<4, 2, 3, 5, 6, 7>(batch, [&](auto B) {
        csr_row_fused_kernel<B><<<g, 256, 0, stream>>>(A->M, A->row_ptr, A->col_idx, A->values, x, y, ep);
    });
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

// ---- the FLAT form (two-launch iterated product): one CTA per 256 rows; the batch is timed at plan time ----
static int flat_grid(long long M) { return (int)std::max<long long>(1, (M + 255) / 256); }

static int launch_fused_flat(const spmv_b200_csr *A, const double *x, double *y, const Epilogue &ep, cudaStream_t stream,
                             int batch) {
    const int g = flat_grid(A->M);
    const XPolicy keep = matrix_policy(A->row_ptr, (size_t)(A->M + 1) * sizeof(int));
    SPMV_TRY_CUDA((with_batch<4, 2, 3, 5, 6, 7>(batch, [&](auto B) {
        return launch_x(csr_row_flat_kernel<B>, g, 256, 0, stream, keep, A->M, A->row_ptr, A->col_idx, A->values, x, y, ep);
    })));
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int check_peers(const spmv_b200_peers_t *peers, int M, const char *what) {
    if (!peers) return SPMV_B200_OK;
    if (peers->count < 0 || peers->count > SPMV_B200_MAX_PEERS) return fail(SPMV_B200_ERR_INVALID, "%s: bad peer count %d", what, peers->count);
    for (int p = 0; p < peers->count; ++p)
        if (peers->lo[p] < 0 || peers->hi[p] > M || peers->lo[p] > peers->hi[p])
            return fail(SPMV_B200_ERR_INVALID, "%s: peer %d: bad row range [%d,%d) of %d rows", what, p, peers->lo[p], peers->hi[p], M);
    return SPMV_B200_OK;
}

int boundary_first_order(const spmv_b200_peers_t &peers, int M, ChunkOrder &order) {
    order = ChunkOrder();
    SPMV_TRY(check_peers(&peers, M, "fused product"));
    std::vector<std::pair<int, int>> iv;
    for (int p = 0; p < peers.count; ++p)
        if (peers.hi[p] > peers.lo[p]) iv.emplace_back(peers.lo[p] >> 8, (peers.hi[p] + 255) >> 8);
    std::sort(iv.begin(), iv.end());
    for (const auto &r : iv) {
        if (order.count > 0 && r.first <= order.hi[order.count - 1]) {
            order.hi[order.count - 1] = std::max(order.hi[order.count - 1], r.second);
        } else {
            order.lo[order.count] = r.first;
            order.hi[order.count] = r.second;
            ++order.count;
        }
    }
    for (int i = 0; i < order.count; ++i) order.boundary_chunks += order.hi[i] - order.lo[i];
    return SPMV_B200_OK;
}

// Per-launch access-policy windows (handles.cuh).  The device-wide persisting carve-out is raised once per device.
static bool persisting_limits(size_t &carve_out, size_t &max_window_out) {
    static int ready[64];
    static size_t carve[64], max_window[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return false;
    if (!ready[dev]) {
        int max_persist = 0, max_win = 0;
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
        cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, dev);
        size_t want = (size_t)std::max(max_persist, 0);
        const int mb = env_int("SPMV_B200_L2_PERSIST_MB", 0);
        if (mb > 0) want = std::min(want, (size_t)mb << 20);
        size_t got = 0;
        if (want > 0 && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess)
            cudaDeviceGetLimit(&got, cudaLimitPersistingL2CacheSize);
        carve[dev] = got;
        max_window[dev] = (size_t)std::max(max_win, 0);
        ready[dev] = 1;
        cudaGetLastError();
    }
    carve_out = carve[dev];
    max_window_out = max_window[dev];
    return carve[dev] > 0 && max_window[dev] > 0;
}

XPolicy x_policy(const void *x, size_t bytes) {
    XPolicy p;
    if (!x || bytes == 0 || env_int("SPMV_B200_L2_PERSIST", kL2PersistDefault) == 0) return p;
    size_t carve = 0, max_window = 0;
    if (!persisting_limits(carve, max_window)) return p;
    const size_t window = std::min(bytes, max_window);
    float ratio = window <= carve ? 1.0f : (float)((double)carve / (double)window);
    const int pct = env_int("SPMV_B200_L2_HIT_PCT", 0);
    if (pct > 0 && pct <= 100) ratio = std::min(ratio, pct / 100.0f);
    cudaAccessPolicyWindow w = {};
    w.base_ptr = const_cast<void *>(x);
    w.num_bytes = window;
    w.hitRatio = ratio;
    w.hitProp = cudaAccessPropertyPersisting;
    w.missProp = env_int("SPMV_B200_L2_MISS_NORMAL", 0) ? cudaAccessPropertyNormal : cudaAccessPropertyStreaming;
    p.attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
    p.attr[0].val.accessPolicyWindow = w;
    p.count = 1;
    return p;
}

// The head of a matrix array (row_ptr of the thread-per-row CSR kernels; JA of the HLL row kernels) kept in the persisting
// carve-out ACROSS products: an iterated product re-reads the whole matrix every launch, and whatever part of it the L2
// holds on to is DRAM traffic saved on every launch after the first (64 MiB of 1.34 GB on lap2d 4096^2).  The window is
// clamped to the carve-out (hitRatio 1: no thrashing among the persisting lines); everything outside it is untouched.
XPolicy matrix_policy(const void *head, size_t bytes) {
    XPolicy p;
    if (!head || bytes == 0 || env_int("SPMV_B200_MATRIX_PERSIST", kMatrixPersistDefault) == 0) return p;
    size_t carve = 0, max_window = 0;
    if (!persisting_limits(carve, max_window)) return p;
    const int pct = env_int("SPMV_B200_MATRIX_PERSIST_PCT", 100);
    const size_t budget = (size_t)((double)carve * std::min(std::max(pct, 1), 100) / 100.0);
    cudaAccessPolicyWindow w = {};
    w.base_ptr = const_cast<void *>(head);
    w.num_bytes = std::min(std::min(bytes, max_window), budget);
    w.hitRatio = 1.0f;
    w.hitProp = cudaAccessPropertyPersisting;
    w.missProp = cudaAccessPropertyNormal;
    p.attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
    p.attr[0].val.accessPolicyWindow = w;
    p.count = 1;
    return p;
}

static int check_device() {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(SPMV_B200_ERR_NO_DEVICE, "no usable CUDA device (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    return SPMV_B200_OK;
}

}  // namespace spmv

// ================================================================================================
// C-ABI
// ================================================================================================
using namespace spmv;

extern "C" {

int spmv_b200_csr_upload(int M, int N, long long nnz, const int *row_ptr, const int *col_idx, const double *values,
                         spmv_b200_csr **out) {
    if (!out) return fail(SPMV_B200_ERR_INVALID, "csr_upload: out is NULL");
    *out = nullptr;
    if (M < 0 || N < 0 || nnz < 0 || nnz > 0x7fffffffLL || !row_ptr || (nnz > 0 && (!col_idx || !values)))
        return fail(SPMV_B200_ERR_INVALID, "csr_upload: bad arguments (M=%d N=%d nnz=%lld)", M, N, nnz);
    SPMV_TRY(check_device());
    spmv_b200_csr *A = new (std::nothrow) spmv_b200_csr();
    if (!A) return fail(SPMV_B200_ERR_NOMEM, "csr_upload: out of host memory");
    A->M = M;
    A->N = N;
    A->nnz = nnz;
    A->owns = true;
    int rc = SPMV_B200_OK;
    auto bail = [&](cudaError_t e, const char *what) {
        rc = fail(e == cudaErrorMemoryAllocation ? SPMV_B200_ERR_NOMEM : SPMV_B200_ERR_CUDA, "csr_upload: %s: %s", what,
                  cudaGetErrorString(e));
        spmv_b200_csr_free(A);
        return rc;
    };
    cudaError_t e;
    // pad the element arrays to a multiple of 4 so that aligned vector loads near the end stay in bounds
    const size_t padded = ((size_t)nnz + 3) & ~(size_t)3;
    if ((e = cudaMalloc(&A->row_ptr, ((size_t)M + 1) * sizeof(int))) != cudaSuccess) return bail(e, "cudaMalloc row_ptr");
    if ((e = cudaMalloc(&A->col_idx, std::max<size_t>(padded, 4) * sizeof(int))) != cudaSuccess) return bail(e, "cudaMalloc col_idx");
    if ((e = cudaMalloc(&A->values, std::max<size_t>(padded, 4) * sizeof(double))) != cudaSuccess) return bail(e, "cudaMalloc values");
    if ((e = cudaMemcpy(A->row_ptr, row_ptr, ((size_t)M + 1) * sizeof(int), cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "H2D row_ptr");
    if (nnz > 0) {
        if ((e = cudaMemcpy(A->col_idx, col_idx, (size_t)nnz * sizeof(int), cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "H2D col_idx");
        if ((e = cudaMemcpy(A->values, values, (size_t)nnz * sizeof(double), cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "H2D values");
    }
    rc = build_plan(A, nullptr);
    if (rc != SPMV_B200_OK) {
        spmv_b200_csr_free(A);
        return rc;
    }
    *out = A;
    return SPMV_B200_OK;
}

}  // extern "C"

// a handle over device arrays; owns: freed with the handle, and eligible for the private image (the caller of
// wrap_device may rewrite its arrays, which would leave an image stale)
static int csr_from_device(int M, int N, long long nnz, const int *d_row_ptr, const int *d_col_idx, const double *d_values,
                           bool owns, void *stream, spmv_b200_csr **out) {
    if (!out) return fail(SPMV_B200_ERR_INVALID, "csr_wrap_device: out is NULL");
    *out = nullptr;
    if (M < 0 || N < 0 || nnz < 0 || nnz > 0x7fffffffLL || !d_row_ptr || (nnz > 0 && (!d_col_idx || !d_values)))
        return fail(SPMV_B200_ERR_INVALID, "csr_wrap_device: bad arguments (M=%d N=%d nnz=%lld)", M, N, nnz);
    if ((reinterpret_cast<uintptr_t>(d_col_idx) & 15) || (reinterpret_cast<uintptr_t>(d_values) & 31) ||
        (reinterpret_cast<uintptr_t>(d_row_ptr) & 15))
        return fail(SPMV_B200_ERR_INVALID, "csr_wrap_device: row_ptr / col_idx must be 16-byte and values 32-byte "
                                           "aligned (cudaMalloc'ed arrays are)");
    SPMV_TRY(check_device());
    spmv_b200_csr *A = new (std::nothrow) spmv_b200_csr();
    if (!A) return fail(SPMV_B200_ERR_NOMEM, "csr_wrap_device: out of host memory");
    A->M = M;
    A->N = N;
    A->nnz = nnz;
    A->row_ptr = const_cast<int *>(d_row_ptr);
    A->col_idx = const_cast<int *>(d_col_idx);
    A->values = const_cast<double *>(d_values);
    A->owns = owns;
    int rc = build_plan(A, as_stream(stream));
    if (rc != SPMV_B200_OK) {
        A->owns = false;  // on failure the arrays stay the caller's
        spmv_b200_csr_free(A);
        return rc;
    }
    *out = A;
    return SPMV_B200_OK;
}

extern "C" {

int spmv_b200_csr_wrap_device(int M, int N, long long nnz, const int *d_row_ptr, const int *d_col_idx,
                              const double *d_values, void *stream, spmv_b200_csr **out) {
    return csr_from_device(M, N, nnz, d_row_ptr, d_col_idx, d_values, false, stream, out);
}

// used by synth.cu and convert.cu: adopt freshly generated device arrays
int spmv_b200_csr_adopt_device_(int M, int N, long long nnz, int *d_row_ptr, int *d_col_idx, double *d_values,
                                void *stream, spmv_b200_csr **out) {
    return csr_from_device(M, N, nnz, d_row_ptr, d_col_idx, d_values, true, stream, out);
}

int spmv_b200_csr_replan(spmv_b200_csr *A, int tile_items, int long_threshold, int threads_per_row, void *stream) {
    if (!A) return fail(SPMV_B200_ERR_INVALID, "csr_replan: NULL matrix");
    if (threads_per_row < 0 || threads_per_row > 32 || (threads_per_row & (threads_per_row - 1)))
        return fail(SPMV_B200_ERR_INVALID, "csr_replan: threads_per_row must be 0 or a power of two <= 32");
    if (tile_items < 0 || long_threshold < 0) return fail(SPMV_B200_ERR_INVALID, "csr_replan: negative parameter");
    if (tile_items > 0) A->tile_items = std::max(tile_items, 96);
    if (long_threshold > 0) A->long_threshold = long_threshold;
    A->forced_tpr = threads_per_row;
    return build_plan(A, as_stream(stream));
}

int spmv_b200_csr_info(const spmv_b200_csr *A, spmv_b200_csr_info_t *info) {
    if (!A || !info) return fail(SPMV_B200_ERR_INVALID, "csr_info: NULL argument");
    info->M = A->M;
    info->N = A->N;
    info->nnz = A->nnz;
    info->num_tiles = A->num_tiles;
    info->num_long_rows = A->num_long;
    info->num_fragments = A->num_frag;
    info->threads_per_row = A->forced_tpr;
    info->tile_items = A->tile_items;
    info->long_threshold = A->long_threshold;
    info->algorithmic_bytes = A->nnz * 12 + 4LL * ((long long)A->M + 1) + 8LL * A->M + 8LL * A->N;
    info->max_row_nnz = A->max_row;
    switch (csr_resolve(A, SPMV_B200_ALGO_AUTO)) {
        case kPathRow: info->auto_algo = SPMV_B200_ALGO_ROW; break;
        case kPathImage: info->auto_algo = SPMV_B200_ALGO_ROW_IMAGE; break;
        case kPathStream: info->auto_algo = SPMV_B200_ALGO_STREAM; break;
        case kPathVector: info->auto_algo = SPMV_B200_ALGO_VECTOR; break;
        case kPathBinned: info->auto_algo = SPMV_B200_ALGO_BINNED; break;
        default: info->auto_algo = SPMV_B200_ALGO_TILE; break;
    }
    info->row_batch = A->row_batch;
    info->fused_batch = A->fused_batch;
    info->flat_batch = A->flat_batch;
    info->flat_chunks = 1;
    image_info(A->image, info);
    return SPMV_B200_OK;
}

int spmv_b200_csr_device_arrays(const spmv_b200_csr *A, const int **d_row_ptr, const int **d_col_idx,
                                const double **d_values) {
    if (!A) return fail(SPMV_B200_ERR_INVALID, "csr_device_arrays: NULL matrix");
    if (d_row_ptr) *d_row_ptr = A->row_ptr;
    if (d_col_idx) *d_col_idx = A->col_idx;
    if (d_values) *d_values = A->values;
    return SPMV_B200_OK;
}

int spmv_b200_csr_download(const spmv_b200_csr *A, int *row_ptr, int *col_idx, double *values) {
    if (!A) return fail(SPMV_B200_ERR_INVALID, "csr_download: NULL matrix");
    if (row_ptr) SPMV_TRY_CUDA(cudaMemcpy(row_ptr, A->row_ptr, ((size_t)A->M + 1) * sizeof(int), cudaMemcpyDeviceToHost));
    if (col_idx && A->nnz) SPMV_TRY_CUDA(cudaMemcpy(col_idx, A->col_idx, (size_t)A->nnz * sizeof(int), cudaMemcpyDeviceToHost));
    if (values && A->nnz) SPMV_TRY_CUDA(cudaMemcpy(values, A->values, (size_t)A->nnz * sizeof(double), cudaMemcpyDeviceToHost));
    return SPMV_B200_OK;
}

int spmv_b200_csr_spmv(const spmv_b200_csr *A, const double *d_x, double *d_y, int accumulate, int algo, void *stream) {
    if (!A || !d_y || (A->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "csr_spmv: NULL argument");
    if (A->M == 0) return SPMV_B200_OK;
    if (algo < SPMV_B200_ALGO_AUTO || algo > SPMV_B200_ALGO_ROW_IMAGE) return fail(SPMV_B200_ERR_INVALID, "csr_spmv: unknown algo %d", algo);
    if (algo == SPMV_B200_ALGO_ROW_IMAGE && !A->image)
        return fail(SPMV_B200_ERR_INVALID, "csr_spmv: the matrix holds no image (spmv_b200_csr_set_image)");
    const CsrPath path = csr_resolve(A, algo);
    const bool by_rows = path == kPathVector || path == kPathRow || path == kPathImage;
    return csr_launch_window(A, path, 0, by_rows ? A->M : A->num_tiles, d_x, d_y, accumulate, as_stream(stream));
}

int spmv_b200_csr_partials_count(const spmv_b200_csr *A) {
    if (!A) return 0;
    return std::max(std::max(A->stream_grid, fused_row_grid(A)), 1);
}

int spmv_b200_csr_spmv_fused(const spmv_b200_csr *A, const double *d_x, double *d_y, const double *d_prev_sumsq,
                             double *d_partials, const spmv_b200_peers_t *peers, void *stream) {
    if (!A || !d_y || (A->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused: NULL argument");
    if (A->num_long > 0)
        return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused: %d rows exceed the long-row threshold; use csr_spmv", A->num_long);
    SPMV_TRY(check_peers(peers, A->M, "csr_spmv_fused"));
    Epilogue ep;
    ep.prev_sumsq = d_prev_sumsq;
    ep.partials = d_partials;
    ep.partials_total = spmv_b200_csr_partials_count(A);
    if (peers) ep.peers = *peers;
    if (A->M == 0) return SPMV_B200_OK;
    if (peers && env_int("SPMV_B200_FUSED_BOUNDARY_FIRST", 0)) SPMV_TRY(boundary_first_order(ep.peers, A->M, ep.order));
    return launch_fused(A, d_x, d_y, ep, as_stream(stream), -1);
}

int spmv_b200_csr_flat_partials_count(const spmv_b200_csr *A) {
    if (!A) return 0;
    return flat_grid(A->M);
}

int spmv_b200_csr_spmv_fused_flat(const spmv_b200_csr *A, const double *d_x, double *d_y, const double *d_inv_norm,
                                  double *d_partials, const spmv_b200_peers_t *peers, void *stream) {
    if (!A || !d_y || (A->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_flat: NULL argument");
    if (A->max_row > kRowKernelMaxLen)
        return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_flat: rows of up to %d nonzeros only (longest row: %d)", kRowKernelMaxLen, A->max_row);
    SPMV_TRY(check_peers(peers, A->M, "csr_spmv_fused_flat"));
    if (A->M == 0) return SPMV_B200_OK;
    Epilogue ep;
    ep.inv_norm = d_inv_norm;
    ep.partials = d_partials;
    ep.partials_total = flat_grid(A->M);
    if (peers) ep.peers = *peers;
    return launch_fused_flat(A, d_x, d_y, ep, as_stream(stream), env_int("SPMV_B200_FLAT_BATCH", A->flat_batch));
}

int spmv_b200_csr_spmv_fused_mail(const spmv_b200_csr *A, const double *d_x, double *d_y, double *d_partials,
                                  const spmv_b200_peers_t *peers, const spmv_b200_mail_t *mail, void *stream) {
    if (!A || !d_y || !d_partials || !mail || (A->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_mail: NULL argument");
    if (A->num_long > 0)
        return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_mail: %d rows exceed the long-row threshold; use csr_spmv", A->num_long);
    if (A->M == 0 || A->num_tiles == 0) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_mail: a rank without rows cannot take part in the exchange");
    SPMV_TRY(check_peers(peers, A->M, "csr_spmv_fused_mail"));
    if (mail->world < 1 || mail->world > SPMV_B200_MAX_RANKS || mail->rank < 0 || mail->rank >= mail->world || !mail->counter ||
        !mail->status)
        return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_mail: bad mailbox description (world %d, rank %d)", mail->world, mail->rank);
    for (int r = 0; r < mail->world; ++r)
        if (!mail->box[r]) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_mail: mailbox of rank %d is NULL", r);
    Epilogue ep;
    ep.partials = d_partials;
    ep.partials_total = spmv_b200_csr_partials_count(A);
    if (peers) ep.peers = *peers;
    ep.mail = *mail;
    if (peers && env_int("SPMV_B200_FUSED_BOUNDARY_FIRST", 0)) SPMV_TRY(boundary_first_order(ep.peers, A->M, ep.order));
    return launch_fused(A, d_x, d_y, ep, as_stream(stream), -1);
}

int spmv_b200_csr_spmv_fused_async(const spmv_b200_csr *A, const double *d_x, double *d_y, double *d_partials,
                                   const spmv_b200_peers_t *peers, const spmv_b200_async_t *as, void *stream) {
    if (!A || !d_y || !d_partials || !as || (A->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_async: NULL argument");
    if (A->max_row > kRowKernelMaxLen) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_async: rows of up to %d nonzeros only (longest row: %d)", kRowKernelMaxLen, A->max_row);
    if (A->M == 0) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_async: a rank without rows cannot take part in the exchange");
    if (as->world < 1 || as->world > SPMV_B200_MAX_RANKS || as->rank < 0 || as->rank >= as->world || !as->counter || !as->bcounter ||
        !as->status || as->num_recv < 0 || as->num_recv > SPMV_B200_MAX_PEERS)
        return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_async: bad exchange description (world %d, rank %d)", as->world, as->rank);
    for (int r = 0; r < as->world; ++r)
        if (!as->box[r]) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_async: mailbox of rank %d is NULL", r);
    for (int i = 0; i < as->num_recv; ++i)  // a halo tag is read at box[rank] + 8 world + recv_from[i]
        if (as->recv_from[i] < 0 || as->recv_from[i] >= as->world)
            return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_async: sender %d: bad rank %d", i, as->recv_from[i]);
    SPMV_TRY(check_peers(peers, A->M, "csr_spmv_fused_async"));
    spmv_b200_peers_t ps;
    ps.count = 0;
    if (peers) ps = *peers;
    ChunkOrder order;
    for (int p = 0; p < ps.count; ++p)
        if (as->send_to[p] < 0 || as->send_to[p] >= as->world) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_fused_async: peer %d: bad rank", p);
    SPMV_TRY(boundary_first_order(ps, A->M, order));
    if (env_int("SPMV_B200_ASYNC_NO_REORDER", 0)) {  // experiment: rows in their natural order, halo tags at the end
        order.count = 0;
        order.boundary_chunks = 0;
    }
    const int g = fused_row_grid(A);
    cudaStream_t st = as_stream(stream);
    AsyncArgs args;
    args.peers = ps;
    args.as = *as;
    args.order = order;
    with_batch<4, 2, 3, 5, 6, 7>(A->fused_batch > 0 ? A->fused_batch : A->row_batch, [&](auto B) {
        csr_row_async_kernel<B><<<g, 256, 0, st>>>(A->M, A->row_ptr, A->col_idx, A->values, d_x, d_y, d_partials, args);
    });
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int spmv_b200_csr_remap_columns(spmv_b200_csr *A, int nparts, const long long *starts, long long stride, void *stream) {
    if (!A || !starts) return fail(SPMV_B200_ERR_INVALID, "csr_remap_columns: NULL argument");
    if (!A->owns) return fail(SPMV_B200_ERR_INVALID, "csr_remap_columns: the matrix wraps arrays it does not own");
    if (nparts < 1 || nparts > SPMV_B200_MAX_RANKS || stride < 1 || (long long)nparts * stride > 0x7fffffffLL)
        return fail(SPMV_B200_ERR_INVALID, "csr_remap_columns: bad layout (%d parts, stride %lld)", nparts, stride);
    RemapTable t;
    t.nparts = nparts;
    t.stride = stride;
    for (int p = 0; p <= nparts; ++p) {
        t.starts[p] = starts[p];
        if (p > 0 && (starts[p] < starts[p - 1] || starts[p] - starts[p - 1] > stride))
            return fail(SPMV_B200_ERR_INVALID, "csr_remap_columns: part %d does not fit the stride", p - 1);
    }
    if (starts[0] != 0 || starts[nparts] != A->N) return fail(SPMV_B200_ERR_INVALID, "csr_remap_columns: the parts must cover [0, N)");
    if (A->nnz > 0) {
        remap_columns_kernel<<<blocks_for(A->nnz, 256), 256, 0, as_stream(stream)>>>(A->nnz, A->col_idx, t);
        SPMV_TRY_CUDA(cudaGetLastError());
    }
    A->N = (int)(nparts * stride);  // plans, tiles and the fp32 copy of the values do not depend on the column ids;
    image_free(A->image);           // the private image does, and so do the pieces of X the multi-vector host
    host_pipe_free(A->spmm_pipe);   // product uploads
    A->spmm_pipe = nullptr;
    SPMV_TRY_CUDA(cudaStreamSynchronize(as_stream(stream)));
    return SPMV_B200_OK;
}

int spmv_b200_csr_set_image(spmv_b200_csr *A, int mode, void *stream) {
    if (!A) return fail(SPMV_B200_ERR_INVALID, "csr_set_image: NULL matrix");
    if (mode < 0 || mode > 3) return fail(SPMV_B200_ERR_INVALID, "csr_set_image: unknown mode %d", mode);
    if (mode == 0) {
        image_free(A->image);
        return SPMV_B200_OK;
    }
    return image_build(A, mode, as_stream(stream));
}

int spmv_b200_csr_interior_rows(const spmv_b200_csr *A, long long col_lo, long long col_hi, int *row_lo, int *row_hi,
                                void *stream) {
    if (!A || !row_lo || !row_hi) return fail(SPMV_B200_ERR_INVALID, "csr_interior_rows: NULL argument");
    *row_lo = 0;
    *row_hi = A->M;
    if (A->M == 0) return SPMV_B200_OK;
    int *d_out = nullptr, out[2] = {0, A->M};
    SPMV_TRY_CUDA(cudaMalloc(&d_out, sizeof out));
    cudaError_t e = cudaMemcpyAsync(d_out, out, sizeof out, cudaMemcpyHostToDevice, as_stream(stream));
    if (e == cudaSuccess) {
        interior_rows_kernel<<<blocks_for(A->M, 256), 256, 0, as_stream(stream)>>>(A->M, A->M / 2, A->row_ptr, A->col_idx, col_lo,
                                                                                 col_hi, d_out);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, sizeof out, cudaMemcpyDeviceToHost, as_stream(stream));
    if (e == cudaSuccess) e = cudaStreamSynchronize(as_stream(stream));
    cudaFree(d_out);
    SPMV_TRY_CUDA(e);
    *row_lo = out[0];
    *row_hi = std::max(out[0], out[1]);
    return SPMV_B200_OK;
}

int spmv_b200_mail_exchange(double *d_partials, int count, const spmv_b200_mail_t *mail, double *d_sumsq_out, void *stream) {
    if (!d_partials || count < 1 || !mail || !d_sumsq_out) return fail(SPMV_B200_ERR_INVALID, "mail_exchange: bad arguments");
    if (mail->world < 1 || mail->world > SPMV_B200_MAX_RANKS || mail->rank < 0 || mail->rank >= mail->world || !mail->status)
        return fail(SPMV_B200_ERR_INVALID, "mail_exchange: bad mailbox description (world %d, rank %d)", mail->world, mail->rank);
    for (int r = 0; r < mail->world; ++r)
        if (!mail->box[r]) return fail(SPMV_B200_ERR_INVALID, "mail_exchange: mailbox of rank %d is NULL", r);
    // one CTA up to 8192 partials; beyond that up to 64 CTAs of at least 4096 (the last one to finish does the exchange)
    int ctas = (count <= 8192 || !mail->counter) ? 1 : std::min(64, (count + 4095) / 4096);
    ctas = std::max(1, std::min(ctas, env_int("SPMV_B200_EXCHANGE_CTAS", ctas)));
    const int chunk = (((count + ctas - 1) / ctas) + 3) & ~3;
    ctas = (count + chunk - 1) / chunk;
    mail_exchange_kernel<<<ctas, 1024, 0, as_stream(stream)>>>(d_partials, count, chunk, *mail, d_sumsq_out);
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int spmv_b200_csr_spmv_rows(const spmv_b200_csr *A, int row_begin, int row_end, const double *d_x, double *d_y,
                            void *stream) {
    if (!A || !d_y || !d_x) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_rows: NULL argument");
    if (row_begin < 0 || row_end > A->M || row_begin > row_end)
        return fail(SPMV_B200_ERR_INVALID, "csr_spmv_rows: range [%d,%d) outside [0,%d)", row_begin, row_end, A->M);
    if (A->image && image_any_rows(A->image))  // the private image where it takes any row range: the same bits
        return image_launch(A->image, row_begin, row_end, d_x, d_y, 0, as_stream(stream));
    if (A->max_row <= kRowKernelMaxLen)  // stencils: the thread-per-row kernel with the batch tuned at plan time (serial order)
        return launch_rows(row_begin, row_end, A->row_ptr, A->col_idx, A->values, d_x, d_y, A->row_batch, 0, as_stream(stream));
    return launch_vector(row_begin, row_end, A->row_ptr, A->col_idx, A->values, d_x, d_y,
                         pick_vector_width(A->nnz, A->M), 0, as_stream(stream), (size_t)A->N * sizeof(double), safe_vector_nnz(A));
}

int spmv_b200_csr_spmv_raw(int M, long long nnz, const int *d_row_ptr, const int *d_col_idx, const double *d_values,
                           const double *d_x, double *d_y, int threads_per_row, void *stream) {
    if (M < 0 || nnz < 0 || !d_row_ptr || !d_y) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_raw: bad arguments");
    const int vec = threads_per_row > 0 ? threads_per_row : pick_vector_width(nnz, M);
    return launch_vector(0, M, d_row_ptr, d_col_idx, d_values, d_x, d_y, vec, 0, as_stream(stream));
}

// ---- fp32 storage, fp64 arithmetic (SURVEY.md section 8(f).3; BASELINE.json: y within 1e-5 relative) ----------------
int spmv_b200_csr_enable_f32(spmv_b200_csr *A, void *stream) {
    if (!A) return fail(SPMV_B200_ERR_INVALID, "csr_enable_f32: NULL matrix");
    if (A->values32) return SPMV_B200_OK;
    const size_t padded = std::max<size_t>(((size_t)A->nnz + 3) & ~(size_t)3, 4);
    SPMV_TRY_CUDA(cudaMalloc(&A->values32, padded * sizeof(float)));
    SPMV_TRY_CUDA(cudaMemsetAsync(A->values32, 0, padded * sizeof(float), as_stream(stream)));
    if (A->nnz) {
        to_f32_kernel<<<blocks_for(A->nnz, 256), 256, 0, as_stream(stream)>>>(A->values, A->values32, A->nnz);
        SPMV_TRY_CUDA(cudaGetLastError());
    }
    A->row_batch32 = A->row_batch;
    if (A->max_row <= kRowKernelMaxLen && A->nnz >= kAutotuneMinNnz && env_int("SPMV_B200_AUTOTUNE", 1) &&
        env_int("SPMV_B200_ROW_BATCH", 0) == 0) {  // the best batch differs with the element size: time it again
        // candidates: one row per thread with batch 2..7, and the multi-row forms (csr_rowm_kernel, ids >= 16); all give
        // the same bits.  SPMV_B200_ROW_MULTI_TUNE=0 keeps the one-row forms only.
        int ids[8 + kNumRowmVariants], n = 0, fallback = 0;
        for (int batch = 2; batch <= 7; ++batch) {
            if (batch == A->row_batch) fallback = n;
            ids[n++] = batch;
        }
        if (env_int("SPMV_B200_ROW_MULTI_TUNE", 1))
            for (int v = 0; v < kNumRowmVariants; ++v) ids[n++] = 16 + v;
        const int pick = tune_candidates(A->M, A->N, n, fallback, as_stream(stream), [&](int i, double *x, double *y) {
            return launch_rows<float>(0, A->M, A->row_ptr, A->col_idx, A->values32, reinterpret_cast<const float *>(x),
                                      reinterpret_cast<float *>(y), ids[i], 0, as_stream(stream));
        });
        A->row_batch32 = ids[pick];
    }
    return SPMV_B200_OK;
}

int spmv_b200_csr_spmv_f32(const spmv_b200_csr *A, const float *d_x, float *d_y, int accumulate, int algo, void *stream) {
    if (!A || !d_y || (A->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_f32: NULL argument");
    if (!A->values32) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_f32: call spmv_b200_csr_enable_f32 first");
    if (A->M == 0) return SPMV_B200_OK;
    CsrPath path;
    switch (algo) {
        case SPMV_B200_ALGO_AUTO:
            path = A->max_row <= kRowKernelMaxLen ? kPathRow : csr_resolve(A, SPMV_B200_ALGO_AUTO);
            if (path == kPathStream || path == kPathTile) path = kPathBinned;  // no fp32 stream / tile kernels
            break;
        case SPMV_B200_ALGO_ROW: path = kPathRow; break;
        case SPMV_B200_ALGO_VECTOR: path = kPathVector; break;
        case SPMV_B200_ALGO_BINNED: path = kPathBinned; break;
        default: return fail(SPMV_B200_ERR_INVALID, "csr_spmv_f32: algo %d has no fp32 kernel (AUTO, VECTOR, BINNED, ROW)", algo);
    }
    cudaStream_t s = as_stream(stream);
    if (path == kPathRow) return launch_rows<float>(0, A->M, A->row_ptr, A->col_idx, A->values32, d_x, d_y, A->row_batch32, accumulate, s);
    if (path == kPathVector)
        return launch_vector<float>(0, A->M, A->row_ptr, A->col_idx, A->values32, d_x, d_y, pick_vector_width(A->nnz, A->M), accumulate, s,
                                    (size_t)A->N * sizeof(float), safe_vector_nnz(A));
    return launch_binned<float>(A, A->values32, d_x, d_y, accumulate, s);
}

int spmv_b200_csr_row_form_f32(const spmv_b200_csr *A) { return A && A->values32 ? A->row_batch32 : 0; }

int spmv_b200_row_forms(int format) {
    if (format == SPMV_B200_FORMAT_CSR) return kNumRowmVariants;
    if (format == SPMV_B200_FORMAT_HLL) return hll_row_forms();
    return 0;
}

int spmv_b200_row_form_describe(int format, int index, int *rows_per_thread, int *batch, int *ctas_per_sm) {
    int rows = 0, b = 0, ctas = 0;
    if (format == SPMV_B200_FORMAT_CSR && index >= 0 && index < kNumRowmVariants) {
        rows = kRowmVariants[index].rows;
        b = kRowmVariants[index].batch;
        ctas = kRowmVariants[index].ctas;
    } else if (format != SPMV_B200_FORMAT_HLL || hll_row_form(index, &rows, &b, &ctas) != 0) {
        return fail(SPMV_B200_ERR_INVALID, "row_form_describe: no form %d of format %d", index, format);
    }
    if (rows_per_thread) *rows_per_thread = rows;
    if (batch) *batch = b;
    if (ctas_per_sm) *ctas_per_sm = ctas;
    return SPMV_B200_OK;
}

int spmv_b200_csr_spmv_host_f32(spmv_b200_csr *A, const float *x, float *y) {
    if (!A || (A->M > 0 && !y) || (A->N > 0 && A->nnz > 0 && !x)) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_host_f32: NULL argument");
    if (A->M == 0) return SPMV_B200_OK;
    SPMV_TRY(spmv_b200_csr_enable_f32(A, nullptr));
    if (!A->stage_x) SPMV_TRY_CUDA(cudaMalloc(&A->stage_x, std::max<size_t>(A->N, 1) * sizeof(double)));
    if (!A->stage_y) SPMV_TRY_CUDA(cudaMalloc(&A->stage_y, std::max<size_t>(A->M, 1) * sizeof(double)));
    float *dx = reinterpret_cast<float *>(A->stage_x), *dy = reinterpret_cast<float *>(A->stage_y);
    if (A->N && x) SPMV_TRY_CUDA(cudaMemcpyAsync(dx, x, (size_t)A->N * sizeof(float), cudaMemcpyHostToDevice, nullptr));
    SPMV_TRY(spmv_b200_csr_spmv_f32(A, dx, dy, 0, SPMV_B200_ALGO_AUTO, nullptr));
    SPMV_TRY_CUDA(cudaMemcpyAsync(y, dy, (size_t)A->M * sizeof(float), cudaMemcpyDeviceToHost, nullptr));
    SPMV_TRY_CUDA(cudaStreamSynchronize(nullptr));
    return SPMV_B200_OK;
}

void spmv_b200_csr_free(spmv_b200_csr *A) {
    if (!A) return;
    free_plan(A);
    if (A->owns) {
        cudaFree(A->row_ptr);
        cudaFree(A->col_idx);
        cudaFree(A->values);
    }
    cudaFree(A->stage_x);
    cudaFree(A->stage_y);
    cudaFree(A->values32);
    host_pipe_free(A->pipe);
    host_pipe_free(A->spmm_pipe);
    delete A;
}

}  // extern "C"
