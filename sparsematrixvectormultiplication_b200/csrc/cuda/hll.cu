// hll.cu -- HLL (hacked ELLPACK, hack size 32) y = A*x for sm_100a: device image, slice kernel,
// conversions and the C-ABI entry points.
//
// Replaces the reference's spmv_hll_{naive,warp,warp_shared_v1}_kernel
// (reference cuda_src/hll_matrix.cu:346-479) and its array-of-structs device layout with one
// cudaMalloc pair per block (main_cuda.cu:369-402).
//
// Device image (DESIGN.md section 2): one flat arena, hack b occupies slots
// [hack_off[b], hack_off[b+1]) = 32*MAXNZ_b, COLUMN-MAJOR and hack-aligned:
//       slot(b, r, j) = hack_off[b] + j*32 + r          r in [0,32), j in [0,MAXNZ_b)
// Every hack holds 32 rows (the reference's short last block is padded with JA=0 / AS=0 rows), so
// every slice starts on a 128 B (JA) / 256 B (AS) boundary.  The host HLLMatrix stays in the
// reference's row-major layout; spmv_b200_hll_download converts back bit-exactly.
//
// Slice kernel: one warp per hack.  Lane = (jj, q) with jj = lane/8, q = lane%8 owns rows
// 4q..4q+3 of column j = 4*i + jj: one 128-bit load brings the 4 column indices, one 256-bit load
// the 4 values, so a warp consumes 4 whole columns (512 B + 1 KB, fully coalesced) per step.  The
// four partial sums per row are combined with two xor-shuffles.
#include <cub/cub.cuh>

#include <algorithm>
#include <type_traits>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "common.cuh"
#include "handles.cuh"

namespace spmv {

constexpr int kHack = HACK_SIZE;
constexpr int kHllThreads = 256;
constexpr int kHllWarps = kHllThreads / 32;
constexpr int kPadMark = (int)0x80000000u;  // bit 31 of JA: a padding slot of a CSR handle's private image (masked kernels)
constexpr int kPadMark16 = 0x8000;          // bit 15 of JA16: the same in the narrow image
constexpr int kDeltaMin = -16384, kDeltaMax = 16383;  // col - row of every slot of a narrow image (15-bit two's complement)

// The column field of a slot of a CSR handle's private image: the column a slot gathers, whether it adds, and the field of
// a slot past the width of its hack (gathers an in-range column, never adds).  int: the column, kPadMark on padding.
// uint16_t (JA16): bits 0-14 hold col - row, kPadMark16 on padding; a padding slot carries the delta of an in-range column
// too, so no gather is predicated on the loaded field.  first: the field of the first slot of the same batch.
__device__ __forceinline__ int ldg_stream_index(const int *p) { return ldg_stream_s32(p); }
__device__ __forceinline__ int ldg_stream_index(const uint16_t *p) { return ldg_stream_u16(p); }

template <typename I>
__device__ __forceinline__ int image_column(int c, unsigned row) {
    if constexpr (sizeof(I) == 2) return (int)(row + (unsigned)((int)((unsigned)c << 17) >> 17));  // modulo 2^32: exact
    else return c & ~kPadMark;
}

template <typename I>
__device__ __forceinline__ bool image_adds(int c) {
    if constexpr (sizeof(I) == 2) return (c & kPadMark16) == 0;
    else return c >= 0;
}

template <typename I>
__device__ __forceinline__ int image_past_width(int first) {
    if constexpr (sizeof(I) == 2) return first | kPadMark16;
    else return kPadMark;
}

// The value field of a slot: fp64 (or fp32 storage) as loaded, or a 1-byte code (S = uint8_t: the coded private image of a
// CSR handle) into the CTA's copy of the image's value table (image_table, staged by stage_image_table).  The load returns
// the code; the table is read at the multiply, so the step's global loads all go out ahead of it.
template <typename S>
using stored_t = typename std::conditional<sizeof(S) == 1, int, double>::type;
__device__ __forceinline__ double ldg_stream_value(const double *p) { return ldg_stream_f64(p); }
__device__ __forceinline__ double ldg_stream_value(const float *p) { return ldg_stream_f64(p); }
__device__ __forceinline__ int ldg_stream_value(const uint8_t *p) { return ldg_stream_u8(p); }
__device__ __forceinline__ double image_value(double v, const double *) { return v; }
__device__ __forceinline__ double image_value(int code, const double *tab) { return tab[code]; }

// the table of a coded image into shared memory (K >= 1 entries, dynamic shared memory of 8 K bytes); every thread of the
// CTA calls it, ahead of the kernel's warp-uniform early return
template <typename S>
__device__ __forceinline__ const double *stage_image_table(const double *__restrict__ table, int K) {
    extern __shared__ double image_table[];
    if constexpr (sizeof(S) == 1) {
        for (int i = threadIdx.x; i < K; i += blockDim.x) image_table[i] = __ldg(table + i);
        __syncthreads();
    }
    return image_table;
}

__device__ __forceinline__ void ldg_stream_f64x4(const float *p, double (&v)[4]) {  // fp32 storage: one 128-bit load
    float4 f;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(f.x), "=f"(f.y), "=f"(f.z), "=f"(f.w) : "l"(p));
    v[0] = f.x;
    v[1] = f.y;
    v[2] = f.z;
    v[3] = f.w;
}

template <typename V>
__device__ __forceinline__ void hll_step(const int *__restrict__ JA, const V *__restrict__ AS,
                                         const V *__restrict__ x, long long slot, double (&acc)[4]) {
    const int4 c = ldg_stream_s32x4(JA + slot);
    double v[4];
    ldg_stream_f64x4(AS + slot, v);
    acc[0] = fma(v[0], ldg_x(x, c.x), acc[0]);
    acc[1] = fma(v[1], ldg_x(x, c.y), acc[1]);
    acc[2] = fma(v[2], ldg_x(x, c.z), acc[2]);
    acc[3] = fma(v[3], ldg_x(x, c.w), acc[3]);
}

template <typename V>
__global__ void __launch_bounds__(kHllThreads)
hll_slice_kernel(int hack_begin, int hack_end, const long long *__restrict__ hack_off, const int *__restrict__ JA,
                 const V *__restrict__ AS, const V *__restrict__ x, V *__restrict__ y, int M) {
    const int hack = hack_begin + blockIdx.x * kHllWarps + (threadIdx.x >> 5);
    if (hack >= hack_end) return;  // warp-uniform
    const int lane = threadIdx.x & 31;
    const int jj = lane >> 3, q = lane & 7;
    const long long off = __ldg(hack_off + hack);
    const int width = (int)((__ldg(hack_off + hack + 1) - off) >> 5);
    const long long base = off + 4 * q;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    int j = jj;
    for (; j + 4 < width; j += 8) {  // two column groups in flight
        double a2[4] = {0.0, 0.0, 0.0, 0.0};
        hll_step(JA, AS, x, base + (long long)j * kHack, acc);
        hll_step(JA, AS, x, base + (long long)(j + 4) * kHack, a2);
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[e] += a2[e];
    }
    if (j < width) hll_step(JA, AS, x, base + (long long)j * kHack, acc);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 8);
        acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 16);
    }
    if (jj == 0) {
        const int row = hack * kHack + 4 * q;
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (row + e < M) y[row + e] = (V)acc[e];
    }
}

// The hack-row loop of every lane-per-row HLL kernel: acc plus the products of row `row` of a hack, whose slot j lies at
// base + j * 32 (j < width), BATCH slots requested before the first gather.  One lane per row, sequential in j, mul and
// add rounded separately: bit-identical to the reference's spmv_hll_serial (src/hll_matrix.c:294-306), padding slots
// (x 0.0) included.  MASKED: the private image of a CSR handle (image.cu), whose padding slots carry bit 31 of the
// column (I = int) or bit 15 of a row-relative 16-bit field (I = uint16_t, image_column).  Such a slot gathers its column
// like any other and skips the add: bit-identical to csr_row_kernel for every x.  (Adding the padding's 0 * x[c] would
// give NaN for an infinite x[c], and +0 turns an untouched -0.0 positive.)  The loads are never predicated on the loaded
// column.  S: the stored value type -- V, or uint8_t for codes into `tab` (unused otherwise).
template <int BATCH, typename V, bool MASKED = false, typename I = int, typename S = V>
__device__ __forceinline__ double hack_row_sum(long long base, int width, long long row, const I *__restrict__ JA,
                                               const S *__restrict__ AS, const V *__restrict__ x, const double *tab,
                                               double acc) {
    for (int j = 0; j < width; j += BATCH) {
        int c[BATCH];
        stored_t<S> v[BATCH];
        double xv[BATCH];
#pragma unroll
        for (int u = 0; u < BATCH; ++u)  // u = 0 is always within the width
            c[u] = j + u < width ? ldg_stream_index(JA + base + (long long)(j + u) * kHack) : (MASKED ? image_past_width<I>(u ? c[0] : 0) : -1);
#pragma unroll
        for (int u = 0; u < BATCH; ++u) v[u] = j + u < width ? ldg_stream_value(AS + base + (long long)(j + u) * kHack) : 0;
#pragma unroll
        for (int u = 0; u < BATCH; ++u)
            xv[u] = MASKED ? ldg_x(x, image_column<I>(c[u], (unsigned)row)) : (c[u] >= 0 ? ldg_x(x, c[u]) : 0.0);
#pragma unroll
        for (int u = 0; u < BATCH; ++u)
            if (MASKED ? image_adds<I>(c[u]) : c[u] >= 0) acc = __dadd_rn(acc, __dmul_rn(image_value(v[u], tab), xv[u]));
    }
    return acc;
}

// Row kernel for narrow hacks (stencils): one warp per hack, lane = row, the column-major image makes every load of a
// warp one contiguous 128 B (JA) / 256 B (AS) segment -- no shared memory, no reliance on L1 for the stream.  MASKED, I
// and S as in hack_row_sum; ACCUM: the sum starts from y[row].  ACCUM is a template flag, not an argument: a y[row] load
// hoisted ahead of the step holds two of the 32 registers and pushed two of the 15 loads of hll_rowu_kernel<5> behind the
// first multiply (cuobjdump, tools/rowm_survey.py).  The coded image's `table` (K entries) is staged in shared memory.
template <int BATCH, typename V, bool MASKED = false, bool ACCUM = false, typename I = int, typename S = V>
__global__ void __launch_bounds__(256, 8)
hll_row_kernel(int hack_begin, int hack_end, const long long *__restrict__ hack_off, const I *__restrict__ JA,
               const S *__restrict__ AS, const V *__restrict__ x, V *__restrict__ y, int M, const double *__restrict__ table, int K) {
    static_assert(sizeof(I) == 4 || (MASKED && sizeof(V) == 8), "the narrow index exists in the fp64 private image only");
    static_assert(sizeof(S) == sizeof(V) || (MASKED && sizeof(V) == 8), "value codes exist in the fp64 private image only");
    const double *tab = stage_image_table<S>(table, K);
    const int hack = hack_begin + blockIdx.x * 8 + (threadIdx.x >> 5);
    if (hack >= hack_end) return;  // warp-uniform
    const int lane = threadIdx.x & 31;
    const long long row = (long long)hack * kHack + lane;
    const long long off = __ldg(hack_off + hack);
    const int width = (int)((__ldg(hack_off + hack + 1) - off) >> 5);
    const long long base = off + lane;
    const double acc = hack_row_sum<BATCH, V, MASKED, I, S>(base, width, row, JA, AS, x, tab, ACCUM && row < M ? (double)y[row] : 0.0);
    if (row < M) y[row] = (V)acc;
}

// hll_row_kernel in a second form (round 2e; candidates of the fp32 path; see csr_rowm_kernel in csr.cu): slots past the
// width of a hack gather x[0] and are skipped by `j < width` instead of being predicated on the LOADED column, so every
// predicate is index arithmetic and ptxas issues all loads of a step ahead of the first multiply (17 of 17 for <5, 1, 8,
// float> against 9 of 17).  lap2d 4096^2, fp32 storage: 145.8 us against 166.5 us for the best hll_row_kernel batch
// (profiles/r02e_rowm_probe_second_pass.log); not so on lap3d 256^3 or with fp64 storage, hence plan-time candidates.
// HACKS > 1 (every lane owns row `lane` of HACKS consecutive hacks, CTAS CTAs per SM) tested the idea that more rows in
// flight per SM would cover the latency of the lighter fp32 rows: refuted, 10-100 % slower; kept for the record.
// Order of the sums unchanged, padding slots (x 0.0) included: the same bits as hll_row_kernel.
template <int BATCH, int HACKS, int CTAS, typename V>
__global__ void __launch_bounds__(256, CTAS)
hll_rowm_kernel(int hack_begin, int hack_end, const long long *__restrict__ hack_off, const int *__restrict__ JA,
                const V *__restrict__ AS, const V *__restrict__ x, V *__restrict__ y, int M) {
    const int first = hack_begin + (blockIdx.x * 8 + (threadIdx.x >> 5)) * HACKS;
    if (first >= hack_end) return;  // warp-uniform
    const int lane = threadIdx.x & 31;
    long long off[HACKS + 1];
#pragma unroll
    for (int h = 0; h <= HACKS; ++h) off[h] = __ldg(hack_off + min(first + h, hack_end));
    int width[HACKS], widest = 0;
    double acc[HACKS];
#pragma unroll
    for (int h = 0; h < HACKS; ++h) {
        width[h] = first + h < hack_end ? (int)((off[h + 1] - off[h]) >> 5) : 0;
        widest = max(widest, width[h]);
        acc[h] = 0.0;
    }
    for (int j = 0; j < widest; j += BATCH) {
        int c[HACKS][BATCH];
        double v[HACKS][BATCH], xv[HACKS][BATCH];
#pragma unroll
        for (int h = 0; h < HACKS; ++h)
#pragma unroll
            for (int u = 0; u < BATCH; ++u)
                c[h][u] = j + u < width[h] ? ldg_stream_s32(JA + off[h] + lane + (long long)(j + u) * kHack) : 0;
#pragma unroll
        for (int h = 0; h < HACKS; ++h)
#pragma unroll
            for (int u = 0; u < BATCH; ++u)
                v[h][u] = j + u < width[h] ? ldg_stream_f64(AS + off[h] + lane + (long long)(j + u) * kHack) : 0.0;
#pragma unroll
        for (int h = 0; h < HACKS; ++h)
#pragma unroll
            for (int u = 0; u < BATCH; ++u) xv[h][u] = ldg_x(x, c[h][u]);
#pragma unroll
        for (int h = 0; h < HACKS; ++h)
#pragma unroll
            for (int u = 0; u < BATCH; ++u)
                if (j + u < width[h]) acc[h] = __dadd_rn(acc[h], __dmul_rn(v[h][u], xv[h][u]));
    }
#pragma unroll
    for (int h = 0; h < HACKS; ++h) {
        const long long row = (long long)(first + h) * kHack + lane;
        if (first + h < hack_end && row < M) y[row] = (V)acc[h];
    }
}

// The lane-per-row kernel WITHOUT the hack_off round trip (round 2e; fp32 path and regular images only): when the image
// consists of at most kMaxHllSegments runs of hacks of equal width -- a 2-D stencil: one run per grid-row class, three
// on lap2d -- a warp finds its run with a handful of compares on kernel parameters and computes its first slot, so the
// row's dependent chain is two memory round trips (JA / AS -> x) instead of three.  Same loop, same order, same bits as
// hll_rowm_kernel<BATCH, 1, 8>.  Form ids 64 + BATCH of the fp32 tuner.  Measured (lap2d 4096^2, fp32 storage,
// profiles/r02e_rowm_probe_third_pass.log): 139.9 us against 146.0 us for hll_rowm_kernel<5, 1, 8> and 166.4 us for
// hll_row_kernel<5> -- the first round trip is worth 4 %, not the third of the time a pure latency model gives it.  Two
// other ways to shorten that trip on images that are NOT regular, tried and removed: the hack_off line of the CTA N CTAs
// further on prefetched into L2 by one thread per CTA (141-142 us at every N from 148 to 9472: the same 3 %), and the
// offset array held in the persisting L2 carve-out (194.6 us: the carve-out costs the gathers more than the trip saves).
// MASKED / ACCUM / I / S: as in hll_row_kernel -- the private image of a CSR handle, bit for bit csr_row_kernel.
template <int BATCH, typename V, bool MASKED = false, bool ACCUM = false, typename I = int, typename S = V>
__global__ void __launch_bounds__(256, 8)
hll_rowu_kernel(int hack_begin, int hack_end, const __grid_constant__ HllSegments seg, const I *__restrict__ JA,
                const S *__restrict__ AS, const V *__restrict__ x, V *__restrict__ y, int M, const double *__restrict__ table, int K) {
    static_assert(sizeof(I) == 4 || (MASKED && sizeof(V) == 8), "the narrow index exists in the fp64 private image only");
    static_assert(sizeof(S) == sizeof(V) || (MASKED && sizeof(V) == 8), "value codes exist in the fp64 private image only");
    const double *tab = stage_image_table<S>(table, K);
    const int hack = hack_begin + blockIdx.x * 8 + (threadIdx.x >> 5);
    if (hack >= hack_end) return;  // warp-uniform
    const int lane = threadIdx.x & 31;
    int first = seg.begin[0], width = seg.width[0];
    long long base = seg.base[0];
#pragma unroll
    for (int s = 1; s < kMaxHllSegments; ++s)
        if (hack >= seg.begin[s]) {  // unused entries hold INT_MAX (hll_find_segments)
            first = seg.begin[s];
            width = seg.width[s];
            base = seg.base[s];
        }
    const long long off = base + (long long)(hack - first) * kHack * width + lane;
    const long long row = (long long)hack * kHack + lane;
    double acc = ACCUM && row < M && width != BATCH ? (double)y[row] : 0.0;
    if (width == BATCH) {
        // the run's width IS the batch (the form the tuner ends up with on a stencil): straight-line code, no predicates.
        // ncu on the predicated loop alone (profiles/r02e_ncu_f32_summary.md): issue slots 70 % busy, SM throughput 84 %
        // -- without the offset trip this kernel is close to instruction-issue bound, so instructions count.
        int c[BATCH];
        stored_t<S> v[BATCH];
        double xv[BATCH];
#pragma unroll
        for (int u = 0; u < BATCH; ++u) c[u] = ldg_stream_index(JA + off + (long long)u * kHack);
#pragma unroll
        for (int u = 0; u < BATCH; ++u) v[u] = ldg_stream_value(AS + off + (long long)u * kHack);
#pragma unroll
        for (int u = 0; u < BATCH; ++u) xv[u] = ldg_x(x, MASKED ? image_column<I>(c[u], (unsigned)row) : c[u]);
        if (ACCUM && row < M) acc = y[row];  // after the step's loads: held from the start, it pushed the narrow form to spill
#pragma unroll
        for (int u = 0; u < BATCH; ++u)
            if (!MASKED || image_adds<I>(c[u])) acc = __dadd_rn(acc, __dmul_rn(image_value(v[u], tab), xv[u]));
    } else
    for (int j = 0; j < width; j += BATCH) {
        int c[BATCH];
        stored_t<S> v[BATCH];
        double xv[BATCH];
#pragma unroll
        for (int u = 0; u < BATCH; ++u)  // u = 0 is always within the width
            c[u] = j + u < width ? ldg_stream_index(JA + off + (long long)(j + u) * kHack) : (MASKED ? image_past_width<I>(u ? c[0] : 0) : 0);
#pragma unroll
        for (int u = 0; u < BATCH; ++u) v[u] = j + u < width ? ldg_stream_value(AS + off + (long long)(j + u) * kHack) : 0;
#pragma unroll
        for (int u = 0; u < BATCH; ++u) xv[u] = ldg_x(x, MASKED ? image_column<I>(c[u], (unsigned)row) : c[u]);
#pragma unroll
        for (int u = 0; u < BATCH; ++u)
            if (j + u < width && (!MASKED || image_adds<I>(c[u]))) acc = __dadd_rn(acc, __dmul_rn(image_value(v[u], tab), xv[u]));
    }
    if (row < M) y[row] = (V)acc;
}

// (HACKS, BATCH, CTAS per SM) forms of hll_rowm_kernel offered to the plan-time tuner of the fp32 path
struct HllRowmVariant {
    int hacks, batch, ctas;
};
#define SPMV_HLL_ROWM_VARIANTS(X) \
    X(1, 4, 8) X(1, 5, 8) X(1, 6, 8) X(1, 7, 8) X(1, 7, 6) X(2, 3, 5) X(2, 5, 4) X(3, 3, 4)
#define HROWM_ENTRY(H, B, C) {H, B, C},
static const HllRowmVariant kHllRowmVariants[] = {SPMV_HLL_ROWM_VARIANTS(HROWM_ENTRY)};
#undef HROWM_ENTRY
constexpr int kNumHllRowmVariants = (int)(sizeof kHllRowmVariants / sizeof kHllRowmVariants[0]);

int hll_row_forms() { return kNumHllRowmVariants; }
int hll_row_form(int index, int *hacks, int *batch, int *ctas) {
    if (index < 0 || index >= kNumHllRowmVariants) return -1;
    *hacks = kHllRowmVariants[index].hacks;
    *batch = kHllRowmVariants[index].batch;
    *ctas = kHllRowmVariants[index].ctas;
    return 0;
}

// hll_row_kernel with the tail of the two-launch iterated product (spmv_b200_hll_spmv_fused_flat): one warp per hack, one
// CTA per 8 hacks = 256 rows, no chunk walk and no waiting -- the body of the plain kernel, then scale by 1/|w_prev| (read
// from memory), store, mirror boundary rows, one partial sum of squares per CTA (see csr_row_flat_kernel).  Thread t of
// CTA b owns row 256 b + t as in the CSR kernel: same partials, bitwise the CSR iteration on the same partition.
template <int BATCH>
__global__ void __launch_bounds__(256, 8)
hll_row_flat_kernel(int num_hacks, const long long *__restrict__ hack_off, const int *__restrict__ JA,
                    const double *__restrict__ AS, const double *__restrict__ x, double *__restrict__ y, int M,
                    const __grid_constant__ Epilogue ep) {
    __shared__ double warp_sq[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int hack = blockIdx.x * 8 + warp;
    const long long row = (long long)blockIdx.x * 256 + threadIdx.x;
    double acc = 0.0;
    if (hack < num_hacks) {  // warp-uniform
        const long long off = __ldg(hack_off + hack);
        const int width = (int)((__ldg(hack_off + hack + 1) - off) >> 5);
        const long long base = off + lane;
        acc = hack_row_sum<BATCH, double>(base, width, row, JA, AS, x, nullptr, 0.0);
        if (row < M) {
            if (ep.inv_norm != nullptr) acc *= __ldg(ep.inv_norm);
            y[row] = acc;
            if (fused_chunk_is_boundary(ep, (long long)blockIdx.x * 256)) fused_peer_store(ep, row, acc);
        } else {
            acc = 0.0;  // padding rows of the last hack
        }
    }
    if (ep.partials == nullptr) return;
    double sq = acc * acc;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, off);
    if (lane == 0) warp_sq[warp] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double total = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) total += warp_sq[w];
        ep.partials[blockIdx.x] = total;
    }
}

// The lane-per-row kernel with the fused tail of the iterated product (Epilogue, handles.cuh): the HLL twin of
// csr_row_fused_kernel.  A fixed grid walks the hacks in chunks of 8 (= 256 rows, one warp per hack, thread t of the CTA
// owns row chunk*256 + t exactly as in the CSR kernel), so for the same row partition both formats produce the same
// per-CTA partials: |w|^2, lambda and x are bitwise equal to the CSR iteration on rows without padding effects (a
// padding slot adds v*x = +0.0, which leaves every finite sum unchanged).  Reference: spmv_hll (src/hll_matrix.c:376-408)
// computes the per-block-range product; the scale / norm / exchange tail has no reference counterpart (BASELINE config 5).
template <int BATCH>
__global__ void __launch_bounds__(256, 8)
hll_row_fused_kernel(int num_hacks, const long long *__restrict__ hack_off, const int *__restrict__ JA,
                     const double *__restrict__ AS, const double *__restrict__ x, double *__restrict__ y, int M,
                     const __grid_constant__ Epilogue ep) {
    __shared__ double warp_sq[8];
    __shared__ double mail_total;
    bool scaled;
    const double inv_norm = fused_inv_norm(ep, scaled, &mail_total);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double sq = 0.0;
    const int chunks = (M + 255) >> 8;
    for (int q = blockIdx.x; q < chunks; q += gridDim.x) {  // the walk of csr_row_fused_kernel, chunk for chunk
        const long long chunk_lo = (long long)ordered_chunk(ep.order, q) * 256;
        const bool boundary = ep.order.boundary_chunks > 0 ? q < ep.order.boundary_chunks : fused_chunk_is_boundary(ep, chunk_lo);
        const int hack = (int)(chunk_lo >> 5) + warp;
        if (hack >= num_hacks) continue;  // warp-uniform
        const long long off = __ldg(hack_off + hack);
        const int width = (int)((__ldg(hack_off + hack + 1) - off) >> 5);
        const long long base = off + lane;
        double acc = hack_row_sum<BATCH, double>(base, width, chunk_lo + threadIdx.x, JA, AS, x, nullptr, 0.0);
        const long long row = chunk_lo + threadIdx.x;
        if (row >= M) continue;
        if (scaled) acc *= inv_norm;
        sq = fma(acc, acc, sq);
        y[row] = acc;
        if (boundary) fused_peer_store(ep, row, acc);
    }
    fused_finish(ep, sq, warp_sq);
}

// ---- CSR -> HLL on the device ----------------------------------------------------------------------
__global__ void hll_width_kernel(int M, int num_hacks, const int *__restrict__ row_ptr, long long *__restrict__ slots) {
    const int hack = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (hack > num_hacks) return;
    const int lane = threadIdx.x & 31;
    int len = 0;
    if (hack < num_hacks) {
        const long long r = (long long)hack * kHack + lane;
        if (r < M) len = row_ptr[r + 1] - row_ptr[r];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, off));
    if (lane == 0) slots[hack] = (long long)len * kHack;  // slots[num_hacks] = 0: the scan ends with the total
}

// the column field of a slot (mark: OR'ed into a padding slot's column of the wide image; the narrow one is always masked)
__device__ __forceinline__ void put_index(int *JA, long long slot, int col, long long, bool pad, int mark) {
    JA[slot] = pad ? col | mark : col;
}
__device__ __forceinline__ void put_index(uint16_t *JA, long long slot, int col, long long row, bool pad, int) {
    JA[slot] = (uint16_t)(((unsigned long long)(col - row) & 0x7fffu) | (pad ? kPadMark16 : 0));
}

// the code of a value in the ascending table of the K distinct 64-bit patterns of a coded image (the pattern is there)
__device__ __forceinline__ int value_code(const double *__restrict__ table, int K, double v) {
    const unsigned long long k = (unsigned long long)__double_as_longlong(v);
    int lo = 0, hi = K - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((unsigned long long)__double_as_longlong(table[mid]) < k) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// AS (fp64 values) and AC (1-byte codes into table[K]) are each filled when not NULL; a padding slot holds 0.0 / code 0
template <typename I>
__global__ void hll_fill_kernel(int M, int N, int num_hacks, const int *__restrict__ row_ptr, const int *__restrict__ col_idx,
                                const double *__restrict__ values, const long long *__restrict__ hack_off,
                                I *__restrict__ JA, double *__restrict__ AS, uint8_t *__restrict__ AC,
                                const double *__restrict__ table, int K, int mark) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= (long long)num_hacks * kHack) return;
    const int hack = (int)(r / kHack), lr = (int)(r % kHack);
    const long long off = hack_off[hack];
    const int width = (int)((hack_off[hack + 1] - off) >> 5);
    int begin = 0, len = 0;
    if (r < M) {
        begin = row_ptr[r];
        len = row_ptr[r + 1] - begin;
    }
    // reference: padding repeats the last real column, 0 for an empty row.  The narrow image stores col - row, so an
    // empty row (or a row past M) gathers the in-range column nearest to it instead (hll_narrow_check_kernel)
    int pad_col = sizeof(I) == 2 ? (int)min(r, (long long)N - 1) : 0;
    for (int j = 0; j < width; ++j) {
        const long long slot = off + (long long)j * kHack + lr;
        if (j < len) {
            pad_col = col_idx[begin + j];
            put_index(JA, slot, pad_col, r, false, mark);
            const double v = values[begin + j];
            if (AS) AS[slot] = v;
            if (AC) AC[slot] = (uint8_t)value_code(table, K, v);
        } else {
            put_index(JA, slot, pad_col, r, true, mark);
            if (AS) AS[slot] = 0.0;
            if (AC) AC[slot] = 0;
        }
    }
}

// Does every slot of the image fit the narrow field (col - row in [kDeltaMin, kDeltaMax])?  One thread per row of the
// padded image: a real slot holds col - row, a padding slot repeats the delta of its row's last real column or, in a row
// without one that still has slots, gathers min(row, N - 1) (hll_fill_kernel).  Clears *fits.
__global__ void hll_narrow_check_kernel(int M, int N, int num_hacks, const int *__restrict__ row_ptr,
                                        const int *__restrict__ col_idx, const long long *__restrict__ hack_off,
                                        int *__restrict__ fits) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= (long long)num_hacks * kHack) return;
    int begin = 0, end = 0;
    if (r < M) {
        begin = row_ptr[r];
        end = row_ptr[r + 1];
    }
    bool ok = true;
    for (int k = begin; k < end; ++k) {
        const long long d = col_idx[k] - r;
        ok = ok && d >= kDeltaMin && d <= kDeltaMax;
    }
    if (begin == end && hack_off[r / kHack + 1] > hack_off[r / kHack]) ok = r - (N - 1) <= -kDeltaMin;
    if (!ok) *fits = 0;
}

}  // namespace spmv


using namespace spmv;

template <typename V>
static int hll_launch_rows_t(const spmv_b200_hll *H, const V *AS, int hack_begin, int hack_end, const V *d_x, V *d_y,
                             cudaStream_t stream, int batch = -1) {
    if (hack_end <= hack_begin) return SPMV_B200_OK;
    if (batch < 0) batch = sizeof(V) == 4 ? H->row_batch32 : (H->row_form > 0 ? H->row_form : H->row_batch);
    const XPolicy keep = matrix_policy(H->JA, (size_t)H->slots * sizeof(int));   // head of JA held in L2 across products
    // batch >= 16: hll_rowm_kernel, form kHllRowmVariants[batch - 16].  SPMV_B200_ROW_MULTI=k (k >= 1) sends EVERY
    // row-kernel launch through form k - 1 (parity runs: tests/test_gpu_parity.py walks all forms, fp64 bit for bit)
    const int forced_multi = env_int("SPMV_B200_ROW_MULTI", 0);
    // ids 64 + B: hll_rowu_kernel<B> (offsets by arithmetic; regular images only).  SPMV_B200_HLL_UNIFORM=B forces it
    // on every row launch of an image that qualifies (parity runs).
    const int forced_uniform = env_int("SPMV_B200_HLL_UNIFORM", 0);
    const int uniform = batch >= 64 ? batch - 64 : (forced_uniform >= 3 && forced_uniform <= 7 && H->segments.count > 0 ? forced_uniform : 0);
    if (uniform > 0) {
        if (H->segments.count <= 0) return fail(SPMV_B200_ERR_INVALID, "hll row kernel: the image is not regular enough for the offset-free form");
        const unsigned int gu = blocks_for(hack_end - hack_begin, 8);
        SPMV_TRY_CUDA((with_batch<5, 3, 4, 6, 7>(uniform, [&](auto B) {
            return launch_x(hll_rowu_kernel<B, V>, gu, 256, 0, stream, keep, hack_begin, hack_end, H->segments, H->JA, AS, d_x, d_y, H->M, nullptr, 0);
        })));
        SPMV_TRY_CUDA(cudaGetLastError());
        return SPMV_B200_OK;
    }
    const int variant = forced_multi >= 1 ? std::min(forced_multi, kNumHllRowmVariants) - 1 : batch - 16;
    if (variant >= 0) {
        if (variant >= kNumHllRowmVariants) return fail(SPMV_B200_ERR_INVALID, "hll row kernel: unknown multi-hack form %d", variant);
        const unsigned int gm = blocks_for(hack_end - hack_begin, 8 * kHllRowmVariants[variant].hacks);
        int at = 0;
#define HROWM_CASE(R, B, C)                                                                                                  \
    if (at++ == variant)                                                                                                     \
        SPMV_TRY_CUDA(launch_x(hll_rowm_kernel<B, R, C, V>, gm, 256, 0, stream, keep, hack_begin, hack_end, H->hack_off, H->JA, AS, \
                               d_x, d_y, H->M));
        SPMV_HLL_ROWM_VARIANTS(HROWM_CASE)
#undef HROWM_CASE
        SPMV_TRY_CUDA(cudaGetLastError());
        return SPMV_B200_OK;
    }
    const unsigned int g = blocks_for(hack_end - hack_begin, 8);
    SPMV_TRY_CUDA((with_batch<4, 1, 2, 3, 5, 6, 7, 8>(batch, [&](auto B) {
        return launch_x(hll_row_kernel<B, V>, g, 256, 0, stream, keep, hack_begin, hack_end, H->hack_off, H->JA, AS, d_x, d_y, H->M, nullptr, 0);
    })));
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

// grid of the fused row kernel: 8 CTAs of 256 threads per SM, whatever the matrix size (same rule as the CSR kernel)
static int hll_fused_grid(const spmv_b200_hll *H) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (int)std::max<long long>(1, std::min<long long>((long long)fused_ctas_per_sm() * sms, ((long long)H->M + 255) / 256));
}

static int hll_launch_fused(const spmv_b200_hll *H, const double *d_x, double *d_y, const Epilogue &ep, cudaStream_t stream,
                            int batch = -1) {
    if (batch < 0) batch = env_int("SPMV_B200_HLL_FUSED_BATCH", H->fused_batch > 0 ? H->fused_batch : H->row_batch);
    const int g = hll_fused_grid(H);
    with_batch<4, 2, 3, 5, 6, 7>(batch, [&](auto B) {
        hll_row_fused_kernel<B><<<g, 256, 0, stream>>>(H->num_hacks, H->hack_off, H->JA, H->AS, d_x, d_y, H->M, ep);
    });
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

// the FLAT form (two-launch iterated product): one CTA per 8 hacks; the batch is timed at plan time
static int hll_flat_grid(long long M) { return (int)std::max<long long>(1, (M + 255) / 256); }

static int hll_launch_fused_flat(const spmv_b200_hll *H, const double *d_x, double *d_y, const Epilogue &ep, cudaStream_t stream,
                                 int batch) {
    const int g = hll_flat_grid(H->M);
    const XPolicy keep = matrix_policy(H->JA, (size_t)H->slots * sizeof(int));
    SPMV_TRY_CUDA((with_batch<4, 2, 3, 5, 6, 7>(batch, [&](auto B) {
        return launch_x(hll_row_flat_kernel<B>, g, 256, 0, stream, keep, H->num_hacks, H->hack_off, H->JA, H->AS, d_x, d_y, H->M, ep);
    })));
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

static const int kHllFlatCandidates[] = {2, 3, 4, 5, 6, 7};

static int hll_launch_rows(const spmv_b200_hll *H, int hack_begin, int hack_end, const double *d_x, double *d_y,
                           cudaStream_t stream) {
    return hll_launch_rows_t<double>(H, H->AS, hack_begin, hack_end, d_x, d_y, stream);
}

static int hll_launch(const spmv_b200_hll *H, int hack_begin, int hack_end, const double *d_x, double *d_y,
                      cudaStream_t stream) {
    if (hack_end <= hack_begin) return SPMV_B200_OK;
    SPMV_TRY_CUDA(launch_x(hll_slice_kernel<double>, blocks_for(hack_end - hack_begin, kHllWarps), kHllThreads, 0, stream,
                           x_policy(d_x, (size_t)H->N * sizeof(double)), hack_begin, hack_end, H->hack_off, H->JA, H->AS, d_x,
                           d_y, H->M));
    return SPMV_B200_OK;
}

static int hll_alloc_arena(spmv_b200_hll *H) {
    const size_t n = (size_t)std::max<long long>(H->slots, 32);
    SPMV_TRY_CUDA(cudaMalloc(&H->JA, n * sizeof(int)));
    SPMV_TRY_CUDA(cudaMalloc(&H->AS, n * sizeof(double)));
    return SPMV_B200_OK;
}

namespace spmv {
// no hack wider than 16 columns (stencils): lane-per-row kernel, coalesced by the column-major layout; narrow on
// average: TMA stream kernel; wide hacks are gather bound and need the occupancy of the slice kernel
HllPath hll_resolve(const spmv_b200_hll *H) {
    if (H->max_width <= kRowKernelMaxLen) return H->narrow_stream ? kHllStream : kHllRows;
    return H->slots <= 12LL * 32 * H->num_hacks ? kHllStream : kHllSlice;
}

int hll_launch_window(const spmv_b200_hll *H, HllPath path, int unit_begin, int unit_end, const double *x, double *y,
                      cudaStream_t stream) {
    if (path == kHllStream) return stream_launch_hll(H, x, y, stream, unit_begin, unit_end - unit_begin);
    if (path == kHllRows) return hll_launch_rows(H, unit_begin, unit_end, x, y, stream);
    return hll_launch(H, unit_begin, unit_end, x, y, stream);
}

// batch of the lane-per-row kernel: the hack width when it is uniform and small; timed at plan time on large images
// runs of hacks of equal width, from the host copy of the offsets (HllSegments, handles.cuh)
HllSegments hll_find_segments(const std::vector<long long> &off, int num_hacks) {
    HllSegments seg;
    bool regular = (int)off.size() == num_hacks + 1 && num_hacks > 0;
    for (int h = 0; regular && h < num_hacks; ++h) {
        const int w = (int)((off[h + 1] - off[h]) / kHack);
        if (seg.count > 0 && seg.width[seg.count - 1] == w) continue;
        if (seg.count == kMaxHllSegments) {
            regular = false;
            break;
        }
        seg.begin[seg.count] = h;
        seg.width[seg.count] = w;
        seg.base[seg.count] = off[h];
        ++seg.count;
    }
    if (!regular) seg = HllSegments();
    else {
        seg.begin[seg.count] = num_hacks;
        for (int s = seg.count + 1; s <= kMaxHllSegments; ++s) seg.begin[s] = 0x7fffffff;  // never reached: the kernel tests no count
    }
    return seg;
}

static void hll_pick_row_batch(spmv_b200_hll *H, cudaStream_t stream) {
    H->segments = hll_find_segments(H->host_off, H->num_hacks);
    const int forced = env_int("SPMV_B200_HLL_ROW_BATCH", 0);
    H->narrow_stream = false;
    H->row_form = 0;
    const long long mean = H->num_hacks > 0 ? (H->slots / 32 + H->num_hacks - 1) / H->num_hacks : 4;
    H->row_batch = (int)std::max<long long>(2, std::min<long long>(7, mean));
    if (forced >= 1 && forced <= 8) {
        H->row_batch = forced;
    } else if (H->max_width <= kRowKernelMaxLen && H->slots >= (1 << 22) && env_int("SPMV_B200_AUTOTUNE", 1)) {
        const int best = tune_batch(H->M, H->N, H->row_batch, stream, [&](int batch, double *x, double *y) {
            if (batch == 0) return stream_launch_hll(H, x, y, stream);
            const int keep = H->row_batch;
            H->row_batch = batch;
            const int rc = hll_launch_rows(H, 0, H->num_hacks, x, y, stream);
            H->row_batch = keep;
            return rc;
        }, 0);
        if (best == 0) H->narrow_stream = true;
        else H->row_batch = best;
        // regular images: hll_rowu_kernel (no hack_off round trip; ids 64 + batch) against the winner so far -- same bits.
        // lap2d 4096^2, fp64: 182.1 us against 201.3 us (profiles/r02e_rowm_probe_fourth_pass.log)
        if (H->segments.count > 0 && env_int("SPMV_B200_HLL_UNIFORM_TUNE", 1)) {
            const int ids[5] = {-1, 64 + 4, 64 + 5, 64 + 6, 64 + 7};  // -1: the winner so far
            const int pick = tune_candidates(H->M, H->N, 5, 0, stream, [&](int i, double *x, double *y) {
                if (ids[i] < 0)
                    return H->narrow_stream ? stream_launch_hll(H, x, y, stream) : hll_launch_rows(H, 0, H->num_hacks, x, y, stream);
                return hll_launch_rows_t<double>(H, H->AS, 0, H->num_hacks, x, y, stream, ids[i]);
            });
            if (pick > 0) {
                H->row_form = ids[pick];
                H->narrow_stream = false;
            }
        }
        // the fused iterated product (scale + |w|^2 partials in the tail) has its own best batch
        double *partials = nullptr;
        const int count = hll_fused_grid(H);
        if (cudaMalloc(&partials, (size_t)count * sizeof(double)) == cudaSuccess) {
            Epilogue ep;
            ep.partials = partials;
            ep.partials_total = count;
            H->fused_batch = tune_batch(H->M, H->N, H->row_batch, stream, [&](int batch, double *x, double *y) {
                return hll_launch_fused(H, x, y, ep, stream, batch);
            });
        }
        cudaGetLastError();
        cudaFree(partials);
        partials = nullptr;
        if (cudaMalloc(&partials, (size_t)hll_flat_grid(H->M) * sizeof(double)) == cudaSuccess) {  // the FLAT form
            Epilogue fe;
            fe.partials = partials;
            fe.partials_total = hll_flat_grid(H->M);
            fe.inv_norm = partials;  // any finite double will do for the timing
            const int n = (int)(sizeof kHllFlatCandidates / sizeof kHllFlatCandidates[0]);
            const int pick = tune_candidates(H->M, H->N, n, 1, stream, [&](int i, double *x, double *y) {
                return hll_launch_fused_flat(H, x, y, fe, stream, kHllFlatCandidates[i]);
            });
            H->flat_batch = kHllFlatCandidates[pick];
        }
        cudaGetLastError();
        cudaFree(partials);
    }
}

int hll_layout(int M, int N, const int *row_ptr, const int *col_idx, cudaStream_t stream, long long **hack_off,
               std::vector<long long> &host_off, int *max_width, bool *narrow) {
    const int nb = (M + kHack - 1) / kHack;
    long long *slots = nullptr;
    void *temp = nullptr;
    int *d_fits = nullptr, fits = 1;
    auto body = [&]() -> int {
        SPMV_TRY_CUDA(cudaMalloc(hack_off, ((size_t)nb + 1) * sizeof(long long)));
        SPMV_TRY_CUDA(cudaMalloc(&slots, ((size_t)nb + 1) * sizeof(long long)));
        hll_width_kernel<<<blocks_for(nb + 1, 8), 256, 0, stream>>>(M, nb, row_ptr, slots);
        SPMV_TRY_CUDA(cudaGetLastError());
        size_t temp_bytes = 0;
        SPMV_TRY_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, slots, *hack_off, nb + 1, stream));
        SPMV_TRY_CUDA(cudaMalloc(&temp, temp_bytes ? temp_bytes : 1));
        SPMV_TRY_CUDA(cub::DeviceScan::ExclusiveSum(temp, temp_bytes, slots, *hack_off, nb + 1, stream));
        if (narrow && nb > 0) {
            SPMV_TRY_CUDA(cudaMalloc(&d_fits, sizeof(int)));
            SPMV_TRY_CUDA(cudaMemcpyAsync(d_fits, &fits, sizeof(int), cudaMemcpyHostToDevice, stream));
            hll_narrow_check_kernel<<<blocks_for((long long)nb * kHack, 256), 256, 0, stream>>>(M, N, nb, row_ptr, col_idx,
                                                                                            *hack_off, d_fits);
            SPMV_TRY_CUDA(cudaGetLastError());
            SPMV_TRY_CUDA(cudaMemcpyAsync(&fits, d_fits, sizeof(int), cudaMemcpyDeviceToHost, stream));
        }
        host_off.resize((size_t)nb + 1);
        SPMV_TRY_CUDA(cudaMemcpyAsync(host_off.data(), *hack_off, ((size_t)nb + 1) * sizeof(long long), cudaMemcpyDeviceToHost,
                                      stream));
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
        return SPMV_B200_OK;
    };
    const int rc = body();
    cudaFree(slots);
    cudaFree(temp);
    cudaFree(d_fits);
    if (narrow) *narrow = fits != 0;
    *max_width = 0;
    for (int h = 0; rc == SPMV_B200_OK && h < nb; ++h) *max_width = std::max(*max_width, (int)((host_off[h + 1] - host_off[h]) / kHack));
    return rc;
}

int hll_fill(int M, int N, const int *row_ptr, const int *col_idx, const double *values, int num_hacks,
             const long long *hack_off, int *JA, uint16_t *JA16, double *AS, uint8_t *AC, const double *table, int K,
             bool masked, cudaStream_t stream) {
    if (num_hacks == 0) return SPMV_B200_OK;
    const unsigned int g = blocks_for((long long)num_hacks * kHack, 256);
    if (JA16) hll_fill_kernel<<<g, 256, 0, stream>>>(M, N, num_hacks, row_ptr, col_idx, values, hack_off, JA16, AS, AC, table, K, 0);
    else hll_fill_kernel<<<g, 256, 0, stream>>>(M, N, num_hacks, row_ptr, col_idx, values, hack_off, JA, AS, AC, table, K, masked ? kPadMark : 0);
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int hll_masked_launch(int hack_begin, int hack_end, int M, const long long *hack_off, const HllSegments &seg, const int *JA,
                      const uint16_t *JA16, long long slots, const double *AS, const uint8_t *AC, const double *table, int K,
                      int batch, bool offset_free, int accumulate, const double *x, double *y, cudaStream_t stream) {
    if (hack_end <= hack_begin) return SPMV_B200_OK;
    if (offset_free && seg.count <= 0) return fail(SPMV_B200_ERR_INVALID, "csr image: not regular enough for the offset-free form");
    const unsigned int g = blocks_for(hack_end - hack_begin, 8);
    auto launch = [&](auto accum, const auto *ja, const auto *as) {
        constexpr bool ACCUM = decltype(accum)::value;
        using I = std::remove_cv_t<std::remove_reference_t<decltype(*ja)>>;
        using S = std::remove_cv_t<std::remove_reference_t<decltype(*as)>>;
        const XPolicy keep = matrix_policy(ja, (size_t)slots * sizeof(I));
        const size_t smem = sizeof(S) == 1 ? (size_t)K * sizeof(double) : 0;  // the staged table of a coded image
        if (offset_free)
            return with_batch<5, 3, 4, 6, 7>(batch, [&](auto B) {
                return launch_x(hll_rowu_kernel<B, double, true, ACCUM, I, S>, g, 256, smem, stream, keep, hack_begin, hack_end, seg, ja, as, x, y, M, table, K);
            });
        return with_batch<4, 2, 3, 5, 6, 7>(batch, [&](auto B) {
            return launch_x(hll_row_kernel<B, double, true, ACCUM, I, S>, g, 256, smem, stream, keep, hack_begin, hack_end, hack_off, ja, as, x, y, M, table, K);
        });
    };
    auto values = [&](auto accum, const auto *ja) { return AC ? launch(accum, ja, AC) : launch(accum, ja, AS); };
    auto columns = [&](auto accum) { return JA16 ? values(accum, JA16) : values(accum, JA); };
    SPMV_TRY_CUDA(accumulate ? columns(std::true_type{}) : columns(std::false_type{}));
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}
}  // namespace spmv

// CSR -> HLL on the device (spmv_b200_hll_from_csr): the layout, then the column and value streams
static int hll_convert(const spmv_b200_csr *A, cudaStream_t stream, spmv_b200_hll *H) {
    H->M = A->M;
    H->N = A->N;
    const int nb = H->num_hacks = (A->M + kHack - 1) / kHack;
    SPMV_TRY(hll_layout(A->M, A->N, A->row_ptr, A->col_idx, stream, &H->hack_off, H->host_off, &H->max_width, nullptr));
    H->slots = H->host_off[nb];
    // reference layout keeps the last block short: its padded rows do not exist there
    const int last_rows = nb > 0 ? A->M - (nb - 1) * kHack : 0;
    H->ref_slots = H->slots;
    if (nb > 0) H->ref_slots -= ((H->host_off[nb] - H->host_off[nb - 1]) / kHack) * (kHack - last_rows);
    SPMV_TRY(hll_alloc_arena(H));
    SPMV_TRY(hll_fill(A->M, A->N, A->row_ptr, A->col_idx, A->values, nb, H->hack_off, H->JA, nullptr, H->AS, nullptr, nullptr, 0,
                      false, stream));
    SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
    return SPMV_B200_OK;
}

extern "C" {

int spmv_b200_hll_upload(const HLLMatrix *hll, int M, int N, spmv_b200_hll **out) {
    if (!out) return fail(SPMV_B200_ERR_INVALID, "hll_upload: out is NULL");
    *out = nullptr;
    if (!hll || hll->num_blocks < 0 || (hll->num_blocks > 0 && !hll->blocks) || M < 0 || N < 0)
        return fail(SPMV_B200_ERR_INVALID, "hll_upload: bad arguments");
    const int nb = hll->num_blocks;
    if (nb != (M + kHack - 1) / kHack) return fail(SPMV_B200_ERR_INVALID, "hll_upload: %d blocks do not cover %d rows", nb, M);
    std::vector<long long> off((size_t)nb + 1, 0);
    long long ref_slots = 0;
    int max_w = 0;
    for (int b = 0; b < nb; ++b) {
        const ELLPACKBlock &blk = hll->blocks[b];
        const int expect = (b == nb - 1) ? M - b * kHack : kHack;
        if (blk.M != expect || blk.MAXNZ < 0 || (blk.MAXNZ > 0 && (!blk.JA || !blk.AS)))
            return fail(SPMV_B200_ERR_INVALID, "hll_upload: block %d is malformed (M=%d, expected %d, MAXNZ=%d)", b, blk.M,
                        expect, blk.MAXNZ);
        off[b + 1] = off[b] + (long long)blk.MAXNZ * kHack;
        ref_slots += (long long)blk.MAXNZ * blk.M;
        max_w = std::max(max_w, blk.MAXNZ);
    }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
        return fail(SPMV_B200_ERR_NO_DEVICE, "hll_upload: no usable CUDA device; this library has no CPU fallback");
    spmv_b200_hll *H = new (std::nothrow) spmv_b200_hll();
    if (!H) return fail(SPMV_B200_ERR_NOMEM, "hll_upload: out of host memory");
    H->M = M;
    H->N = N;
    H->num_hacks = nb;
    H->max_width = max_w;
    H->slots = off[nb];
    H->ref_slots = ref_slots;
    H->host_off = off;
    // row-major host blocks -> column-major, 32-row padded staging image
    const size_t n = (size_t)std::max<long long>(H->slots, 1);
    int *ja = static_cast<int *>(std::calloc(n, sizeof(int)));
    double *as = static_cast<double *>(std::calloc(n, sizeof(double)));
    int rc = (ja && as) ? SPMV_B200_OK : fail(SPMV_B200_ERR_NOMEM, "hll_upload: out of host memory");
    if (rc == SPMV_B200_OK) {
#pragma omp parallel for schedule(dynamic, 256)
        for (int b = 0; b < nb; ++b) {
            const ELLPACKBlock &blk = hll->blocks[b];
            const int w = blk.MAXNZ;
            for (int r = 0; r < blk.M; ++r)
                for (int j = 0; j < w; ++j) {
                    ja[off[b] + (long long)j * kHack + r] = blk.JA[(size_t)r * w + j];
                    as[off[b] + (long long)j * kHack + r] = blk.AS[(size_t)r * w + j];
                }
        }
        auto dev = [&]() -> int {
            SPMV_TRY_CUDA(cudaMalloc(&H->hack_off, ((size_t)nb + 1) * sizeof(long long)));
            SPMV_TRY(hll_alloc_arena(H));
            SPMV_TRY_CUDA(cudaMemcpy(H->hack_off, off.data(), ((size_t)nb + 1) * sizeof(long long), cudaMemcpyHostToDevice));
            if (H->slots) {
                SPMV_TRY_CUDA(cudaMemcpy(H->JA, ja, (size_t)H->slots * sizeof(int), cudaMemcpyHostToDevice));
                SPMV_TRY_CUDA(cudaMemcpy(H->AS, as, (size_t)H->slots * sizeof(double), cudaMemcpyHostToDevice));
            }
            return SPMV_B200_OK;
        };
        rc = dev();
        if (rc == SPMV_B200_OK) rc = stream_plan_hll(H, nullptr);
        if (rc == SPMV_B200_OK) hll_pick_row_batch(H, nullptr);
    }
    std::free(ja);
    std::free(as);
    if (rc != SPMV_B200_OK) {
        spmv_b200_hll_free(H);
        return rc;
    }
    *out = H;
    return SPMV_B200_OK;
}

int spmv_b200_hll_from_csr(const spmv_b200_csr *A, void *stream_, spmv_b200_hll **out) {
    if (!out) return fail(SPMV_B200_ERR_INVALID, "hll_from_csr: out is NULL");
    *out = nullptr;
    if (!A) return fail(SPMV_B200_ERR_INVALID, "hll_from_csr: NULL matrix");
    cudaStream_t stream = as_stream(stream_);
    spmv_b200_hll *H = new (std::nothrow) spmv_b200_hll();
    if (!H) return fail(SPMV_B200_ERR_NOMEM, "hll_from_csr: out of host memory");
    int rc = hll_convert(A, stream, H);
    if (rc == SPMV_B200_OK) rc = stream_plan_hll(H, stream);
    if (rc != SPMV_B200_OK) {
        spmv_b200_hll_free(H);
        return rc;
    }
    hll_pick_row_batch(H, stream);
    *out = H;
    return SPMV_B200_OK;
}

int spmv_b200_hll_info(const spmv_b200_hll *H, spmv_b200_hll_info_t *info) {
    if (!H || !info) return fail(SPMV_B200_ERR_INVALID, "hll_info: NULL argument");
    info->M = H->M;
    info->N = H->N;
    info->num_hacks = H->num_hacks;
    info->max_maxnz = H->max_width;
    info->slots = H->slots;
    info->nnz_reference_slots = H->ref_slots;
    info->algorithmic_bytes = H->slots * 12 + 8LL * ((long long)H->num_hacks + 1) + 8LL * H->M + 8LL * H->N;
    info->auto_kernel = (int)hll_resolve(H);
    info->row_batch = H->row_batch;
    info->fused_batch = H->fused_batch;
    info->flat_batch = H->flat_batch;
    info->flat_chunks = 1;
    return SPMV_B200_OK;
}

int spmv_b200_hll_device_arrays(const spmv_b200_hll *H, const long long **d_hack_off, const int **d_JA, const double **d_AS) {
    if (!H) return fail(SPMV_B200_ERR_INVALID, "hll_device_arrays: NULL matrix");
    if (d_hack_off) *d_hack_off = H->hack_off;
    if (d_JA) *d_JA = H->JA;
    if (d_AS) *d_AS = H->AS;
    return SPMV_B200_OK;
}

int spmv_b200_hll_download(const spmv_b200_hll *H, HLLMatrix *out) {
    if (!H || !out) return fail(SPMV_B200_ERR_INVALID, "hll_download: NULL argument");
    const int nb = H->num_hacks;
    out->num_blocks = nb;
    out->blocks = static_cast<ELLPACKBlock *>(std::calloc((size_t)std::max(nb, 1), sizeof(ELLPACKBlock)));
    const size_t n = (size_t)std::max<long long>(H->slots, 1);
    int *ja = static_cast<int *>(std::malloc(n * sizeof(int)));
    double *as = static_cast<double *>(std::malloc(n * sizeof(double)));
    if (!out->blocks || !ja || !as) {
        std::free(ja);
        std::free(as);
        std::free(out->blocks);
        out->blocks = nullptr;
        out->num_blocks = 0;
        return fail(SPMV_B200_ERR_NOMEM, "hll_download: out of host memory");
    }
    if (H->slots) {
        cudaError_t e1 = cudaMemcpy(ja, H->JA, (size_t)H->slots * sizeof(int), cudaMemcpyDeviceToHost);
        cudaError_t e2 = cudaMemcpy(as, H->AS, (size_t)H->slots * sizeof(double), cudaMemcpyDeviceToHost);
        if (e1 != cudaSuccess || e2 != cudaSuccess) {
            std::free(ja);
            std::free(as);
            std::free(out->blocks);
            out->blocks = nullptr;
            out->num_blocks = 0;
            return fail(SPMV_B200_ERR_CUDA, "hll_download: D2H copy failed");
        }
    }
    bool oom = false;
    for (int b = 0; b < nb; ++b) {
        ELLPACKBlock &blk = out->blocks[b];
        const int w = (int)((H->host_off[b + 1] - H->host_off[b]) / kHack);
        blk.M = (b == nb - 1) ? H->M - b * kHack : kHack;
        blk.N = H->N;
        blk.MAXNZ = w;
        blk.JA = nullptr;
        blk.AS = nullptr;
        if (w == 0) continue;
        blk.JA = static_cast<int *>(std::malloc((size_t)w * blk.M * sizeof(int)));
        blk.AS = static_cast<double *>(std::malloc((size_t)w * blk.M * sizeof(double)));
        if (!blk.JA || !blk.AS) {
            oom = true;
            break;
        }
        for (int r = 0; r < blk.M; ++r)
            for (int j = 0; j < w; ++j) {
                blk.JA[(size_t)r * w + j] = ja[H->host_off[b] + (long long)j * kHack + r];
                blk.AS[(size_t)r * w + j] = as[H->host_off[b] + (long long)j * kHack + r];
            }
    }
    std::free(ja);
    std::free(as);
    if (oom) {
        for (int b = 0; b < nb; ++b) {
            std::free(out->blocks[b].JA);
            std::free(out->blocks[b].AS);
        }
        std::free(out->blocks);
        out->blocks = nullptr;
        out->num_blocks = 0;
        return fail(SPMV_B200_ERR_NOMEM, "hll_download: out of host memory");
    }
    return SPMV_B200_OK;
}


int spmv_b200_hll_spmv(const spmv_b200_hll *H, const double *d_x, double *d_y, void *stream) {
    if (!H || !d_y || (H->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv: NULL argument");
    const HllPath path = hll_resolve(H);
    return hll_launch_window(H, path, 0, path == kHllStream ? H->num_tiles : H->num_hacks, d_x, d_y, as_stream(stream));
}

int spmv_b200_hll_spmv_stream(const spmv_b200_hll *H, const double *d_x, double *d_y, void *stream) {
    if (!H || !d_y || (H->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_stream: NULL argument");
    return stream_launch_hll(H, d_x, d_y, as_stream(stream));
}

int spmv_b200_hll_spmv_rows(const spmv_b200_hll *H, const double *d_x, double *d_y, void *stream) {
    if (!H || !d_y || (H->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_rows: NULL argument");
    return hll_launch_rows(H, 0, H->num_hacks, d_x, d_y, as_stream(stream));
}

int spmv_b200_hll_spmv_slice(const spmv_b200_hll *H, const double *d_x, double *d_y, void *stream) {
    if (!H || !d_y || (H->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_slice: NULL argument");
    return hll_launch(H, 0, H->num_hacks, d_x, d_y, as_stream(stream));
}

int spmv_b200_hll_partials_count(const spmv_b200_hll *H) { return H ? hll_fused_grid(H) : 0; }

int spmv_b200_hll_spmv_fused(const spmv_b200_hll *H, const double *d_x, double *d_y, const double *d_prev_sumsq,
                             double *d_partials, const spmv_b200_peers_t *peers, void *stream) {
    if (!H || !d_y || (H->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_fused: NULL argument");
    SPMV_TRY(check_peers(peers, H->M, "hll_spmv_fused"));
    if (H->M == 0) return SPMV_B200_OK;
    Epilogue ep;
    ep.prev_sumsq = d_prev_sumsq;
    ep.partials = d_partials;
    ep.partials_total = hll_fused_grid(H);
    if (peers) ep.peers = *peers;
    if (peers && env_int("SPMV_B200_FUSED_BOUNDARY_FIRST", 0)) SPMV_TRY(boundary_first_order(ep.peers, H->M, ep.order));
    return hll_launch_fused(H, d_x, d_y, ep, as_stream(stream));
}

int spmv_b200_hll_flat_partials_count(const spmv_b200_hll *H) {
    if (!H) return 0;
    return hll_flat_grid(H->M);
}

int spmv_b200_hll_spmv_fused_flat(const spmv_b200_hll *H, const double *d_x, double *d_y, const double *d_inv_norm,
                                  double *d_partials, const spmv_b200_peers_t *peers, void *stream) {
    if (!H || !d_y || (H->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_fused_flat: NULL argument");
    SPMV_TRY(check_peers(peers, H->M, "hll_spmv_fused_flat"));
    if (H->M == 0) return SPMV_B200_OK;
    Epilogue ep;
    ep.inv_norm = d_inv_norm;
    ep.partials = d_partials;
    ep.partials_total = hll_flat_grid(H->M);
    if (peers) ep.peers = *peers;
    return hll_launch_fused_flat(H, d_x, d_y, ep, as_stream(stream), env_int("SPMV_B200_HLL_FLAT_BATCH", H->flat_batch));
}

int spmv_b200_hll_spmv_fused_mail(const spmv_b200_hll *H, const double *d_x, double *d_y, double *d_partials,
                                  const spmv_b200_peers_t *peers, const spmv_b200_mail_t *mail, void *stream) {
    if (!H || !d_y || !d_partials || !mail || (H->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_fused_mail: NULL argument");
    if (H->M == 0) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_fused_mail: a rank without rows cannot take part in the exchange");
    SPMV_TRY(check_peers(peers, H->M, "hll_spmv_fused_mail"));
    if (mail->world < 1 || mail->world > SPMV_B200_MAX_RANKS || mail->rank < 0 || mail->rank >= mail->world || !mail->counter ||
        !mail->status)
        return fail(SPMV_B200_ERR_INVALID, "hll_spmv_fused_mail: bad mailbox description (world %d, rank %d)", mail->world, mail->rank);
    for (int r = 0; r < mail->world; ++r)
        if (!mail->box[r]) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_fused_mail: mailbox of rank %d is NULL", r);
    Epilogue ep;
    ep.partials = d_partials;
    ep.partials_total = hll_fused_grid(H);
    if (peers) ep.peers = *peers;
    ep.mail = *mail;
    if (peers && env_int("SPMV_B200_FUSED_BOUNDARY_FIRST", 0)) SPMV_TRY(boundary_first_order(ep.peers, H->M, ep.order));
    return hll_launch_fused(H, d_x, d_y, ep, as_stream(stream));
}

int spmv_b200_hll_spmv_hacks(const spmv_b200_hll *H, int hack_begin, int hack_end, const double *d_x, double *d_y,
                             void *stream) {
    if (!H || !d_y || !d_x) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_hacks: NULL argument");
    if (hack_begin < 0 || hack_end > H->num_hacks || hack_begin > hack_end)
        return fail(SPMV_B200_ERR_INVALID, "hll_spmv_hacks: range [%d,%d) outside [0,%d)", hack_begin, hack_end, H->num_hacks);
    return hll_launch(H, hack_begin, hack_end, d_x, d_y, as_stream(stream));
}

// ---- fp32 storage, fp64 arithmetic --------------------------------------------------------------------------------
__global__ void hll_to_f32_kernel(const double *__restrict__ in, float *__restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)in[i];
}

int spmv_b200_hll_enable_f32(spmv_b200_hll *H, void *stream) {
    if (!H) return fail(SPMV_B200_ERR_INVALID, "hll_enable_f32: NULL matrix");
    if (H->AS32) return SPMV_B200_OK;
    const size_t n = (size_t)std::max<long long>(H->slots, 32);
    SPMV_TRY_CUDA(cudaMalloc(&H->AS32, n * sizeof(float)));
    SPMV_TRY_CUDA(cudaMemsetAsync(H->AS32, 0, n * sizeof(float), as_stream(stream)));
    if (H->slots) {
        hll_to_f32_kernel<<<blocks_for(H->slots, 256), 256, 0, as_stream(stream)>>>(H->AS, H->AS32, H->slots);
        SPMV_TRY_CUDA(cudaGetLastError());
    }
    H->row_batch32 = H->row_batch;
    if (H->max_width <= kRowKernelMaxLen && H->slots >= (1 << 22) && env_int("SPMV_B200_AUTOTUNE", 1) &&
        env_int("SPMV_B200_HLL_ROW_BATCH", 0) == 0) {
        // candidates: one hack per warp with batch 2..7, and the forms of hll_rowm_kernel (ids >= 16); all give the same
        // bits.  SPMV_B200_ROW_MULTI_TUNE=0 keeps the one-hack forms only.
        int ids[12 + kNumHllRowmVariants], n = 0, fallback = 0;
        for (int batch = 2; batch <= 7; ++batch) {
            if (batch == H->row_batch) fallback = n;
            ids[n++] = batch;
        }
        if (env_int("SPMV_B200_ROW_MULTI_TUNE", 1)) {
            for (int v = 0; v < kNumHllRowmVariants; ++v) ids[n++] = 16 + v;
            if (H->segments.count > 0)  // regular image: the forms without the hack_off round trip
                for (int batch = 4; batch <= 7; ++batch) ids[n++] = 64 + batch;
        }
        const int pick = tune_candidates(H->M, H->N, n, fallback, as_stream(stream), [&](int i, double *x, double *y) {
            return hll_launch_rows_t<float>(H, H->AS32, 0, H->num_hacks, reinterpret_cast<const float *>(x),
                                            reinterpret_cast<float *>(y), as_stream(stream), ids[i]);
        });
        H->row_batch32 = ids[pick];
    }
    return SPMV_B200_OK;
}

int spmv_b200_hll_spmv_f32(const spmv_b200_hll *H, const float *d_x, float *d_y, void *stream) {
    if (!H || !d_y || (H->N > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_f32: NULL argument");
    if (!H->AS32) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_f32: call spmv_b200_hll_enable_f32 first");
    if (H->num_hacks == 0) return SPMV_B200_OK;
    if (H->max_width <= kRowKernelMaxLen) return hll_launch_rows_t<float>(H, H->AS32, 0, H->num_hacks, d_x, d_y, as_stream(stream));
    SPMV_TRY_CUDA(launch_x(hll_slice_kernel<float>, blocks_for(H->num_hacks, kHllWarps), kHllThreads, 0, as_stream(stream),
                           x_policy(d_x, (size_t)H->N * sizeof(float)), 0, H->num_hacks, H->hack_off, H->JA, H->AS32, d_x, d_y,
                           H->M));
    return SPMV_B200_OK;
}

int spmv_b200_hll_row_form_f32(const spmv_b200_hll *H) { return H && H->AS32 ? H->row_batch32 : 0; }
int spmv_b200_hll_row_form(const spmv_b200_hll *H) { return !H ? 0 : (H->row_form > 0 ? H->row_form : H->row_batch); }

int spmv_b200_hll_spmv_host_f32(spmv_b200_hll *H, const float *x, float *y) {
    if (!H || (H->M > 0 && !y) || (H->N > 0 && H->slots > 0 && !x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_host_f32: NULL argument");
    if (H->M == 0) return SPMV_B200_OK;
    SPMV_TRY(spmv_b200_hll_enable_f32(H, nullptr));
    if (!H->stage_x) SPMV_TRY_CUDA(cudaMalloc(&H->stage_x, std::max<size_t>(H->N, 1) * sizeof(double)));
    if (!H->stage_y) SPMV_TRY_CUDA(cudaMalloc(&H->stage_y, std::max<size_t>(H->M, 1) * sizeof(double)));
    float *dx = reinterpret_cast<float *>(H->stage_x), *dy = reinterpret_cast<float *>(H->stage_y);
    if (H->N && x) SPMV_TRY_CUDA(cudaMemcpyAsync(dx, x, (size_t)H->N * sizeof(float), cudaMemcpyHostToDevice, nullptr));
    SPMV_TRY(spmv_b200_hll_spmv_f32(H, dx, dy, nullptr));
    SPMV_TRY_CUDA(cudaMemcpyAsync(y, dy, (size_t)H->M * sizeof(float), cudaMemcpyDeviceToHost, nullptr));
    SPMV_TRY_CUDA(cudaStreamSynchronize(nullptr));
    return SPMV_B200_OK;
}

void spmv_b200_hll_free(spmv_b200_hll *H) {
    if (!H) return;
    cudaFree(H->AS32);
    cudaFree(H->tiles);
    cudaFree(H->hack_off);
    cudaFree(H->JA);
    cudaFree(H->AS);
    cudaFree(H->stage_x);
    cudaFree(H->stage_y);
    host_pipe_free(H->pipe);
    host_pipe_free(H->spmm_pipe);
    delete H;
}

}  // extern "C"
