// synth.cu -- device-side generators for the BASELINE.json synthetic matrices (SURVEY.md section
// 8(d): C2 2-D 5-point Laplacian, C3 uniform 32 nnz/row with stratified columns, C5 3-D 7-point
// Laplacian), the dense-vector helpers of the iterated product, and the library bookkeeping
// (last error, device queries).  The reference has no generator for these shapes (its
// src/matrix_generator.py writes 10x10 files); the numpy twins in
// sparsematrixvectormultiplication_b200/synth.py produce bit-identical arrays on the CPU so the
// oracle can check the GPU results.
#include <algorithm>
#include <cstring>

#include "common.cuh"
#include "handles.cuh"

// csr.cu
extern "C" int spmv_b200_csr_adopt_device_(int M, int N, long long nnz, int *d_row_ptr, int *d_col_idx,
                                           double *d_values, void *stream, spmv_b200_csr **out);

namespace spmv {

// ---- error plumbing -----------------------------------------------------------------------------
static thread_local char g_error[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof g_error, fmt, ap);
    va_end(ap);
}

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof g_error, fmt, ap);
    va_end(ap);
    return code;
}

// ---- closed-form row offsets -------------------------------------------------------------------
// Number of nonzeros in rows [0, r) of the n x n 5-point Laplacian (row r = i*n + j).
__host__ __device__ inline long long lap2d_offset(long long n, long long r) {
    const long long top = r < n ? r : n;                              // rows with i == 0
    const long long bottom = r > (n - 1) * n ? r - (n - 1) * n : 0;   // rows with i == n-1
    const long long left = (r + n - 1) / n;                           // rows with j == 0
    const long long right = r / n;                                    // rows with j == n-1
    return 5 * r - top - bottom - left - right;
}

// Rows [0, r) of the n^3 7-point Laplacian (row r = (i*n + j)*n + k).
__host__ __device__ inline long long lap3d_offset(long long n, long long r) {
    const long long n2 = n * n;
    const long long i = r / n2, j = (r / n) % n, k = r % n;
    const long long i_lo = r < n2 ? r : n2;
    const long long i_hi = r > (n - 1) * n2 ? r - (n - 1) * n2 : 0;
    const long long j_lo = i * n + (j > 0 ? n : k);
    const long long j_hi = i * n + (j == n - 1 ? k : 0);
    const long long k_lo = (r + n - 1) / n;
    const long long k_hi = r / n;
    return 7 * r - i_lo - i_hi - j_lo - j_hi - k_lo - k_hi;
}

__host__ __device__ inline long long synth_offset(int kind, long long p0, int p2, long long r) {
    switch (kind) {
        case SPMV_B200_SYNTH_LAP2D: return lap2d_offset(p0, r);
        case SPMV_B200_SYNTH_LAP3D: return lap3d_offset(p0, r);
        default: return (long long)p2 * r;
    }
}

// ---- fill kernels ------------------------------------------------------------------------------
__global__ void lap2d_fill_kernel(long long n, long long row_begin, long long rows, int *__restrict__ row_ptr,
                                  int *__restrict__ col_idx, double *__restrict__ values) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t > rows) return;
    const long long r = row_begin + t;
    const long long base = lap2d_offset(n, row_begin);
    long long o = lap2d_offset(n, r) - base;
    row_ptr[t] = (int)o;
    if (t == rows) return;
    const long long i = r / n, j = r % n;
    if (i > 0) { col_idx[o] = (int)(r - n); values[o++] = -1.0; }
    if (j > 0) { col_idx[o] = (int)(r - 1); values[o++] = -1.0; }
    col_idx[o] = (int)r; values[o++] = 4.0;
    if (j < n - 1) { col_idx[o] = (int)(r + 1); values[o++] = -1.0; }
    if (i < n - 1) { col_idx[o] = (int)(r + n); values[o++] = -1.0; }
}

__global__ void lap3d_fill_kernel(long long n, long long row_begin, long long rows, int *__restrict__ row_ptr,
                                  int *__restrict__ col_idx, double *__restrict__ values) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t > rows) return;
    const long long r = row_begin + t;
    const long long base = lap3d_offset(n, row_begin);
    long long o = lap3d_offset(n, r) - base;
    row_ptr[t] = (int)o;
    if (t == rows) return;
    const long long n2 = n * n;
    const long long i = r / n2, j = (r / n) % n, k = r % n;
    if (i > 0) { col_idx[o] = (int)(r - n2); values[o++] = -1.0; }
    if (j > 0) { col_idx[o] = (int)(r - n); values[o++] = -1.0; }
    if (k > 0) { col_idx[o] = (int)(r - 1); values[o++] = -1.0; }
    col_idx[o] = (int)r; values[o++] = 6.0;
    if (k < n - 1) { col_idx[o] = (int)(r + 1); values[o++] = -1.0; }
    if (j < n - 1) { col_idx[o] = (int)(r + n); values[o++] = -1.0; }
    if (i < n - 1) { col_idx[o] = (int)(r + n2); values[o++] = -1.0; }
}

// Exactly k nonzeros per row; column of entry e lies in stratum e: e*stride + hash % stride, so a
// row is sorted and duplicate free by construction.  One thread per entry (coalesced stores).
__global__ void uniform_fill_kernel(long long row_begin, long long rows, long long ncols, int k,
                                    unsigned long long seed, int *__restrict__ row_ptr, int *__restrict__ col_idx,
                                    double *__restrict__ values) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t <= rows) row_ptr[t] = (int)(t * k);
    if (t >= rows * k) return;
    const unsigned long long r = (unsigned long long)(row_begin + t / k), e = (unsigned long long)(t % k);
    const unsigned long long stride = (unsigned long long)(ncols / k);
    col_idx[t] = (int)(e * stride + hash3(seed, r, e) % stride);
    values[t] = unit_interval(hash3(seed + 0x5851F42D4C957F2DULL, r, e));
}

__global__ void vector_hash_kernel(double *__restrict__ x, long long n, unsigned long long seed) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = unit_interval(hash3(seed, (unsigned long long)i, 0x7Eull));
}

__global__ void vector_fill_kernel(double *__restrict__ v, long long n, double value) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = value;
}

// ---- deterministic sum of squares ----------------------------------------------------------------
constexpr int kSumsqCtas = 1184;  // 148 SMs x 8
constexpr int kSumsqThreads = 256;

__device__ __forceinline__ double block_sum(double v, double *scratch) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    double total = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) total += scratch[w];
    return total;  // valid in thread 0
}

__global__ void __launch_bounds__(kSumsqThreads) sumsq_stage1_kernel(const double *__restrict__ v, long long n,
                                                                     double *__restrict__ ws) {
    __shared__ double scratch[kSumsqThreads / 32];
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * kSumsqThreads + threadIdx.x; i < n; i += (long long)kSumsqCtas * kSumsqThreads) {
        const double a = v[i];
        acc = fma(a, a, acc);
    }
    const double total = block_sum(acc, scratch);
    if (threadIdx.x == 0) ws[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kSumsqThreads) sumsq_stage2_kernel(const double *__restrict__ ws, double *__restrict__ out) {
    __shared__ double scratch[kSumsqThreads / 32];
    double acc = 0.0;
    for (int i = threadIdx.x; i < kSumsqCtas; i += kSumsqThreads) acc += ws[i];
    const double total = block_sum(acc, scratch);
    if (threadIdx.x == 0) *out = total;
}

__global__ void __launch_bounds__(kSumsqThreads) sum_small_kernel(const double *__restrict__ in, int n, double *__restrict__ out) {
    __shared__ double scratch[kSumsqThreads / 32];
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += kSumsqThreads) acc += in[i];
    const double total = block_sum(acc, scratch);
    if (threadIdx.x == 0) *out = total;
}

__global__ void scale_by_inv_norm_kernel(double *__restrict__ dst, const double *__restrict__ src, long long n,
                                         const double *__restrict__ sumsq) {
    const double norm = sqrt(*sumsq);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i] / norm;
}

// dst_p[i] = src[i] for every peer p: the all-gather of a slice written against peer memory (NVLink stores).  A
// persistent grid of one CTA per SM is all the links need; 256-bit loads, 256-bit peer stores.  The source and every
// target sit at the SAME offset of equally aligned buffers (a row range of the replicas of x), so one scalar head of
// up to three elements brings all of them onto a 32-byte boundary; targets aligned differently take the scalar path.
struct PushTargets {
    int count;
    int vector_ok;
    double *dst[SPMV_B200_MAX_PEERS];
};

template <int UNROLL, int WIDTH>
__global__ void __launch_bounds__(512)
vec_push_kernel(const double *__restrict__ src, long long n, const __grid_constant__ PushTargets t) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    if (!t.vector_ok) {
        for (long long i = tid; i < n; i += stride) {
            const double v = __ldg(src + i);
            for (int p = 0; p < t.count; ++p) t.dst[p][i] = v;
        }
        return;
    }
    const long long head = min(n, (long long)(((32 - (reinterpret_cast<uintptr_t>(src) & 31)) & 31) >> 3));
    const long long quads = (n - head) >> 2;
    if constexpr (WIDTH == 32) {
        // a lane moves whole 32-byte sectors (LDG.256 / STG.256): a warp instruction covers 1 KB of contiguous peer memory
        for (long long q0 = tid; q0 < quads; q0 += UNROLL * stride) {
            double v[UNROLL][4];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const long long q = q0 + u * stride;
                if (q < quads)
                    asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                                 : "=d"(v[u][0]), "=d"(v[u][1]), "=d"(v[u][2]), "=d"(v[u][3]) : "l"(src + head + 4 * q));
            }
            for (int p = 0; p < t.count; ++p) {
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) {
                    const long long q = q0 + u * stride;
                    if (q < quads)
                        asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(t.dst[p] + head + 4 * q), "d"(v[u][0]), "d"(v[u][1]),
                                     "d"(v[u][2]), "d"(v[u][3]) : "memory");
                }
            }
        }
    } else {
        // a lane moves 16 bytes, a warp instruction 512 contiguous bytes (the classic coalesced pattern)
        const long long pairs = quads * 2;
        const double2 *s2 = reinterpret_cast<const double2 *>(src + head);
        for (long long i0 = tid; i0 < pairs; i0 += UNROLL * stride) {
            double2 v[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const long long i = i0 + u * stride;
                if (i < pairs)
                    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(v[u].x), "=d"(v[u].y) : "l"(s2 + i));
            }
            for (int p = 0; p < t.count; ++p) {
                double2 *d2 = reinterpret_cast<double2 *>(t.dst[p] + head);
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) {
                    const long long i = i0 + u * stride;
                    if (i < pairs) d2[i] = v[u];
                }
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < 8) {  // up to three elements at either end
        const long long tail = head + 4 * quads;
        const long long i = threadIdx.x < 4 ? threadIdx.x : tail + (threadIdx.x - 4);
        const bool mine = threadIdx.x < 4 ? i < head : i < n;
        if (mine) {
            const double v = src[i];
            for (int p = 0; p < t.count; ++p) t.dst[p][i] = v;
        }
    }
}

}  // namespace spmv

using namespace spmv;

extern "C" {

const char *spmv_b200_last_error(void) { return g_error; }
void spmv_b200_clear_error(void) { g_error[0] = '\0'; }

int spmv_b200_version(void) { return 108; }  // 101: spmv_b200_csr_spmm / spmv_b200_hll_spmm; 102: spmv_b200_csr_set_image;
                                              // 103: the narrow private image, spmv_b200_csr_info_t::image_index_bytes;
                                              // 104: the coded private image (set_image mode 2), image_value_bytes;
                                              // 105: spmv_b200_csr_spmm_f32 / spmv_b200_hll_spmm_f32;
                                              // 106: the pattern form of the private image (set_image mode 3), image_patterns;
                                              // 107: image_windows (the tiled kernel of the pattern form);
                                              // 108: spmv_b200_{csr,hll}_spmm_host[_f32]

int spmv_b200_device_count(int *count) {
    if (!count) return fail(SPMV_B200_ERR_INVALID, "device_count: NULL argument");
    *count = 0;
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess) {
        *count = 0;
        return fail(SPMV_B200_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    return SPMV_B200_OK;
}

int spmv_b200_device_info(char *name, int len, int *sm_count, long long *l2_bytes, long long *mem_bytes) {
    int dev = 0;
    SPMV_TRY_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    SPMV_TRY_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (name && len > 0) {
        strncpy(name, prop.name, (size_t)len - 1);
        name[len - 1] = '\0';
    }
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (l2_bytes) *l2_bytes = prop.l2CacheSize;
    if (mem_bytes) *mem_bytes = (long long)prop.totalGlobalMem;
    return SPMV_B200_OK;
}

long long spmv_b200_synth_row_offset(int kind, long long p0, long long p1, int p2, long long row) {
    (void)p1;
    return synth_offset(kind, p0, p2, row);
}

int spmv_b200_synth_csr(int kind, long long p0, long long p1, int p2, unsigned long long seed, long long row_begin,
                        long long row_end, void *stream_, spmv_b200_csr **out) {
    if (!out) return fail(SPMV_B200_ERR_INVALID, "synth_csr: out is NULL");
    *out = nullptr;
    long long M_global, N_global;
    switch (kind) {
        case SPMV_B200_SYNTH_LAP2D: M_global = N_global = p0 * p0; break;
        case SPMV_B200_SYNTH_LAP3D: M_global = N_global = p0 * p0 * p0; break;
        case SPMV_B200_SYNTH_UNIFORM:
            M_global = p0;
            N_global = p1;
            if (p2 <= 0 || p1 < p2) return fail(SPMV_B200_ERR_INVALID, "synth_csr: uniform needs 0 < nnz_per_row <= N");
            break;
        default: return fail(SPMV_B200_ERR_INVALID, "synth_csr: unknown kind %d", kind);
    }
    if (p0 <= 0 || M_global > 0x7fffffffLL || N_global > 0x7fffffffLL)
        return fail(SPMV_B200_ERR_INVALID, "synth_csr: dimensions out of int32 range");
    if (row_begin < 0 || row_end > M_global || row_begin > row_end)
        return fail(SPMV_B200_ERR_INVALID, "synth_csr: row range [%lld,%lld) outside [0,%lld)", row_begin, row_end, M_global);
    const long long rows = row_end - row_begin;
    const long long nnz = synth_offset(kind, p0, p2, row_end) - synth_offset(kind, p0, p2, row_begin);
    if (nnz > 0x7fffffffLL) return fail(SPMV_B200_ERR_INVALID, "synth_csr: %lld nonzeros exceed int32 indexing", nnz);
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
        return fail(SPMV_B200_ERR_NO_DEVICE, "synth_csr: no usable CUDA device; this library has no CPU fallback");
    cudaStream_t stream = as_stream(stream_);
    int *row_ptr = nullptr, *col_idx = nullptr;
    double *values = nullptr;
    const size_t padded = std::max<size_t>(((size_t)nnz + 3) & ~(size_t)3, 4);
    auto body = [&]() -> int {
        SPMV_TRY_CUDA(cudaMalloc(&row_ptr, ((size_t)rows + 1) * sizeof(int)));
        SPMV_TRY_CUDA(cudaMalloc(&col_idx, padded * sizeof(int)));
        SPMV_TRY_CUDA(cudaMalloc(&values, padded * sizeof(double)));
        SPMV_TRY_CUDA(cudaMemsetAsync(col_idx + (padded - 4), 0, 4 * sizeof(int), stream));
        SPMV_TRY_CUDA(cudaMemsetAsync(values + (padded - 4), 0, 4 * sizeof(double), stream));
        if (kind == SPMV_B200_SYNTH_LAP2D)
            lap2d_fill_kernel<<<blocks_for(rows + 1, 256), 256, 0, stream>>>(p0, row_begin, rows, row_ptr, col_idx, values);
        else if (kind == SPMV_B200_SYNTH_LAP3D)
            lap3d_fill_kernel<<<blocks_for(rows + 1, 256), 256, 0, stream>>>(p0, row_begin, rows, row_ptr, col_idx, values);
        else
            uniform_fill_kernel<<<blocks_for(std::max(rows * p2, rows + 1), 256), 256, 0, stream>>>(
                row_begin, rows, p1, p2, seed, row_ptr, col_idx, values);
        SPMV_TRY_CUDA(cudaGetLastError());
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
        return SPMV_B200_OK;
    };
    int rc = body();
    if (rc == SPMV_B200_OK)
        rc = spmv_b200_csr_adopt_device_((int)rows, (int)N_global, nnz, row_ptr, col_idx, values, stream_, out);
    if (rc != SPMV_B200_OK) {
        cudaFree(row_ptr);
        cudaFree(col_idx);
        cudaFree(values);
    }
    return rc;
}

int spmv_b200_synth_vector(double *d_x, long long n, unsigned long long seed, void *stream) {
    if (n < 0 || (n > 0 && !d_x)) return fail(SPMV_B200_ERR_INVALID, "synth_vector: bad arguments");
    if (n == 0) return SPMV_B200_OK;
    vector_hash_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(d_x, n, seed);
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int spmv_b200_vec_fill(double *d_v, long long n, double value, void *stream) {
    if (n < 0 || (n > 0 && !d_v)) return fail(SPMV_B200_ERR_INVALID, "vec_fill: bad arguments");
    if (n == 0) return SPMV_B200_OK;
    vector_fill_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(d_v, n, value);
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int spmv_b200_vec_ws_doubles(void) { return kSumsqCtas; }

int spmv_b200_vec_sumsq(const double *d_v, long long n, double *d_ws, double *d_out, void *stream) {
    if (n < 0 || (n > 0 && !d_v) || !d_ws || !d_out) return fail(SPMV_B200_ERR_INVALID, "vec_sumsq: bad arguments");
    sumsq_stage1_kernel<<<kSumsqCtas, kSumsqThreads, 0, as_stream(stream)>>>(d_v, n, d_ws);
    SPMV_TRY_CUDA(cudaGetLastError());
    sumsq_stage2_kernel<<<1, kSumsqThreads, 0, as_stream(stream)>>>(d_ws, d_out);
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int spmv_b200_vec_sum(const double *d_in, int n, double *d_out, void *stream) {
    if (n < 0 || (n > 0 && !d_in) || !d_out) return fail(SPMV_B200_ERR_INVALID, "vec_sum: bad arguments");
    sum_small_kernel<<<1, kSumsqThreads, 0, as_stream(stream)>>>(d_in, n, d_out);
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int spmv_b200_ipc_alloc(long long bytes, void **d_ptr, unsigned char handle[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (bytes <= 0 || !d_ptr || !handle) return fail(SPMV_B200_ERR_INVALID, "ipc_alloc: bad arguments");
    *d_ptr = nullptr;
    // cudaMalloc packs small requests into shared 2 MiB blocks and an IPC handle maps the whole block from its base:
    // round up so that the buffer IS the block and the peer's pointer is the buffer's first byte
    const size_t granule = (size_t)2 << 20;
    SPMV_TRY_CUDA(cudaMalloc(d_ptr, ((size_t)bytes + granule - 1) / granule * granule));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, *d_ptr);
    if (e != cudaSuccess) {
        cudaFree(*d_ptr);
        *d_ptr = nullptr;
        return fail(SPMV_B200_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    }
    memcpy(handle, &h, 64);
    return SPMV_B200_OK;
}

int spmv_b200_ipc_open(const unsigned char handle[64], void **d_peer_ptr) {
    if (!handle || !d_peer_ptr) return fail(SPMV_B200_ERR_INVALID, "ipc_open: bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    SPMV_TRY_CUDA(cudaIpcOpenMemHandle(d_peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return SPMV_B200_OK;
}

int spmv_b200_ipc_close(void *d_peer_ptr) {
    if (d_peer_ptr) SPMV_TRY_CUDA(cudaIpcCloseMemHandle(d_peer_ptr));
    return SPMV_B200_OK;
}

int spmv_b200_ipc_free(void *d_ptr) {
    if (d_ptr) SPMV_TRY_CUDA(cudaFree(d_ptr));
    return SPMV_B200_OK;
}

int spmv_b200_vec_push(const double *d_src, long long n, int npeers, double *const *d_peer_dst, int ctas, void *stream) {
    if (n < 0 || npeers < 0 || npeers > SPMV_B200_MAX_PEERS || (npeers > 0 && !d_peer_dst) || (n > 0 && !d_src))
        return fail(SPMV_B200_ERR_INVALID, "vec_push: bad arguments");
    if (n == 0 || npeers == 0) return SPMV_B200_OK;
    if (reinterpret_cast<uintptr_t>(d_src) & 7) return fail(SPMV_B200_ERR_INVALID, "vec_push: the source must be 8-byte aligned");
    PushTargets t;
    t.count = npeers;
    t.vector_ok = 1;
    for (int p = 0; p < npeers; ++p) {
        if (!d_peer_dst[p] || (reinterpret_cast<uintptr_t>(d_peer_dst[p]) & 7))
            return fail(SPMV_B200_ERR_INVALID, "vec_push: peer %d: NULL or not 8-byte aligned", p);
        if ((reinterpret_cast<uintptr_t>(d_peer_dst[p]) & 31) != (reinterpret_cast<uintptr_t>(d_src) & 31)) t.vector_ok = 0;
        t.dst[p] = d_peer_dst[p];
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = ctas > 0 ? ctas : 2 * sms;
    const int unroll = env_int("SPMV_B200_PUSH_UNROLL", 2), width = env_int("SPMV_B200_PUSH_WIDTH", 32);
#define PUSH_CASE(U, W) vec_push_kernel<U, W><<<grid, 512, 0, as_stream(stream)>>>(d_src, n, t)
    if (width == 32) {
        if (unroll == 1) PUSH_CASE(1, 32); else if (unroll == 4) PUSH_CASE(4, 32); else PUSH_CASE(2, 32);
    } else {
        if (unroll == 1) PUSH_CASE(1, 16); else if (unroll == 4) PUSH_CASE(4, 16); else PUSH_CASE(2, 16);
    }
#undef PUSH_CASE
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

int spmv_b200_vec_scale_by_inv_norm(double *d_dst, const double *d_src, long long n, const double *d_sumsq,
                                    void *stream) {
    if (n < 0 || (n > 0 && (!d_dst || !d_src)) || !d_sumsq)
        return fail(SPMV_B200_ERR_INVALID, "vec_scale_by_inv_norm: bad arguments");
    if (n == 0) return SPMV_B200_OK;
    scale_by_inv_norm_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(d_dst, d_src, n, d_sumsq);
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

}  // extern "C"
