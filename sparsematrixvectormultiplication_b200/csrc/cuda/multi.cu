// multi.cu -- the row-partitioned product and the iterated product (power method, BASELINE config 5) on 1..8 GPUs of
// one box behind plain C entry points: ONE process, one host thread, peer access between the devices.
//
// The reference has no multi-GPU path (main_cuda.cu:128-200 drives device 0 only); what it does have is the
// partitioner for its OpenMP threads -- contiguous row ranges balanced by nnz (src/csr_matrix.c:167-266), cut on
// 32-row block boundaries for HLL (src/hll_matrix.c:471-498) -- and this file reuses exactly that rule with GPUs in the
// role of threads.  The per-GPU kernels are the ones of csr.cu / hll.cu; the torch.distributed path of
// distributed.py (one process per GPU, cudaIpc) drives the same kernels for bench.py.
//
// Layout of x (every GPU holds a full replica): PADDED rank-major, part p's entries at [p*stride, p*stride + rows_p),
// stride = largest part rounded up to 32; the column indices of every part are rewritten once on the device
// (spmv_b200_csr_remap_columns).  With equal slots one in-place ncclAllGather refreshes the replicas (exchange mode
// ALLGATHER), and the fused mailbox kernels (exchange mode MAILBOX) address the very same slots through peer pointers.
//
// Exchange modes of spmv_b200_multi_iterate:
//   MAILBOX    product, lazy normalisation, |w|^2 partials, boundary rows stored straight into the neighbours' replicas,
//              |w|^2 and an iteration tag published into every GPU's mailbox; no collective call.  Rows of up to 12
//              nonzeros: two launches per GPU per iteration (flat product that never waits + one-CTA exchange kernel,
//              the fastest form measured); longer rows: one launch (fused stream kernel).  Needs peer access and a
//              matrix without rows above the long-row threshold.
//   ALLGATHER  product (any kernel the plan picks, so skewed matrices work), |y|^2, a 1-double ncclAllReduce, scale of the
//              own slice, one in-place ncclAllGather of x.  NCCL is loaded with dlopen at first use (libnccl.so.2); the
//              library has no link-time dependency on it.
#include <dlfcn.h>
#include <nccl.h>  // types and enums only: every NCCL function is resolved with dlsym

#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "common.cuh"
#include "csr_matrix.h"
#include "handles.cuh"

namespace spmv {

struct Nccl {
    void *so = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

static Nccl *nccl_api() {
    static Nccl api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *name : names)
            if ((api.so = dlopen(name, RTLD_NOW | RTLD_GLOBAL))) break;
        if (api.so) {
#define NCCL_SYM(field, symbol) api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.so, symbol))
            NCCL_SYM(CommInitAll, "ncclCommInitAll");
            NCCL_SYM(CommDestroy, "ncclCommDestroy");
            NCCL_SYM(AllGather, "ncclAllGather");
            NCCL_SYM(AllReduce, "ncclAllReduce");
            NCCL_SYM(GroupStart, "ncclGroupStart");
            NCCL_SYM(GroupEnd, "ncclGroupEnd");
            NCCL_SYM(GetErrorString, "ncclGetErrorString");
#undef NCCL_SYM
            if (!api.CommInitAll || !api.CommDestroy || !api.AllGather || !api.AllReduce || !api.GroupStart || !api.GroupEnd) api.so = nullptr;
        }
    }
    return api.so ? &api : nullptr;
}

#define SPMV_TRY_NCCL(api, expr)                                                                                  \
    do {                                                                                                          \
        ncclResult_t r__ = (expr);                                                                                \
        if (r__ != ncclSuccess)                                                                                   \
            return fail(SPMV_B200_ERR_CUDA, "%s: %s", #expr, (api)->GetErrorString ? (api)->GetErrorString(r__) : "NCCL error"); \
    } while (0)

__global__ void col_minmax_kernel(long long nnz, const int *__restrict__ col_idx, int *__restrict__ out) {
    int lo = 0x7fffffff, hi = -1;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (long long)gridDim.x * blockDim.x) {
        const int c = col_idx[k];
        lo = min(lo, c);
        hi = max(hi, c);
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    if ((threadIdx.x & 31) == 0 && hi >= 0) {  // integer min / max: order independent
        atomicMin(out, lo);
        atomicMax(out + 1, hi);
    }
}

struct Part {
    int dev = 0;
    long long row_begin = 0, row_end = 0, nnz = 0;
    long long need_lo = 0, need_hi = 0;  // referenced columns (original numbering)
    spmv_b200_csr *A = nullptr;
    spmv_b200_hll *H = nullptr;
    bool fusable = true;
    bool flat = false;                  // rows of up to 12 nonzeros: the two-launch form (flat product + exchange kernel)
    double *scale = nullptr;            // {|w|^2, 1/|w|} written by the exchange kernel
    int flat_partials = 0;
    double *x[2] = {nullptr, nullptr};  // padded replicas, double buffered
    double *y = nullptr;                // owned rows (ALLGATHER mode and the plain product)
    double *partials = nullptr, *ws = nullptr, *ss = nullptr;
    unsigned long long *box = nullptr;
    unsigned int *counter = nullptr;    // [0] CTA counter, [1] status
    spmv_b200_peers_t peers[2];
    cudaStream_t stream = nullptr;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    cudaEvent_t pushed = nullptr;       // ALLGATHER_PEER: my slice has been copied into every other replica
    ncclComm_t comm = nullptr;
    long long halo = 0;                 // doubles received from neighbours per iteration (MAILBOX mode)
    int rows() const { return (int)(row_end - row_begin); }
};

}  // namespace spmv

using namespace spmv;

struct spmv_b200_multi {
    int n = 0, format = SPMV_B200_FORMAT_CSR;
    long long M = 0, N = 0, nnz = 0, stride = 0;
    std::vector<Part> parts;
    unsigned long long k = 0;  // launches since the last reset (MAILBOX mode: tag numbering)
    int cur = 0;               // which replica holds the current iterate
    int mode = -1;             // exchange mode of the iterations since the last reset
    bool nccl_ready = false;
    bool flat = false;         // every part has short rows: MAILBOX runs as two launches per iteration (fastest measured)
    double last_sumsq = 0.0;
};

namespace spmv {

static int multi_set(const Part &p) {
    SPMV_TRY_CUDA(cudaSetDevice(p.dev));
    return SPMV_B200_OK;
}

// the reference's greedy rule on a closed-form offset function (partition.py: partition_rows_by_offset)
template <class Offset>
static std::vector<std::pair<long long, long long>> greedy_parts(Offset offset, long long M, int parts) {
    std::vector<std::pair<long long, long long>> out;
    if (M <= 0 || parts <= 0) return out;
    parts = (int)std::min<long long>(parts, M);
    const long long total = offset(M), target = (total + parts - 1) / parts;
    long long start = 0;
    for (int part = 0; part < parts && start < M; ++part) {
        long long end = M;
        if (part != parts - 1) {
            const long long base = offset(start);
            if (offset(M) - base >= target) {
                long long lo = start + 1, hi = M;
                while (lo < hi) {
                    const long long mid = (lo + hi) / 2;
                    if (offset(mid) - base >= target) hi = mid; else lo = mid + 1;
                }
                end = lo;
            }
        }
        if (offset(end) - offset(start) > 0) out.emplace_back(start, end);
        start = end;
    }
    return out;
}

static void hack_align(std::vector<std::pair<long long, long long>> &parts, long long M) {
    std::vector<long long> cuts{0};
    for (size_t i = 0; i + 1 < parts.size(); ++i) cuts.push_back(parts[i].second / HACK_SIZE * HACK_SIZE);
    cuts.push_back(M);
    parts.clear();
    for (size_t i = 0; i + 1 < cuts.size(); ++i)
        if (cuts[i + 1] > cuts[i]) parts.emplace_back(cuts[i], cuts[i + 1]);
}

static int multi_prepare_devices(int ngpus) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
        return fail(SPMV_B200_ERR_NO_DEVICE, "multi: no usable CUDA device; this library has no CPU fallback");
    if (ngpus < 1 || ngpus > SPMV_B200_MAX_RANKS) return fail(SPMV_B200_ERR_INVALID, "multi: ngpus must be 1..%d (got %d)", SPMV_B200_MAX_RANKS, ngpus);
    if (ngpus > count) return fail(SPMV_B200_ERR_INVALID, "multi: %d GPUs requested, %d visible", ngpus, count);
    for (int a = 0; a < ngpus; ++a) {
        SPMV_TRY_CUDA(cudaSetDevice(a));
        for (int b = 0; b < ngpus; ++b) {
            if (a == b) continue;
            int can = 0;
            SPMV_TRY_CUDA(cudaDeviceCanAccessPeer(&can, a, b));
            if (!can) return fail(SPMV_B200_ERR_INVALID, "multi: GPU %d cannot access GPU %d (no NVLink / P2P path)", a, b);
            const cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) SPMV_TRY_CUDA(e);
            cudaGetLastError();
        }
    }
    return SPMV_B200_OK;
}

// after every part has its CSR matrix (global columns) on its device: column ranges, padded layout, remap, HLL, buffers
static int multi_finish(spmv_b200_multi *ctx) {
    const int n = ctx->n;
    long long rows_max = 0;
    for (const Part &p : ctx->parts) rows_max = std::max<long long>(rows_max, p.rows());

    ctx->stride = (rows_max + 31) / 32 * 32;
    if ((long long)n * ctx->stride > 0x7fffffffLL) return fail(SPMV_B200_ERR_INVALID, "multi: padded x exceeds int32 indexing");
    long long starts[SPMV_B200_MAX_RANKS + 1];
    for (int i = 0; i < n; ++i) starts[i] = ctx->parts[i].row_begin;
    starts[n] = ctx->N;
    if (ctx->M != ctx->N) return fail(SPMV_B200_ERR_INVALID, "multi: the iterated product needs a square matrix (M=%lld, N=%lld)", ctx->M, ctx->N);
    for (Part &p : ctx->parts) {
        SPMV_TRY(multi_set(p));
        spmv_b200_csr_info_t info;
        SPMV_TRY(spmv_b200_csr_info(p.A, &info));
        p.nnz = info.nnz;
        p.fusable = info.num_long_rows == 0;
        p.flat = info.max_row_nnz <= 12;
        int mm[2] = {0x7fffffff, -1}, *d_mm = nullptr;
        if (info.nnz > 0) {
            const int *cols = nullptr;
            SPMV_TRY(spmv_b200_csr_device_arrays(p.A, nullptr, &cols, nullptr));
            SPMV_TRY_CUDA(cudaMalloc(&d_mm, sizeof mm));
            cudaError_t e = cudaMemcpy(d_mm, mm, sizeof mm, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) {
                col_minmax_kernel<<<1024, 256>>>(info.nnz, cols, d_mm);
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaMemcpy(mm, d_mm, sizeof mm, cudaMemcpyDeviceToHost);
            cudaFree(d_mm);  // on every path: an error below returns from this function
            SPMV_TRY_CUDA(e);
        }
        p.need_lo = mm[1] >= 0 ? mm[0] : p.row_begin;
        p.need_hi = mm[1] >= 0 ? mm[1] + 1 : p.row_begin;
        if (n > 1) SPMV_TRY(spmv_b200_csr_remap_columns(p.A, n, starts, ctx->stride, nullptr));
        if (ctx->format == SPMV_B200_FORMAT_HLL) {
            SPMV_TRY(spmv_b200_hll_from_csr(p.A, nullptr, &p.H));
            spmv_b200_csr_free(p.A);
            p.A = nullptr;
        }
        const size_t xbytes = (size_t)std::max<long long>(n > 1 ? n * ctx->stride : ctx->N, 1) * sizeof(double);
        for (int b = 0; b < 2; ++b) SPMV_TRY_CUDA(cudaMalloc(&p.x[b], xbytes));
        SPMV_TRY_CUDA(cudaMalloc(&p.y, (size_t)std::max(p.rows(), 1) * sizeof(double)));
        p.flat_partials = p.flat ? (p.A ? spmv_b200_csr_flat_partials_count(p.A) : spmv_b200_hll_flat_partials_count(p.H)) : 0;
        const int pc = std::max(std::max(p.A ? spmv_b200_csr_partials_count(p.A) : spmv_b200_hll_partials_count(p.H), p.flat_partials), 1);
        SPMV_TRY_CUDA(cudaMalloc(&p.partials, (size_t)pc * sizeof(double)));
        SPMV_TRY_CUDA(cudaMemset(p.partials, 0, (size_t)pc * sizeof(double)));
        SPMV_TRY_CUDA(cudaMalloc(&p.scale, 2 * sizeof(double)));
        SPMV_TRY_CUDA(cudaMalloc(&p.ws, (size_t)spmv_b200_vec_ws_doubles() * sizeof(double)));
        SPMV_TRY_CUDA(cudaMalloc(&p.ss, sizeof(double)));
        SPMV_TRY_CUDA(cudaMalloc(&p.box, SPMV_B200_MAILBOX_BYTES));
        SPMV_TRY_CUDA(cudaMalloc(&p.counter, 2 * sizeof(unsigned int)));
        SPMV_TRY_CUDA(cudaStreamCreateWithFlags(&p.stream, cudaStreamNonBlocking));
        SPMV_TRY_CUDA(cudaEventCreate(&p.t0));
        SPMV_TRY_CUDA(cudaEventCreate(&p.t1));
        SPMV_TRY_CUDA(cudaEventCreateWithFlags(&p.pushed, cudaEventDisableTiming));
    }
    ctx->flat = true;
    for (const Part &p : ctx->parts) ctx->flat = ctx->flat && p.flat;
    // who needs which of my rows (ExchangePlan of distributed.py): part j references columns [need_lo, need_hi)
    for (int i = 0; i < n; ++i) {
        Part &me = ctx->parts[i];
        for (int b = 0; b < 2; ++b) me.peers[b].count = 0;
        for (int j = 0; j < n; ++j) {
            if (j == i) continue;
            const Part &peer = ctx->parts[j];
            const long long lo = std::max(me.row_begin, peer.need_lo), hi = std::min(me.row_end, peer.need_hi);
            if (hi <= lo) continue;
            for (int b = 0; b < 2; ++b) {
                spmv_b200_peers_t &ps = me.peers[b];
                ps.dst[ps.count] = peer.x[b] + (long long)i * ctx->stride;  // the peer's slot for MY local row 0
                ps.lo[ps.count] = (int)(lo - me.row_begin);
                ps.hi[ps.count] = (int)(hi - me.row_begin);
                ++ps.count;
            }
            const long long rlo = std::max(peer.row_begin, me.need_lo), rhi = std::min(peer.row_end, me.need_hi);
            if (rhi > rlo) me.halo += rhi - rlo;
        }
    }
    return SPMV_B200_OK;
}

static int multi_nccl(spmv_b200_multi *ctx, Nccl **out) {
    Nccl *api = nccl_api();
    if (!api) return fail(SPMV_B200_ERR_INVALID, "multi: exchange mode ALLGATHER needs NCCL, and libnccl.so.2 could not be loaded (%s)", dlerror());
    if (!ctx->nccl_ready) {
        std::vector<int> devs;
        std::vector<ncclComm_t> comms(ctx->n);
        for (const Part &p : ctx->parts) devs.push_back(p.dev);
        SPMV_TRY_NCCL(api, api->CommInitAll(comms.data(), ctx->n, devs.data()));
        for (int i = 0; i < ctx->n; ++i) ctx->parts[i].comm = comms[i];
        ctx->nccl_ready = true;
    }
    *out = api;
    return SPMV_B200_OK;
}

static double *own_slot(const spmv_b200_multi *ctx, const Part &p, int which, int index) {
    return p.x[which] + (ctx->n > 1 ? (long long)index * ctx->stride : 0);
}

}  // namespace spmv

extern "C" {

int spmv_b200_multi_init_synth(int ngpus, int format, int kind, long long p0, long long p1, int p2, unsigned long long seed,
                               spmv_b200_multi **out) {
    if (!out) return fail(SPMV_B200_ERR_INVALID, "multi_init_synth: out is NULL");
    *out = nullptr;
    if (format != SPMV_B200_FORMAT_CSR && format != SPMV_B200_FORMAT_HLL) return fail(SPMV_B200_ERR_INVALID, "multi_init_synth: unknown format %d", format);
    long long M = 0, N = 0;
    switch (kind) {
        case SPMV_B200_SYNTH_LAP2D: M = N = p0 * p0; break;
        case SPMV_B200_SYNTH_LAP3D: M = N = p0 * p0 * p0; break;
        case SPMV_B200_SYNTH_UNIFORM: M = p0; N = p1; break;
        default: return fail(SPMV_B200_ERR_INVALID, "multi_init_synth: unknown kind %d", kind);
    }
    if (p0 <= 0 || M > 0x7fffffffLL) return fail(SPMV_B200_ERR_INVALID, "multi_init_synth: dimensions out of int32 range");
    SPMV_TRY(multi_prepare_devices(ngpus));
    auto ranges = greedy_parts([&](long long r) { return spmv_b200_synth_row_offset(kind, p0, p1, p2, r); }, M, ngpus);
    if (format == SPMV_B200_FORMAT_HLL) hack_align(ranges, M);
    if (ranges.empty()) return fail(SPMV_B200_ERR_INVALID, "multi_init_synth: empty matrix");
    spmv_b200_multi *ctx = new (std::nothrow) spmv_b200_multi();
    if (!ctx) return fail(SPMV_B200_ERR_NOMEM, "multi_init_synth: out of host memory");
    ctx->n = (int)ranges.size();
    ctx->format = format;
    ctx->M = M;
    ctx->N = N;
    ctx->nnz = spmv_b200_synth_row_offset(kind, p0, p1, p2, M);
    ctx->parts.resize(ctx->n);
    int rc = SPMV_B200_OK;
    for (int i = 0; i < ctx->n && rc == SPMV_B200_OK; ++i) {
        Part &p = ctx->parts[i];
        p.dev = i;
        p.row_begin = ranges[i].first;
        p.row_end = ranges[i].second;
        rc = multi_set(p);
        if (rc == SPMV_B200_OK) rc = spmv_b200_synth_csr(kind, p0, p1, p2, seed, p.row_begin, p.row_end, nullptr, &p.A);
    }
    if (rc == SPMV_B200_OK) rc = multi_finish(ctx);
    if (rc != SPMV_B200_OK) {
        spmv_b200_multi_free(ctx);
        return rc;
    }
    rc = spmv_b200_multi_reset(ctx, nullptr);
    if (rc != SPMV_B200_OK) {
        spmv_b200_multi_free(ctx);
        return rc;
    }
    *out = ctx;
    return SPMV_B200_OK;
}

int spmv_b200_multi_init_csr(int ngpus, int format, int M, int N, long long nnz, const int *row_ptr, const int *col_idx,
                             const double *values, spmv_b200_multi **out) {
    if (!out) return fail(SPMV_B200_ERR_INVALID, "multi_init_csr: out is NULL");
    *out = nullptr;
    if (format != SPMV_B200_FORMAT_CSR && format != SPMV_B200_FORMAT_HLL) return fail(SPMV_B200_ERR_INVALID, "multi_init_csr: unknown format %d", format);
    if (M <= 0 || N <= 0 || nnz < 0 || !row_ptr || (nnz > 0 && (!col_idx || !values)))
        return fail(SPMV_B200_ERR_INVALID, "multi_init_csr: bad arguments (M=%d N=%d nnz=%lld)", M, N, nnz);
    SPMV_TRY(multi_prepare_devices(ngpus));
    // the reference's own partitioner (src/csr_matrix.c:167-266): it returns the number of ranges it used
    int *start = nullptr, *end = nullptr;
    const int used = prepare_thread_distribution(M, row_ptr, ngpus, nnz, &start, &end);
    if (used <= 0 || !start || !end) {
        free(start);
        free(end);
        return fail(SPMV_B200_ERR_INVALID, "multi_init_csr: the row partitioner produced no ranges");
    }
    std::vector<std::pair<long long, long long>> ranges;
    for (int i = 0; i < used; ++i) ranges.emplace_back(start[i], end[i]);
    free(start);
    free(end);
    ranges.front().first = 0;  // rows without nonzeros before the first / after the last range still belong to somebody
    ranges.back().second = M;
    if (format == SPMV_B200_FORMAT_HLL) hack_align(ranges, M);
    spmv_b200_multi *ctx = new (std::nothrow) spmv_b200_multi();
    if (!ctx) return fail(SPMV_B200_ERR_NOMEM, "multi_init_csr: out of host memory");
    ctx->n = (int)ranges.size();
    ctx->format = format;
    ctx->M = M;
    ctx->N = N;
    ctx->nnz = nnz;
    ctx->parts.resize(ctx->n);
    int rc = SPMV_B200_OK;
    std::vector<int> local_ptr;
    for (int i = 0; i < ctx->n && rc == SPMV_B200_OK; ++i) {
        Part &p = ctx->parts[i];
        p.dev = i;
        p.row_begin = ranges[i].first;
        p.row_end = ranges[i].second;
        const int base = row_ptr[p.row_begin];
        local_ptr.resize((size_t)p.rows() + 1);
        for (int r = 0; r <= p.rows(); ++r) local_ptr[r] = row_ptr[p.row_begin + r] - base;
        rc = multi_set(p);
        if (rc == SPMV_B200_OK)
            rc = spmv_b200_csr_upload(p.rows(), N, local_ptr[p.rows()], local_ptr.data(), col_idx + base, values + base, &p.A);
    }
    if (rc == SPMV_B200_OK) rc = multi_finish(ctx);
    if (rc == SPMV_B200_OK) rc = spmv_b200_multi_reset(ctx, nullptr);
    if (rc != SPMV_B200_OK) {
        spmv_b200_multi_free(ctx);
        return rc;
    }
    *out = ctx;
    return SPMV_B200_OK;
}

int spmv_b200_multi_info(const spmv_b200_multi *ctx, spmv_b200_multi_info_t *info) {
    if (!ctx || !info) return fail(SPMV_B200_ERR_INVALID, "multi_info: NULL argument");
    std::memset(info, 0, sizeof *info);
    info->ngpus = ctx->n;
    info->format = ctx->format;
    info->M = ctx->M;
    info->N = ctx->N;
    info->nnz = ctx->nnz;
    info->stride = ctx->stride;
    info->fused_ok = 1;
    for (int i = 0; i < ctx->n; ++i) {
        const Part &p = ctx->parts[i];
        info->row_begin[i] = p.row_begin;
        info->row_end[i] = p.row_end;
        info->nnz_part[i] = p.nnz;
        info->halo_doubles[i] = p.halo;
        if (!p.fusable) info->fused_ok = 0;
    }
    return SPMV_B200_OK;
}

int spmv_b200_multi_reset(spmv_b200_multi *ctx, const double *x0) {
    if (!ctx) return fail(SPMV_B200_ERR_INVALID, "multi_reset: NULL context");
    for (Part &p : ctx->parts) {  // nothing of a previous run may still be in flight when the mailboxes are cleared
        SPMV_TRY(multi_set(p));
        SPMV_TRY_CUDA(cudaStreamSynchronize(p.stream));
    }
    for (Part &p : ctx->parts) {
        SPMV_TRY(multi_set(p));
        for (int b = 0; b < 2; ++b) {
            if (!x0) {
                SPMV_TRY(spmv_b200_vec_fill(p.x[b], ctx->n > 1 ? ctx->n * ctx->stride : ctx->N, 1.0, p.stream));
            } else {
                for (int j = 0; j < ctx->n; ++j) {
                    const Part &q = ctx->parts[j];
                    SPMV_TRY_CUDA(cudaMemcpyAsync(own_slot(ctx, p, b, j), x0 + q.row_begin, (size_t)q.rows() * sizeof(double),
                                                  cudaMemcpyHostToDevice, p.stream));
                }
            }
        }
        SPMV_TRY_CUDA(cudaMemsetAsync(p.box, 0, SPMV_B200_MAILBOX_BYTES, p.stream));
        SPMV_TRY_CUDA(cudaMemsetAsync(p.counter, 0, 2 * sizeof(unsigned int), p.stream));
        SPMV_TRY_CUDA(cudaStreamSynchronize(p.stream));
    }
    ctx->k = 0;
    ctx->cur = 0;
    ctx->mode = -1;
    ctx->last_sumsq = 0.0;
    return SPMV_B200_OK;
}

int spmv_b200_multi_iterate(spmv_b200_multi *ctx, int iters, int exchange, double *lambda, double *ms_per_iteration) {
    if (!ctx || iters < 1) return fail(SPMV_B200_ERR_INVALID, "multi_iterate: bad arguments");
    if (exchange != SPMV_B200_EXCHANGE_MAILBOX && exchange != SPMV_B200_EXCHANGE_ALLGATHER && exchange != SPMV_B200_EXCHANGE_ALLGATHER_PEER)
        return fail(SPMV_B200_ERR_INVALID, "multi_iterate: unknown exchange mode %d", exchange);
    if (ctx->mode >= 0 && ctx->mode != exchange)
        return fail(SPMV_B200_ERR_INVALID, "multi_iterate: the exchange mode changed; call spmv_b200_multi_reset first (MAILBOX keeps "
                                           "the iterate unnormalised between launches, ALLGATHER normalised)");
    const int n = ctx->n;
    Nccl *api = nullptr;
    if (exchange == SPMV_B200_EXCHANGE_MAILBOX) {
        for (const Part &p : ctx->parts)
            if (!p.fusable) return fail(SPMV_B200_ERR_INVALID, "multi_iterate: rows above the long-row threshold on GPU %d; use SPMV_B200_EXCHANGE_ALLGATHER", p.dev);
        for (Part &p : ctx->parts)  // the fused products never read a CSR part's private image
            if (p.A) {
                SPMV_TRY(multi_set(p));
                SPMV_TRY(spmv_b200_csr_set_image(p.A, 0, p.stream));
            }
    } else if (n > 1 && exchange == SPMV_B200_EXCHANGE_ALLGATHER) {
        SPMV_TRY(multi_nccl(ctx, &api));
    }
    ctx->mode = exchange;
    for (Part &p : ctx->parts) {
        SPMV_TRY(multi_set(p));
        SPMV_TRY_CUDA(cudaEventRecord(p.t0, p.stream));
    }
    for (int it = 0; it < iters; ++it) {
        const int cur = ctx->cur, nxt = cur ^ 1;
        if (exchange == SPMV_B200_EXCHANGE_MAILBOX) {
            for (int i = 0; i < n; ++i) {
                Part &p = ctx->parts[i];
                SPMV_TRY(multi_set(p));
                spmv_b200_mail_t mail;
                std::memset(&mail, 0, sizeof mail);
                mail.world = n;
                mail.rank = i;
                mail.iteration = ctx->k;
                for (int r = 0; r < n; ++r) mail.box[r] = ctx->parts[r].box;
                mail.counter = p.counter;
                mail.status = reinterpret_cast<int *>(p.counter + 1);
                double *y = own_slot(ctx, p, nxt, i);
                if (ctx->flat) {  // two launches: flat product (never waits) + one-CTA exchange kernel
                    const double *inv = ctx->k > 0 ? p.scale + 1 : nullptr;
                    if (p.A) SPMV_TRY(spmv_b200_csr_spmv_fused_flat(p.A, p.x[cur], y, inv, p.partials, &p.peers[nxt], p.stream));
                    else SPMV_TRY(spmv_b200_hll_spmv_fused_flat(p.H, p.x[cur], y, inv, p.partials, &p.peers[nxt], p.stream));
                    SPMV_TRY(spmv_b200_mail_exchange(p.partials, p.flat_partials, &mail, p.scale, p.stream));
                } else if (p.A) {
                    SPMV_TRY(spmv_b200_csr_spmv_fused_mail(p.A, p.x[cur], y, p.partials, &p.peers[nxt], &mail, p.stream));
                } else {
                    SPMV_TRY(spmv_b200_hll_spmv_fused_mail(p.H, p.x[cur], y, p.partials, &p.peers[nxt], &mail, p.stream));
                }
            }
            ctx->cur = nxt;
        } else if (exchange == SPMV_B200_EXCHANGE_ALLGATHER_PEER) {
            // No library call: |y|^2 through the mailboxes (the exchange kernel also proves that EVERY GPU has finished
            // reading x for this iteration, so the replicas may be overwritten), then one DMA copy of the own slice per
            // peer, nearest successor first -- at any moment every GPU is the target of one other GPU.
            for (int i = 0; i < n; ++i) {
                Part &p = ctx->parts[i];
                SPMV_TRY(multi_set(p));
                if (p.A) SPMV_TRY(spmv_b200_csr_spmv(p.A, p.x[0], p.y, 0, SPMV_B200_ALGO_AUTO, p.stream));
                else SPMV_TRY(spmv_b200_hll_spmv(p.H, p.x[0], p.y, p.stream));
                SPMV_TRY(spmv_b200_vec_sumsq(p.y, p.rows(), p.ws, p.ss, p.stream));
                spmv_b200_mail_t mail;
                std::memset(&mail, 0, sizeof mail);
                mail.world = n;
                mail.rank = i;
                mail.iteration = ctx->k;
                for (int r = 0; r < n; ++r) mail.box[r] = ctx->parts[r].box;
                mail.counter = p.counter;
                mail.status = reinterpret_cast<int *>(p.counter + 1);
                SPMV_TRY(spmv_b200_mail_exchange(p.ss, 1, &mail, p.scale, p.stream));  // scale[0] = |y|^2 over all GPUs, rank order
                SPMV_TRY(spmv_b200_vec_scale_by_inv_norm(own_slot(ctx, p, 0, i), p.y, p.rows(), p.scale, p.stream));
                for (int step = 1; step < n; ++step) {
                    const int j = (i + step) % n;
                    const Part &q = ctx->parts[j];
                    SPMV_TRY_CUDA(cudaMemcpyPeerAsync(q.x[0] + (long long)i * ctx->stride, q.dev, own_slot(ctx, p, 0, i), p.dev,
                                                      (size_t)p.rows() * sizeof(double), p.stream));
                }
                if (n > 1) SPMV_TRY_CUDA(cudaEventRecord(p.pushed, p.stream));
            }
            for (int j = 0; n > 1 && j < n; ++j) {  // the next product on GPU j starts when every slice has landed there
                Part &q = ctx->parts[j];
                SPMV_TRY(multi_set(q));
                for (int i = 0; i < n; ++i)
                    if (i != j) SPMV_TRY_CUDA(cudaStreamWaitEvent(q.stream, ctx->parts[i].pushed, 0));
            }
        } else {
            for (int i = 0; i < n; ++i) {  // y = A x ; |y|^2
                Part &p = ctx->parts[i];
                SPMV_TRY(multi_set(p));
                if (p.A) SPMV_TRY(spmv_b200_csr_spmv(p.A, p.x[0], p.y, 0, SPMV_B200_ALGO_AUTO, p.stream));
                else SPMV_TRY(spmv_b200_hll_spmv(p.H, p.x[0], p.y, p.stream));
                SPMV_TRY(spmv_b200_vec_sumsq(p.y, p.rows(), p.ws, p.ss, p.stream));
            }
            if (n > 1) {
                SPMV_TRY_NCCL(api, api->GroupStart());
                for (Part &p : ctx->parts) SPMV_TRY_NCCL(api, api->AllReduce(p.ss, p.ss, 1, ncclFloat64, ncclSum, p.comm, p.stream));
                SPMV_TRY_NCCL(api, api->GroupEnd());
            }
            for (int i = 0; i < n; ++i) {  // own slice of x = y / |y|
                Part &p = ctx->parts[i];
                SPMV_TRY(multi_set(p));
                SPMV_TRY(spmv_b200_vec_scale_by_inv_norm(own_slot(ctx, p, 0, i), p.y, p.rows(), p.ss, p.stream));
            }
            if (n > 1) {  // ONE in-place all-gather: every GPU's send buffer is its own slot of the receive buffer
                SPMV_TRY_NCCL(api, api->GroupStart());
                for (int i = 0; i < n; ++i) {
                    Part &p = ctx->parts[i];
                    SPMV_TRY_NCCL(api, api->AllGather(own_slot(ctx, p, 0, i), p.x[0], (size_t)ctx->stride, ncclFloat64, p.comm, p.stream));
                }
                SPMV_TRY_NCCL(api, api->GroupEnd());
            }
        }
        ++ctx->k;
    }
    float worst = 0.0f;
    for (Part &p : ctx->parts) {
        SPMV_TRY(multi_set(p));
        SPMV_TRY_CUDA(cudaEventRecord(p.t1, p.stream));
    }
    for (Part &p : ctx->parts) {
        SPMV_TRY(multi_set(p));
        SPMV_TRY_CUDA(cudaEventSynchronize(p.t1));
        float ms = 0.0f;
        SPMV_TRY_CUDA(cudaEventElapsedTime(&ms, p.t0, p.t1));
        worst = std::max(worst, ms);
    }
    if (ms_per_iteration) *ms_per_iteration = (double)worst / iters;
    // |w_k|^2
    double total = 0.0;
    if ((exchange == SPMV_B200_EXCHANGE_MAILBOX && ctx->flat) || exchange == SPMV_B200_EXCHANGE_ALLGATHER_PEER) {  // the exchange kernel left {|w|^2, 1/|w|} on every GPU
        for (Part &p : ctx->parts) {
            unsigned int sync[2];
            SPMV_TRY(multi_set(p));
            SPMV_TRY_CUDA(cudaMemcpy(sync, p.counter, sizeof sync, cudaMemcpyDeviceToHost));
            if (sync[1] != 0) return fail(SPMV_B200_ERR_CUDA, "multi_iterate: a mailbox wait on GPU %d timed out (a peer did not finish its launch)", p.dev);
        }
        Part &p0 = ctx->parts[0];
        SPMV_TRY(multi_set(p0));
        SPMV_TRY_CUDA(cudaMemcpy(&total, p0.scale, sizeof total, cudaMemcpyDeviceToHost));
    } else if (exchange == SPMV_B200_EXCHANGE_MAILBOX) {
        Part &p0 = ctx->parts[0];
        SPMV_TRY(multi_set(p0));
        unsigned long long host_box[SPMV_B200_MAILBOX_BYTES / 8];
        unsigned int sync[2];
        SPMV_TRY_CUDA(cudaMemcpy(host_box, p0.box, sizeof host_box, cudaMemcpyDeviceToHost));
        for (Part &p : ctx->parts) {
            SPMV_TRY(multi_set(p));
            SPMV_TRY_CUDA(cudaMemcpy(sync, p.counter, sizeof sync, cudaMemcpyDeviceToHost));
            if (sync[1] != 0) return fail(SPMV_B200_ERR_CUDA, "multi_iterate: a mailbox wait on GPU %d timed out (a peer did not finish its launch)", p.dev);
        }
        const int parity = (int)((ctx->k - 1) & 1);
        for (int r = 0; r < n; ++r) {  // rank order, as the kernels add them
            const unsigned long long *slot = host_box + 2 * (parity * n + r);
            if (slot[1] != ctx->k) return fail(SPMV_B200_ERR_CUDA, "multi_iterate: mailbox slot of GPU %d carries tag %llu, expected %llu", r, slot[1], ctx->k);
            double v;
            std::memcpy(&v, &slot[0], sizeof v);
            total += v;
        }
    } else {
        Part &p0 = ctx->parts[0];
        SPMV_TRY(multi_set(p0));
        SPMV_TRY_CUDA(cudaMemcpy(&total, p0.ss, sizeof total, cudaMemcpyDeviceToHost));
    }
    ctx->last_sumsq = total;
    if (lambda) *lambda = std::sqrt(total);
    return SPMV_B200_OK;
}

int spmv_b200_multi_get_x(spmv_b200_multi *ctx, double *x_host) {
    if (!ctx || !x_host) return fail(SPMV_B200_ERR_INVALID, "multi_get_x: NULL argument");
    const int which = ctx->mode == SPMV_B200_EXCHANGE_MAILBOX ? ctx->cur : 0;
    for (int i = 0; i < ctx->n; ++i) {
        Part &p = ctx->parts[i];
        SPMV_TRY(multi_set(p));
        SPMV_TRY_CUDA(cudaStreamSynchronize(p.stream));
        SPMV_TRY_CUDA(cudaMemcpy(x_host + p.row_begin, own_slot(ctx, p, which, i), (size_t)p.rows() * sizeof(double), cudaMemcpyDeviceToHost));
    }
    if (ctx->mode == SPMV_B200_EXCHANGE_MAILBOX && ctx->k > 0 && ctx->last_sumsq > 0.0) {  // stored iterate is w_k: v_k = w_k / |w_k|
        const double norm = std::sqrt(ctx->last_sumsq);
        for (long long r = 0; r < ctx->M; ++r) x_host[r] /= norm;
    }
    return SPMV_B200_OK;
}

int spmv_b200_multi_spmv(spmv_b200_multi *ctx, const double *x_host, double *y_host) {
    if (!ctx || !x_host || !y_host) return fail(SPMV_B200_ERR_INVALID, "multi_spmv: NULL argument");
    // scratch: replica 1 when no iteration is in flight in it (MAILBOX alternates both) -- the product leaves the
    // iteration state alone only after a reset, so it is refused in the middle of a MAILBOX run
    if (ctx->mode == SPMV_B200_EXCHANGE_MAILBOX && ctx->k > 0)
        return fail(SPMV_B200_ERR_INVALID, "multi_spmv: a MAILBOX iteration is in progress; call spmv_b200_multi_reset first");
    for (int i = 0; i < ctx->n; ++i) {
        Part &p = ctx->parts[i];
        SPMV_TRY(multi_set(p));
        for (int j = 0; j < ctx->n; ++j) {
            const Part &q = ctx->parts[j];
            SPMV_TRY_CUDA(cudaMemcpyAsync(own_slot(ctx, p, 1, j), x_host + q.row_begin, (size_t)q.rows() * sizeof(double),
                                          cudaMemcpyHostToDevice, p.stream));
        }
        if (p.A) SPMV_TRY(spmv_b200_csr_spmv(p.A, p.x[1], p.y, 0, SPMV_B200_ALGO_AUTO, p.stream));
        else SPMV_TRY(spmv_b200_hll_spmv(p.H, p.x[1], p.y, p.stream));
        SPMV_TRY_CUDA(cudaMemcpyAsync(y_host + p.row_begin, p.y, (size_t)p.rows() * sizeof(double), cudaMemcpyDeviceToHost, p.stream));
    }
    for (Part &p : ctx->parts) {
        SPMV_TRY(multi_set(p));
        SPMV_TRY_CUDA(cudaStreamSynchronize(p.stream));
    }
    return SPMV_B200_OK;
}

void spmv_b200_multi_free(spmv_b200_multi *ctx) {
    if (!ctx) return;
    Nccl *api = ctx->nccl_ready ? nccl_api() : nullptr;
    for (Part &p : ctx->parts) {
        if (cudaSetDevice(p.dev) != cudaSuccess) continue;
        if (p.stream) cudaStreamSynchronize(p.stream);
    }
    for (Part &p : ctx->parts) {
        if (cudaSetDevice(p.dev) != cudaSuccess) continue;
        if (api && p.comm) api->CommDestroy(p.comm);
        spmv_b200_csr_free(p.A);
        spmv_b200_hll_free(p.H);
        for (int b = 0; b < 2; ++b) cudaFree(p.x[b]);
        cudaFree(p.y);
        cudaFree(p.partials);
        cudaFree(p.scale);
        cudaFree(p.ws);
        cudaFree(p.ss);
        cudaFree(p.box);
        cudaFree(p.counter);
        if (p.t0) cudaEventDestroy(p.t0);
        if (p.t1) cudaEventDestroy(p.t1);
        if (p.pushed) cudaEventDestroy(p.pushed);
        if (p.stream) cudaStreamDestroy(p.stream);
    }
    cudaGetLastError();
    delete ctx;
}

}  // extern "C"
