// hostpath.cu -- the end-to-end entry points spmv_b200_{csr,hll}_spmv_host: host x -> device, product,
// device -> host y, as ONE pipelined pass.
//
// They replace the reference driver's "cudaMemcpy(d_x) ... kernel ... cudaMemcpy(y, DeviceToHost)" sequence
// (reference main_cuda.cu:145,166,183 and :454,471).  A host-buffer product of a resident matrix is bound by the
// PCIe link, not by HBM: 8 bytes up per column and 8 bytes down per row against 12 bytes per nonzero streamed at
// ~100x the speed.  The link is full duplex, so the call is organised to keep BOTH directions busy:
//
//   * the rows are cut into W windows (whole tiles of the plan / rows / hacks);
//   * x travels in pieces on an upload stream, piece w ending exactly where window w's referenced columns end
//     (need[w] = running maximum of max(col)+1 over windows 0..w, found once per matrix by a reduction over col_idx /
//     JA, rounded up to 256 KB), so window w is launched on a compute stream the moment ITS piece has landed;
//   * the rows of window w are copied back on a download stream as soon as its kernel is done.
//
// Measured on the B200 box (round 2, tools/r02_diag.py, profiles/r02d_diag_e2e.log), lap2d 4096^2 = 128 MiB each way:
//   * one direction alone runs at 55.4 GB/s (2.42 ms); both at once, started together, 2.80 ms; but the download of a
//     window can only start when its x has landed and, while the upload is still running, the device-to-host direction
//     gets the smaller share (~42 vs ~52 GB/s), so the pipelined call cannot reach 2.80 ms: ~3.1 ms is its floor;
//   * round 1 (equal chunks of x, a window's halo reaching into the NEXT chunk): 16 windows 3.41 ms, and copies whose
//     boundaries were not multiples of a large power of two were slower still (12 windows 3.67, 24 -> 3.87): that was
//     the "non-monotonic sweep";
//   * upload pieces that end exactly where a window's columns end (256 KB aligned): 8 windows 3.25 ms, 16 -> 3.30;
//   * kernels storing y straight into the caller's pinned buffer (zero-copy, no download copies and no kernel ->
//     copy hand-over): 16 or 32 windows 3.21 ms  <- the default;
//   * tapered windows (small first / last windows, 32 MiB in the middle) are SLOWER, 3.36 ms with copies and 3.58 ms
//     zero-copy: large windows serialise the two directions more than the small ends save (SPMV_B200_HOST_TAPER=1/2
//     keeps them for experiments).
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "handles.cuh"

namespace spmv {

constexpr int kMaxWindows = 64;  // events; the automatic choice stops at kAutoWindows.  Round 1, equal windows, measured on lap2d 4096^2: 4 -> 3.93 ms, 8 -> 3.49, 16 -> 3.42, 24 -> 3.91, 32 -> 3.65, 48 -> 3.89
constexpr int kAutoWindows = 16;
constexpr int kZeroCopyDefault = 1;
constexpr int kTaperDefault = 0;  // equal windows: the tapered schedules measured slower (see the header)
constexpr long long kUnitRows = (2LL << 20) / 8;      // 2 MiB of y
constexpr long long kPieceAlign = (256LL << 10) / 8;  // upload pieces end on 256 KB boundaries of x
constexpr long long kMinWindowBytes = 2LL << 20;  // below 2 MB of x + y per window the launch overheads win

struct HostPipe {
    cudaStream_t up = nullptr, compute = nullptr, down = nullptr;
    std::vector<cudaEvent_t> landed;  // chunk c of x is on the device
    std::vector<cudaEvent_t> done;    // window w is computed
    cudaEvent_t y_landed = nullptr;   // accumulate: the old y is on the device
    // window plan (valid for `path` only)
    int path = -1;
    int windows = 0;
    std::vector<int> unit;        // W+1: first tile / row / hack of every window
    std::vector<long long> row;   // W+1: first row of every window
    std::vector<long long> need;  // W: doubles of x that must be resident before window w starts (running maximum)
    std::vector<long long> piece; // W: upload piece w ends here (need[w] rounded up to kPieceAlign, <= N; non-decreasing)
};

void host_pipe_free(HostPipe *p) {
    if (!p) return;
    for (cudaEvent_t e : p->landed) cudaEventDestroy(e);
    for (cudaEvent_t e : p->done) cudaEventDestroy(e);
    if (p->y_landed) cudaEventDestroy(p->y_landed);
    if (p->up) cudaStreamDestroy(p->up);
    if (p->compute) cudaStreamDestroy(p->compute);
    if (p->down) cudaStreamDestroy(p->down);
    delete p;
}

static int pipe_create(HostPipe **out) {
    HostPipe *p = new (std::nothrow) HostPipe();
    if (!p) return fail(SPMV_B200_ERR_NOMEM, "spmv_host: out of host memory");
    auto body = [&]() -> int {
        SPMV_TRY_CUDA(cudaStreamCreateWithFlags(&p->up, cudaStreamNonBlocking));
        SPMV_TRY_CUDA(cudaStreamCreateWithFlags(&p->compute, cudaStreamNonBlocking));
        SPMV_TRY_CUDA(cudaStreamCreateWithFlags(&p->down, cudaStreamNonBlocking));
        SPMV_TRY_CUDA(cudaEventCreateWithFlags(&p->y_landed, cudaEventDisableTiming));
        p->landed.resize(kMaxWindows, nullptr);
        p->done.resize(kMaxWindows, nullptr);
        for (int i = 0; i < kMaxWindows; ++i) {
            SPMV_TRY_CUDA(cudaEventCreateWithFlags(&p->landed[i], cudaEventDisableTiming));
            SPMV_TRY_CUDA(cudaEventCreateWithFlags(&p->done[i], cudaEventDisableTiming));
        }
        return SPMV_B200_OK;
    };
    const int rc = body();
    if (rc != SPMV_B200_OK) {
        host_pipe_free(p);
        return rc;
    }
    *out = p;
    return SPMV_B200_OK;
}

// out[w] = max(idx[k]) + 1 over k in [bound[w], bound[w+1]); 0 for an empty range.  One launch for all windows.
__global__ void window_need_kernel(const int *__restrict__ idx, const long long *__restrict__ bound, int windows,
                                   int *__restrict__ out) {
    const int w = blockIdx.y;
    const long long lo = bound[w], hi = bound[w + 1];
    int top = 0;
    for (long long k = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x; k < hi; k += (long long)gridDim.x * blockDim.x)
        top = max(top, idx[k] + 1);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) top = max(top, __shfl_xor_sync(0xffffffffu, top, off));
    if ((threadIdx.x & 31) == 0 && top > 0) atomicMax(out + w, top);  // integer max: order independent
}

// need[] from the element ranges of the windows (elements = nonzeros of CSR / slots of HLL)
static int plan_needs(HostPipe *p, const int *d_idx, const std::vector<long long> &elem_bound) {
    const int W = p->windows;
    p->need.assign(W, 0);
    if (W == 0 || elem_bound[W] == elem_bound[0]) return SPMV_B200_OK;
    long long *d_bound = nullptr;
    int *d_out = nullptr;
    std::vector<int> top(W, 0);
    auto body = [&]() -> int {
        SPMV_TRY_CUDA(cudaMalloc(&d_bound, (size_t)(W + 1) * sizeof(long long)));
        SPMV_TRY_CUDA(cudaMalloc(&d_out, (size_t)W * sizeof(int)));
        SPMV_TRY_CUDA(cudaMemcpyAsync(d_bound, elem_bound.data(), (size_t)(W + 1) * sizeof(long long), cudaMemcpyHostToDevice, p->compute));
        SPMV_TRY_CUDA(cudaMemsetAsync(d_out, 0, (size_t)W * sizeof(int), p->compute));
        window_need_kernel<<<dim3(296, W), 256, 0, p->compute>>>(d_idx, d_bound, W, d_out);
        SPMV_TRY_CUDA(cudaGetLastError());
        SPMV_TRY_CUDA(cudaMemcpyAsync(top.data(), d_out, (size_t)W * sizeof(int), cudaMemcpyDeviceToHost, p->compute));
        SPMV_TRY_CUDA(cudaStreamSynchronize(p->compute));
        return SPMV_B200_OK;
    };
    const int rc = body();
    cudaFree(d_bound);
    cudaFree(d_out);
    if (rc != SPMV_B200_OK) return rc;
    long long running = 0;
    for (int w = 0; w < W; ++w) {
        running = std::max<long long>(running, top[w]);
        p->need[w] = running;
    }
    return SPMV_B200_OK;
}

// upload pieces: piece w ends where window w's referenced prefix of x ends, rounded up to a 256 KB boundary
static void plan_pieces(HostPipe *p, long long N) {
    p->piece.assign(p->windows, 0);
    for (int w = 0; w < p->windows; ++w)
        p->piece[w] = std::min(N, (p->need[w] + kPieceAlign - 1) / kPieceAlign * kPieceAlign);
}

static int pick_windows(long long M, long long N, int units) {
    const int forced = env_int("SPMV_B200_HOST_WINDOWS", 0);
    long long w = forced > 0 ? forced : (8 * (M + N)) / kMinWindowBytes;
    w = std::max<long long>(1, std::min<long long>(w, forced > 0 ? kMaxWindows : kAutoWindows));
    return (int)std::max<long long>(1, std::min<long long>(w, units));
}


// Row boundaries of the windows, bounds[0] = 0 .. bounds[W] = M.  Tapered on 2 MiB units (see the header) when the
// vector is large enough and no window count is forced; equal windows otherwise.
static std::vector<long long> window_rows(long long M, long long N, int units) {
    std::vector<long long> bounds;
    const long long total = (M + kUnitRows - 1) / kUnitRows;
    const int taper = env_int("SPMV_B200_HOST_TAPER", kTaperDefault);
    if (env_int("SPMV_B200_HOST_WINDOWS", 0) > 0 || taper == 0 || total < 16 || units < 16) {
        const int W = pick_windows(M, N, units);
        for (int w = 0; w <= W; ++w) {  // equal windows, on 256 KB boundaries when the vector is large
            long long r = M * w / W;
            if (w > 0 && w < W && M / W >= 8 * kPieceAlign) r = r / kPieceAlign * kPieceAlign;
            bounds.push_back(r);
        }
        return bounds;
    }
    // taper 1: ramp 1, 1, 2, 4, 8 units up, 16-unit windows, ramp down; taper 2: ramp 1, 1, 2 up, then 4-unit (8 MiB) windows
    const long long ramp[5] = {1, 1, 2, 4, 8};
    const int max_steps = taper == 2 ? 3 : 5;
    int steps = 0;
    long long ramp_sum = 0;
    while (steps < max_steps && 2 * (ramp_sum + ramp[steps]) <= total / 2) ramp_sum += ramp[steps++];
    const long long middle = total - (taper == 2 ? 1 : 2) * ramp_sum;
    long long mid_size = taper == 2 ? 4 : 16;
    while ((middle + mid_size - 1) / mid_size > kMaxWindows - 12) mid_size *= 2;
    std::vector<long long> sizes(ramp, ramp + steps);
    for (long long left = middle; left > 0; left -= mid_size) sizes.push_back(std::min(mid_size, left));
    if (taper != 2)
        for (int i = steps - 1; i >= 0; --i) sizes.push_back(ramp[i]);
    long long at = 0;
    bounds.push_back(0);
    for (long long sz : sizes) {
        at = std::min(M, at + sz * kUnitRows);
        if (at > bounds.back()) bounds.push_back(at);
    }
    bounds.back() = M;
    return bounds;
}

// A host y that the device can address (pinned or registered, unified addressing): the products can store their rows
// straight into it over PCIe and the download copies -- with their event hand-overs -- disappear.
static double *device_alias_of_host(double *y) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, y) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (attr.type != cudaMemoryTypeHost || attr.devicePointer == nullptr) return nullptr;
    return static_cast<double *>(attr.devicePointer);
}

// The pass itself.  launch(w, y_base) enqueues the kernel(s) of window w on p->compute; they write rows r of the matrix
// to y_base[r].  zero_copy_ok: every row is written exactly once and never read back by the kernels of this path.
template <class Launch>
static int run_pipeline(HostPipe *p, long long M, long long N, const double *x, double *y, double *d_x, double *d_y,
                        bool accumulate, bool zero_copy_ok, Launch launch) {
    const int W = p->windows;
    // SPMV_B200_HOST_ZEROCOPY (default on): kernels store y directly into the caller's pinned buffer
    double *y_alias = (zero_copy_ok && !accumulate && M && env_int("SPMV_B200_HOST_ZEROCOPY", kZeroCopyDefault)) ? device_alias_of_host(y) : nullptr;
    double *y_base = y_alias ? y_alias : d_y;
    // (1) uploads: the old y first (accumulate), then x in W chunks
    if (accumulate && M) {
        SPMV_TRY_CUDA(cudaMemcpyAsync(d_y, y, (size_t)M * sizeof(double), cudaMemcpyHostToDevice, p->up));
        SPMV_TRY_CUDA(cudaEventRecord(p->y_landed, p->up));
    }
    // piece w of x ends where window w's columns end; a window that needs nothing new reuses the previous event.
    // Columns no window references are never uploaded.
    std::vector<int> gate(W, -1);
    long long at = 0;
    int last = -1;
    for (int w = 0; w < W; ++w) {
        const long long upto = std::min(N, p->piece[w]);
        if (upto > at) {
            SPMV_TRY_CUDA(cudaMemcpyAsync(d_x + at, x + at, (size_t)(upto - at) * sizeof(double), cudaMemcpyHostToDevice, p->up));
            SPMV_TRY_CUDA(cudaEventRecord(p->landed[w], p->up));
            last = w;
            at = upto;
        }
        gate[w] = last;
    }
    // (2) products: window w waits for its piece
    for (int w = 0; w < W; ++w) {
        if (accumulate && M && w == 0) SPMV_TRY_CUDA(cudaStreamWaitEvent(p->compute, p->y_landed, 0));
        if (gate[w] >= 0 && (w == 0 || gate[w] != gate[w - 1])) SPMV_TRY_CUDA(cudaStreamWaitEvent(p->compute, p->landed[gate[w]], 0));
        SPMV_TRY(launch(w, y_base));
        if (!y_alias) SPMV_TRY_CUDA(cudaEventRecord(p->done[w], p->compute));
    }
    // (3) downloads, window by window (none when the kernels wrote into the host buffer themselves)
    for (int w = 0; w < W && !y_alias; ++w) {
        const long long r0 = p->row[w], r1 = p->row[w + 1];
        if (r1 <= r0) continue;
        SPMV_TRY_CUDA(cudaStreamWaitEvent(p->down, p->done[w], 0));
        SPMV_TRY_CUDA(cudaMemcpyAsync(y + r0, d_y + r0, (size_t)(r1 - r0) * sizeof(double), cudaMemcpyDeviceToHost, p->down));
    }
    SPMV_TRY_CUDA(cudaStreamSynchronize(p->down));
    SPMV_TRY_CUDA(cudaStreamSynchronize(p->compute));
    SPMV_TRY_CUDA(cudaStreamSynchronize(p->up));
    return SPMV_B200_OK;
}

static void abort_pipeline(HostPipe *p) {  // after an error: nothing of this call may still be in flight
    if (!p) return;
    cudaStreamSynchronize(p->up);
    cudaStreamSynchronize(p->compute);
    cudaStreamSynchronize(p->down);
}

// ---- CSR --------------------------------------------------------------------------------------------------------
static int csr_plan_windows(spmv_b200_csr *A, CsrPath path) {
    HostPipe *p = A->pipe;
    const bool by_tiles = path != kPathVector && path != kPathRow;
    // long rows are computed after every tile (they need all of x and are written last), the binned kernel walks the
    // rows in bin order: one window
    const int units = by_tiles ? A->num_tiles : A->M;
    std::vector<long long> bounds;
    if ((by_tiles && A->num_long > 0) || path == kPathBinned) bounds = {0, A->M};
    else bounds = window_rows(A->M, A->N, units);
    std::vector<int2> tiles_host;
    if (by_tiles && bounds.size() > 2) {  // row boundary -> the first tile that starts at or after it
        tiles_host.resize((size_t)A->num_tiles + 1);
        SPMV_TRY_CUDA(cudaMemcpy(tiles_host.data(), A->tiles, tiles_host.size() * sizeof(int2), cudaMemcpyDeviceToHost));
    }
    p->unit.clear();
    p->row.clear();
    std::vector<long long> elem;
    for (size_t w = 0; w < bounds.size(); ++w) {
        int unit;
        long long row, at;
        if (by_tiles) {
            if (w == 0) unit = 0;
            else if (w + 1 == bounds.size()) unit = A->num_tiles;
            else unit = (int)(std::lower_bound(tiles_host.begin(), tiles_host.end(), bounds[w],
                                               [](const int2 &t, long long r) { return t.x < r; }) - tiles_host.begin());
            int2 t;
            if (!tiles_host.empty()) t = tiles_host[unit];
            else SPMV_TRY_CUDA(cudaMemcpy(&t, A->tiles + unit, sizeof t, cudaMemcpyDeviceToHost));
            row = t.x;
            at = t.y;
        } else {
            unit = (int)bounds[w];
            int off = 0;
            SPMV_TRY_CUDA(cudaMemcpy(&off, A->row_ptr + unit, sizeof off, cudaMemcpyDeviceToHost));
            row = unit;
            at = off;
        }
        if (!p->unit.empty() && unit <= p->unit.back() && w + 1 != bounds.size()) continue;  // an empty window
        p->unit.push_back(unit);
        p->row.push_back(row);
        elem.push_back(at);
    }
    const int W = (int)p->unit.size() - 1;
    p->windows = W;
    SPMV_TRY(plan_needs(p, A->col_idx, elem));
    plan_pieces(p, A->N);
    p->path = (int)path;
    return SPMV_B200_OK;
}

// ---- timing harness (reference protocol, main_cuda.cu:159-200) --------------------------------------------------
template <class Launch>
static int time_products(long long M, long long N, const double *x, double *y, double *d_x, double *d_y, int warmup, int iters,
                         double *mean_seconds, double *min_seconds, Launch launch) {
    if (iters <= 0 || warmup < 0) return fail(SPMV_B200_ERR_INVALID, "time: iters must be positive");
    cudaEvent_t a = nullptr, b = nullptr;
    auto body = [&]() -> int {
        SPMV_TRY_CUDA(cudaEventCreate(&a));
        SPMV_TRY_CUDA(cudaEventCreate(&b));
        if (N && x) SPMV_TRY_CUDA(cudaMemcpy(d_x, x, (size_t)N * sizeof(double), cudaMemcpyHostToDevice));
        double sum = 0.0, best = 0.0;
        for (int i = 0; i < warmup + iters; ++i) {
            SPMV_TRY_CUDA(cudaEventRecord(a, nullptr));
            SPMV_TRY(launch());
            SPMV_TRY_CUDA(cudaEventRecord(b, nullptr));
            SPMV_TRY_CUDA(cudaEventSynchronize(b));
            float ms = 0.0f;
            SPMV_TRY_CUDA(cudaEventElapsedTime(&ms, a, b));
            if (i < warmup) continue;
            sum += ms * 1e-3;
            if (i == warmup || ms * 1e-3 < best) best = ms * 1e-3;
        }
        if (y && M) SPMV_TRY_CUDA(cudaMemcpy(y, d_y, (size_t)M * sizeof(double), cudaMemcpyDeviceToHost));
        if (mean_seconds) *mean_seconds = sum / iters;
        if (min_seconds) *min_seconds = best;
        return SPMV_B200_OK;
    };
    const int rc = body();
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
    return rc;
}

}  // namespace spmv

using namespace spmv;

extern "C" {

int spmv_b200_csr_spmv_host(spmv_b200_csr *A, const double *x, double *y, int accumulate, int algo) {
    if (!A || (A->M > 0 && !y) || (A->N > 0 && A->nnz > 0 && !x)) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_host: NULL argument");
    if (algo < SPMV_B200_ALGO_AUTO || algo > SPMV_B200_ALGO_ROW_IMAGE) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_host: unknown algo %d", algo);
    if (algo == SPMV_B200_ALGO_ROW_IMAGE && !A->image) return fail(SPMV_B200_ERR_INVALID, "csr_spmv_host: the matrix holds no image");
    if (A->M == 0) return SPMV_B200_OK;
    if (!A->stage_x) SPMV_TRY_CUDA(cudaMalloc(&A->stage_x, std::max<size_t>(A->N, 1) * sizeof(double)));
    if (!A->stage_y) SPMV_TRY_CUDA(cudaMalloc(&A->stage_y, std::max<size_t>(A->M, 1) * sizeof(double)));
    if (!A->pipe) SPMV_TRY(pipe_create(&A->pipe));
    CsrPath path = csr_resolve(A, algo);
    if (path == kPathImage) path = kPathRow;  // row windows need not fall on hacks; the row kernel gives the same bits
    if (A->pipe->path != (int)path) SPMV_TRY(csr_plan_windows(A, path));
    HostPipe *p = A->pipe;
    // the binned kernel's long rows are combined by a second kernel that may read y (accumulate); tiles with long rows too
    const bool zero_copy_ok = path != kPathBinned && A->num_long == 0;
    const int rc = run_pipeline(p, A->M, x ? A->N : 0, x, y, A->stage_x, A->stage_y, accumulate != 0, zero_copy_ok, [&](int w, double *y_base) {
        return csr_launch_window(A, path, p->unit[w], p->unit[w + 1], A->stage_x, y_base, accumulate, p->compute);
    });
    if (rc != SPMV_B200_OK) abort_pipeline(p);
    return rc;
}

int spmv_b200_hll_spmv_host(spmv_b200_hll *H, const double *x, double *y) {
    if (!H || (H->M > 0 && !y) || (H->N > 0 && H->slots > 0 && !x)) return fail(SPMV_B200_ERR_INVALID, "hll_spmv_host: NULL argument");
    if (H->M == 0) return SPMV_B200_OK;
    if (!H->stage_x) SPMV_TRY_CUDA(cudaMalloc(&H->stage_x, std::max<size_t>(H->N, 1) * sizeof(double)));
    if (!H->stage_y) SPMV_TRY_CUDA(cudaMalloc(&H->stage_y, std::max<size_t>(H->M, 1) * sizeof(double)));
    if (!H->pipe) SPMV_TRY(pipe_create(&H->pipe));
    const HllPath path = hll_resolve(H);
    const bool stream_kernel = path == kHllStream;
    HostPipe *p = H->pipe;
    if (p->path != (int)path) {
        const int units = stream_kernel ? H->num_tiles : H->num_hacks;
        const std::vector<long long> bounds = window_rows(H->M, H->N, units);
        std::vector<HllTile> tiles_host;
        if (stream_kernel) {
            tiles_host.resize((size_t)H->num_tiles + 1);
            SPMV_TRY_CUDA(cudaMemcpy(tiles_host.data(), H->tiles, tiles_host.size() * sizeof(HllTile), cudaMemcpyDeviceToHost));
        }
        p->unit.clear();
        p->row.clear();
        std::vector<long long> elem;
        for (size_t w = 0; w < bounds.size(); ++w) {
            const long long want_hack = w + 1 == bounds.size() ? H->num_hacks : bounds[w] / HACK_SIZE;  // 2 MiB units are whole hacks
            int unit, hack;
            if (stream_kernel) {
                unit = (int)(std::lower_bound(tiles_host.begin(), tiles_host.end(), want_hack,
                                              [](const HllTile &t, long long h) { return t.hack < h; }) - tiles_host.begin());
                hack = tiles_host[unit].hack;
            } else {
                unit = hack = (int)want_hack;
            }
            if (!p->unit.empty() && unit <= p->unit.back() && w + 1 != bounds.size()) continue;
            p->unit.push_back(unit);
            p->row.push_back(std::min<long long>((long long)hack * HACK_SIZE, H->M));
            elem.push_back(H->host_off[hack]);
        }
        const int W = (int)p->unit.size() - 1;
        p->windows = W;
        SPMV_TRY(plan_needs(p, H->JA, elem));
        plan_pieces(p, H->N);
        p->path = (int)path;
    }
    const int rc = run_pipeline(p, H->M, x ? H->N : 0, x, y, H->stage_x, H->stage_y, false, true, [&](int w, double *y_base) {
        return hll_launch_window(H, path, p->unit[w], p->unit[w + 1], H->stage_x, y_base, p->compute);
    });
    if (rc != SPMV_B200_OK) abort_pipeline(p);
    return rc;
}

int spmv_b200_csr_time(spmv_b200_csr *A, const double *x, double *y, int algo, int warmup, int iters, double *mean_seconds,
                       double *min_seconds) {
    if (!A || (A->N > 0 && A->nnz > 0 && !x)) return fail(SPMV_B200_ERR_INVALID, "csr_time: NULL argument");
    if (!A->stage_x) SPMV_TRY_CUDA(cudaMalloc(&A->stage_x, std::max<size_t>(A->N, 1) * sizeof(double)));
    if (!A->stage_y) SPMV_TRY_CUDA(cudaMalloc(&A->stage_y, std::max<size_t>(A->M, 1) * sizeof(double)));
    return time_products(A->M, A->N, x, y, A->stage_x, A->stage_y, warmup, iters, mean_seconds, min_seconds,
                         [&]() { return spmv_b200_csr_spmv(A, A->stage_x, A->stage_y, 0, algo, nullptr); });
}

int spmv_b200_hll_time(spmv_b200_hll *H, const double *x, double *y, int kernel, int warmup, int iters, double *mean_seconds,
                       double *min_seconds) {
    if (!H || (H->N > 0 && H->slots > 0 && !x)) return fail(SPMV_B200_ERR_INVALID, "hll_time: NULL argument");
    if (kernel < 0 || kernel > 3) return fail(SPMV_B200_ERR_INVALID, "hll_time: kernel must be 0, 1, 2 or 3");
    if (!H->stage_x) SPMV_TRY_CUDA(cudaMalloc(&H->stage_x, std::max<size_t>(H->N, 1) * sizeof(double)));
    if (!H->stage_y) SPMV_TRY_CUDA(cudaMalloc(&H->stage_y, std::max<size_t>(H->M, 1) * sizeof(double)));
    return time_products(H->M, H->N, x, y, H->stage_x, H->stage_y, warmup, iters, mean_seconds, min_seconds, [&]() {
        if (kernel == 1) return spmv_b200_hll_spmv_slice(H, H->stage_x, H->stage_y, nullptr);
        if (kernel == 2) return spmv_b200_hll_spmv_stream(H, H->stage_x, H->stage_y, nullptr);
        if (kernel == 3) return spmv_b200_hll_spmv_rows(H, H->stage_x, H->stage_y, nullptr);
        return spmv_b200_hll_spmv(H, H->stage_x, H->stage_y, nullptr);
    });
}

}  // extern "C"
