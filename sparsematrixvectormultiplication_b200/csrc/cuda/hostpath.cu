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
//
// The multi-vector products spmv_b200_{csr,hll}_spmm_host[_f32] run the same pass over k columns (run_pipeline with
// HostCols): windows of rows (CSR) or hacks (HLL) planned once per handle in a HostPipe of their own, piece w of X ending
// at need[w] rows (aligned to 256 KB of the staged block), the SpMM kernels of spmm.cu launched per window on shifted
// base pointers, the CSR long rows (csr_spmm_long) after a block's last piece.  X, and Y when it is staged, are staged
// in blocks of kc columns (all k when they fit half of the free device memory); a block's pieces and downloads are 2-D
// copies unless the block is contiguous on both sides.
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
    cudaEvent_t x_free = nullptr;     // column blocks: the last kernel of the previous block has read the staged X
    cudaEvent_t y_free = nullptr;     // column blocks: the staged Y of the previous block is downloaded
    // window plan (valid for `path` only)
    int path = -1;
    int windows = 0;
    std::vector<int> unit;        // W+1: first tile / row / hack of every window
    std::vector<long long> row;   // W+1: first row of every window
    std::vector<long long> need;  // W: doubles of x that must be resident before window w starts (running maximum)
    std::vector<long long> piece; // W: upload piece w ends here (need[w] rounded up to kPieceAlign, <= N; non-decreasing)
    std::vector<char> tail_window;  // multi-vector CSR with long rows: W flags, window w holds a long row
    void *stage = nullptr;          // multi-vector products: the staged column block of X, then of Y
    size_t stage_bytes = 0;
};

void host_pipe_free(HostPipe *p) {
    if (!p) return;
    for (cudaEvent_t e : p->landed) cudaEventDestroy(e);
    for (cudaEvent_t e : p->done) cudaEventDestroy(e);
    if (p->y_landed) cudaEventDestroy(p->y_landed);
    if (p->x_free) cudaEventDestroy(p->x_free);
    if (p->y_free) cudaEventDestroy(p->y_free);
    cudaFree(p->stage);
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
        SPMV_TRY_CUDA(cudaEventCreateWithFlags(&p->x_free, cudaEventDisableTiming));
        SPMV_TRY_CUDA(cudaEventCreateWithFlags(&p->y_free, cudaEventDisableTiming));
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

// upload pieces: piece w ends where window w's referenced prefix of x ends, rounded up to `align` rows
static std::vector<long long> pieces_of(const HostPipe *p, long long N, long long align) {
    std::vector<long long> piece(p->windows, 0);
    for (int w = 0; w < p->windows; ++w) piece[w] = std::min(N, (p->need[w] + align - 1) / align * align);
    return piece;
}

// one vector: on 256 KB boundaries of x
static void plan_pieces(HostPipe *p, long long N) { p->piece = pieces_of(p, N, kPieceAlign); }

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
template <class V>
static V *device_alias_of_host(V *y) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, y) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (attr.type != cudaMemoryTypeHost || attr.devicePointer == nullptr) return nullptr;
    return static_cast<V *>(attr.devicePointer);
}

// SPMV_B200_HOST_ZEROCOPY (default on; 0 forces it off): kernels store y directly into the caller's pinned buffer
template <class V>
static V *zero_copy_alias(bool zero_copy_ok, bool accumulate, long long M, V *y) {
    return (zero_copy_ok && !accumulate && M && env_int("SPMV_B200_HOST_ZEROCOPY", kZeroCopyDefault)) ? device_alias_of_host(y) : nullptr;
}

// The columns of a pass: x is N x k with leading dimension ldx and y is M x k with ldy, in elements; one vector is
// k = kc = ldx = ldy = 1.  They travel in blocks of kc columns: the device holds one block of x (and of y when y is
// staged) at a time, with leading dimension kc.
struct HostCols {
    int k = 1, kc = 1;
    long long ldx = 1, ldy = 1;
};

// rows x cols elements between two row-major blocks: one 1-D copy when both are contiguous, one 2-D copy otherwise
template <class V>
static int copy_rows(V *dst, long long ldd, const V *src, long long lds, int cols, long long rows, cudaMemcpyKind kind,
                     cudaStream_t stream) {
    if (ldd == cols && lds == cols)
        SPMV_TRY_CUDA(cudaMemcpyAsync(dst, src, (size_t)rows * cols * sizeof(V), kind, stream));
    else
        SPMV_TRY_CUDA(cudaMemcpy2DAsync(dst, (size_t)ldd * sizeof(V), src, (size_t)lds * sizeof(V), (size_t)cols * sizeof(V),
                                        (size_t)rows, kind, stream));
    return SPMV_B200_OK;
}

// The pass itself.  launch(w, y_base, ld, cols) enqueues the kernel(s) of window w on p->compute for the `cols` columns
// of the current block (x staged at d_x with leading dimension kc); they write row r, column c of the block to
// y_base[r * ld + c].  zero_copy_ok: every element is written exactly once and never read back by the kernels of this
// path.  tail(y_base, ld, cols) runs after the last window of a block (the CSR long rows); the downloads of the windows
// flagged in p->tail_window wait for it.  piece: the W upload pieces of a block, in rows of x.
template <class V, class Launch, class Tail>
static int run_pipeline(HostPipe *p, long long M, long long N, const V *x, V *y, V *d_x, V *d_y, bool accumulate,
                        bool zero_copy_ok, const std::vector<long long> &piece, const HostCols &c, Launch launch, Tail tail) {
    const int W = p->windows;
    V *y_alias = zero_copy_alias(zero_copy_ok, accumulate, M, y);
    const bool tails = !p->tail_window.empty();
    for (int c0 = 0; c0 < c.k; c0 += c.kc) {
        const int cw = std::min(c.kc, c.k - c0);
        const bool first = c0 == 0, more = c0 + c.kc < c.k;
        V *y_base = y_alias ? y_alias + c0 : d_y;
        const long long ld_y = y_alias ? c.ldy : c.kc;
        // (1) uploads: the old y first (accumulate), then x in W chunks.  A later block overwrites the staging of the
        // previous one: its x waits for that block's last kernel, its old y for that block's downloads.
        if (!first) SPMV_TRY_CUDA(cudaStreamWaitEvent(p->up, p->x_free, 0));
        if (accumulate && M) {
            if (!first) SPMV_TRY_CUDA(cudaStreamWaitEvent(p->up, p->y_free, 0));
            SPMV_TRY(copy_rows(d_y, c.kc, y + c0, c.ldy, cw, M, cudaMemcpyHostToDevice, p->up));
            SPMV_TRY_CUDA(cudaEventRecord(p->y_landed, p->up));
        }
        // piece w of x ends where window w's columns end; a window that needs nothing new reuses the previous event.
        // Columns no window references are never uploaded.
        std::vector<int> gate(W, -1);
        long long at = 0;
        int last = -1;
        for (int w = 0; w < W; ++w) {
            const long long upto = std::min(N, piece[w]);
            if (upto > at) {
                SPMV_TRY(copy_rows(d_x + at * c.kc, c.kc, x + at * c.ldx + c0, c.ldx, cw, upto - at, cudaMemcpyHostToDevice, p->up));
                SPMV_TRY_CUDA(cudaEventRecord(p->landed[w], p->up));
                last = w;
                at = upto;
            }
            gate[w] = last;
        }
        // (2) products: window w waits for its piece (and a later block's first window for the staged y to be free)
        for (int w = 0; w < W; ++w) {
            if (!first && !y_alias && w == 0) SPMV_TRY_CUDA(cudaStreamWaitEvent(p->compute, p->y_free, 0));
            if (accumulate && M && w == 0) SPMV_TRY_CUDA(cudaStreamWaitEvent(p->compute, p->y_landed, 0));
            if (gate[w] >= 0 && (w == 0 || gate[w] != gate[w - 1])) SPMV_TRY_CUDA(cudaStreamWaitEvent(p->compute, p->landed[gate[w]], 0));
            SPMV_TRY(launch(w, y_base, ld_y, cw));
            if (!y_alias && !(tails && p->tail_window[w])) SPMV_TRY_CUDA(cudaEventRecord(p->done[w], p->compute));
        }
        SPMV_TRY(tail(y_base, ld_y, cw));
        for (int w = 0; tails && !y_alias && w < W; ++w)
            if (p->tail_window[w]) SPMV_TRY_CUDA(cudaEventRecord(p->done[w], p->compute));
        if (more) SPMV_TRY_CUDA(cudaEventRecord(p->x_free, p->compute));
        // (3) downloads, window by window, those the tail writes into last (none when the kernels wrote into the host
        // buffer themselves)
        for (int pass = 0; pass < (tails ? 2 : 1) && !y_alias; ++pass)
            for (int w = 0; w < W; ++w) {
                const long long r0 = p->row[w], r1 = p->row[w + 1];
                if (r1 <= r0 || (tails && p->tail_window[w] != pass)) continue;
                SPMV_TRY_CUDA(cudaStreamWaitEvent(p->down, p->done[w], 0));
                SPMV_TRY(copy_rows(y + r0 * c.ldy + c0, c.ldy, d_y + r0 * c.kc, c.kc, cw, r1 - r0, cudaMemcpyDeviceToHost, p->down));
            }
        if (more && !y_alias) SPMV_TRY_CUDA(cudaEventRecord(p->y_free, p->down));
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

template <class V>
static int no_tail(V *, long long, int) { return SPMV_B200_OK; }

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

// ---- multi-vector products Y = A X on host buffers ------------------------------------------------------------------
constexpr long long kSpmmPieceBytes = 256LL << 10;  // upload pieces end on 256 KB of the staged block, as for one vector

// Y straight into the caller's pinned buffer (zero-copy) or staged and downloaded window by window.  Measured with
// tools/spmm_host_bench.py --sweep-only on a build where this returns true, both ways in every cell (B200 at 1000 W,
// profiles/r03j_spmm_host_y_sweep.json; DESIGN.md section 3, "Host buffers"), minima of 7 calls:
//   * ldy > k: the 2-D downloads lose to the kernels' stores from 32 bytes a row (lap2d 4096^2 CSR k = 8, ldy = 11:
//     39.2 against 55.9 ms) and are as fast or slower below; at 256 bytes zero-copy is 2-3 % slower on lap2d only;
//   * ldy = k: zero-copy is faster at 8 bytes a row everywhere, at 16 on uniform and R-MAT (lap2d: 2.9 % slower), and
//     from 32 bytes the 1-D downloads are faster on lap2d (k = 32: 91.1 against 102.6 ms) and uniform (3.5-5.5 %) while
//     R-MAT gains 0.5-6 % from zero-copy.
static bool spmm_zero_copy(int k, long long ldy, size_t elem) { return ldy != k || (size_t)k * elem <= 16; }

// The window plan of the multi-vector products (rows for CSR, hacks for HLL), made once per handle and kept apart from
// the single-vector plan, so that alternating the two entry points never plans again.  SPMV_B200_HOST_WINDOWS is read
// here: a changed setting takes effect on a fresh handle.
static int spmm_plan_csr(spmv_b200_csr *A) {
    HostPipe *p = A->spmm_pipe;
    const std::vector<long long> bounds = window_rows(A->M, A->N, A->M);
    p->unit.clear();
    p->row.clear();
    std::vector<long long> elem;
    for (size_t w = 0; w < bounds.size(); ++w) {
        const int row = (int)bounds[w];
        if (!p->unit.empty() && row <= p->unit.back() && w + 1 != bounds.size()) continue;  // an empty window
        int off = 0;
        SPMV_TRY_CUDA(cudaMemcpy(&off, A->row_ptr + row, sizeof off, cudaMemcpyDeviceToHost));
        p->unit.push_back(row);
        p->row.push_back(row);
        elem.push_back(off);
    }
    const int W = (int)p->unit.size() - 1;
    p->windows = W;
    p->tail_window.clear();
    if (A->num_long > 0) {  // the windows whose downloads wait for the long rows
        std::vector<int> long_rows((size_t)A->num_long);
        SPMV_TRY_CUDA(cudaMemcpy(long_rows.data(), A->long_rows, long_rows.size() * sizeof(int), cudaMemcpyDeviceToHost));
        p->tail_window.assign((size_t)W, 0);
        for (int r : long_rows)
            p->tail_window[std::upper_bound(p->row.begin(), p->row.end(), (long long)r) - p->row.begin() - 1] = 1;
    }
    SPMV_TRY(plan_needs(p, A->col_idx, elem));
    p->path = 0;
    return SPMV_B200_OK;
}

static int spmm_plan_hll(spmv_b200_hll *H) {
    HostPipe *p = H->spmm_pipe;
    const std::vector<long long> bounds = window_rows(H->M, H->N, H->num_hacks);
    p->unit.clear();
    p->row.clear();
    std::vector<long long> elem;
    for (size_t w = 0; w < bounds.size(); ++w) {
        const int hack = w + 1 == bounds.size() ? H->num_hacks : (int)(bounds[w] / HACK_SIZE);
        if (!p->unit.empty() && hack <= p->unit.back() && w + 1 != bounds.size()) continue;
        p->unit.push_back(hack);
        p->row.push_back(std::min<long long>((long long)hack * HACK_SIZE, H->M));
        elem.push_back(H->host_off[hack]);
    }
    p->windows = (int)p->unit.size() - 1;
    SPMV_TRY(plan_needs(p, H->JA, elem));
    p->path = 0;
    return SPMV_B200_OK;
}

// The device staging of a k-column product: all k columns of X (and of Y when it is staged) when they fit half of the
// free device memory, else blocks of kc columns that do (SPMV_B200_HOST_SPMM_COLS forces kc).  Kept on the handle, grown
// as needed and freed with it.
template <class V>
static int spmm_stage(HostPipe *p, long long M, long long N, int k, bool stage_y, int *kc, V **d_x, V **d_y) {
    size_t free_bytes = 0, total_bytes = 0;
    SPMV_TRY_CUDA(cudaMemGetInfo(&free_bytes, &total_bytes));
    const size_t budget = (free_bytes + p->stage_bytes) / 2;
    const size_t per_col = (size_t)(N + (stage_y ? M : 0)) * sizeof(V);
    int cols = k;
    if (per_col > 0 && per_col * (size_t)k > budget) cols = (int)std::max<size_t>(1, budget / per_col);
    const int forced = env_int("SPMV_B200_HOST_SPMM_COLS", 0);
    if (forced > 0) cols = std::min(k, forced);
    const size_t x_bytes = ((size_t)N * cols * sizeof(V) + 255) / 256 * 256;
    const size_t bytes = std::max<size_t>(1, x_bytes + (stage_y ? (size_t)M * cols * sizeof(V) : 0));
    if (bytes > p->stage_bytes) {
        cudaFree(p->stage);
        p->stage = nullptr;
        p->stage_bytes = 0;
        SPMV_TRY_CUDA(cudaMalloc(&p->stage, bytes));
        p->stage_bytes = bytes;
    }
    *kc = cols;
    *d_x = static_cast<V *>(p->stage);
    *d_y = reinterpret_cast<V *>(static_cast<char *>(p->stage) + x_bytes);
    return SPMV_B200_OK;
}

// The pass over the columns: staging, pieces aligned in bytes of the staged block, then run_pipeline.
template <class V, class Launch, class Tail>
static int spmm_host_pass(HostPipe *p, long long M, long long N, int k, const V *X, long long ldx, V *Y, long long ldy,
                          bool accumulate, Launch launch, Tail tail) {
    const bool zero_copy_ok = spmm_zero_copy(k, ldy, sizeof(V));
    const bool stage_y = zero_copy_alias(zero_copy_ok, accumulate, M, Y) == nullptr;
    int kc = 0;
    V *d_x = nullptr, *d_y = nullptr;
    SPMV_TRY(spmm_stage(p, M, N, k, stage_y, &kc, &d_x, &d_y));
    const std::vector<long long> piece = pieces_of(p, N, std::max<long long>(1, kSpmmPieceBytes / ((long long)kc * (long long)sizeof(V))));
    const HostCols c{k, kc, ldx, ldy};
    const int rc = run_pipeline(p, M, N, X, Y, d_x, d_y, accumulate, zero_copy_ok, piece, c,
                                [&](int w, V *y_base, long long ld, int cols) { return launch(w, d_x, (long long)kc, y_base, ld, cols); },
                                [&](V *y_base, long long ld, int cols) { return tail(d_x, (long long)kc, y_base, ld, cols); });
    if (rc != SPMV_B200_OK) abort_pipeline(p);
    return rc;
}

template <class V>
static int csr_spmm_host(const char *what, spmv_b200_csr *A, int k, const V *X, long long ldx, V *Y, long long ldy, int accumulate) {
    SPMV_TRY(check_spmm_args(what, A, k, X, ldx, Y, ldy));
    if (k == 0 || A->M == 0) return SPMV_B200_OK;
    if (sizeof(V) == 4) {  // the float copy is made on the NULL stream; the non-blocking streams of the pass do not wait for it
        SPMV_TRY(spmv_b200_csr_enable_f32(A, nullptr));
        SPMV_TRY_CUDA(cudaStreamSynchronize(nullptr));
    }
    const V *values = sizeof(V) == 4 ? (const V *)A->values32 : (const V *)A->values;
    if (!A->spmm_pipe) SPMV_TRY(pipe_create(&A->spmm_pipe));
    HostPipe *p = A->spmm_pipe;
    if (p->path < 0) SPMV_TRY(spmm_plan_csr(A));
    return spmm_host_pass(p, A->M, A->N, k, X, ldx, Y, ldy, accumulate != 0,
        [&](int w, const V *d_x, long long ld_x, V *y_base, long long ld_y, int cols) {
            return csr_spmm_rows(A, values, p->unit[w], p->unit[w + 1], cols, d_x, ld_x, y_base, ld_y, accumulate, p->compute);
        },
        [&](const V *d_x, long long ld_x, V *y_base, long long ld_y, int cols) {
            return csr_spmm_long(A, values, cols, d_x, ld_x, y_base, ld_y, accumulate, p->compute);
        });
}

template <class V>
static int hll_spmm_host(const char *what, spmv_b200_hll *H, int k, const V *X, long long ldx, V *Y, long long ldy) {
    SPMV_TRY(check_spmm_args(what, H, k, X, ldx, Y, ldy));
    if (k == 0 || H->M == 0 || H->num_hacks == 0) return SPMV_B200_OK;
    if (sizeof(V) == 4) {  // the float copy is made on the NULL stream; the non-blocking streams of the pass do not wait for it
        SPMV_TRY(spmv_b200_hll_enable_f32(H, nullptr));
        SPMV_TRY_CUDA(cudaStreamSynchronize(nullptr));
    }
    const V *AS = sizeof(V) == 4 ? (const V *)H->AS32 : (const V *)H->AS;
    if (!H->spmm_pipe) SPMV_TRY(pipe_create(&H->spmm_pipe));
    HostPipe *p = H->spmm_pipe;
    if (p->path < 0) SPMV_TRY(spmm_plan_hll(H));
    return spmm_host_pass(p, H->M, H->N, k, X, ldx, Y, ldy, false,
        [&](int w, const V *d_x, long long ld_x, V *y_base, long long ld_y, int cols) {
            return hll_spmm_hacks(H, AS, p->unit[w], p->unit[w + 1], cols, d_x, ld_x, y_base, ld_y, p->compute);
        },
        [](const V *, long long, V *, long long, int) { return SPMV_B200_OK; });
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
    const int rc = run_pipeline(p, A->M, x ? A->N : 0, x, y, A->stage_x, A->stage_y, accumulate != 0, zero_copy_ok, p->piece, HostCols{},
                                [&](int w, double *y_base, long long, int) {
        return csr_launch_window(A, path, p->unit[w], p->unit[w + 1], A->stage_x, y_base, accumulate, p->compute);
    }, no_tail<double>);
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
    const int rc = run_pipeline(p, H->M, x ? H->N : 0, x, y, H->stage_x, H->stage_y, false, true, p->piece, HostCols{},
                                [&](int w, double *y_base, long long, int) {
        return hll_launch_window(H, path, p->unit[w], p->unit[w + 1], H->stage_x, y_base, p->compute);
    }, no_tail<double>);
    if (rc != SPMV_B200_OK) abort_pipeline(p);
    return rc;
}

int spmv_b200_csr_spmm_host(spmv_b200_csr *A, int k, const double *X, long long ldx, double *Y, long long ldy, int accumulate) {
    return csr_spmm_host("csr_spmm_host", A, k, X, ldx, Y, ldy, accumulate);
}

int spmv_b200_hll_spmm_host(spmv_b200_hll *H, int k, const double *X, long long ldx, double *Y, long long ldy) {
    return hll_spmm_host("hll_spmm_host", H, k, X, ldx, Y, ldy);
}

int spmv_b200_csr_spmm_host_f32(spmv_b200_csr *A, int k, const float *X, long long ldx, float *Y, long long ldy, int accumulate) {
    return csr_spmm_host("csr_spmm_host_f32", A, k, X, ldx, Y, ldy, accumulate);
}

int spmv_b200_hll_spmm_host_f32(spmv_b200_hll *H, int k, const float *X, long long ldx, float *Y, long long ldy) {
    return hll_spmm_host("hll_spmm_host_f32", H, k, X, ldx, Y, ldy);
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
