// handles.cuh -- the opaque handle types of include/spmv_b200.h (internal layout).
#pragma once

#include <type_traits>
#include <vector>

#include "common.cuh"

namespace spmv {

constexpr int kDefaultTileItems = 12288;    // D: 4-byte stream words per CSR tile (3 per nonzero + 1 per row) = 48 KB
constexpr int kDefaultLongThreshold = 512;  // L: longer rows leave the tile kernels
constexpr int kDefaultStages = 2;           // TMA pipeline depth of the stream kernels
constexpr int kHllTileSlots = 3072;         // D_h: slots + rows per HLL tile (12 B per slot; stage = 49.5 KB with the wide margin)
constexpr int kHllWideSlots = 1024;         // hacks with more slots (MAXNZ > 32) are processed straight from HBM

// Optional walk order of the fused row kernels (SPMV_B200_FUSED_BOUNDARY_FIRST=1): the 256-row chunks that hold rows a
// neighbour references come FIRST, so that their NVLink peer stores are long acknowledged when the launch ends.
// Measured neutral on 2 GPUs (1.155 vs 1.156 ms per iteration, row kernel 1.263 vs 1.265: profiles/r02d_*): the 20-50 us
// the peer stores cost are not an end-of-launch wait.  Off by default; the asynchronous form always uses it.
// Chunk = 256 consecutive rows.
struct ChunkOrder {
    int count = 0;                  // boundary intervals (ascending, disjoint), in chunks
    int lo[SPMV_B200_MAX_PEERS] = {}, hi[SPMV_B200_MAX_PEERS] = {};
    int boundary_chunks = 0;        // sum of the interval lengths; 0 = natural order
};

__device__ __forceinline__ int ordered_chunk(const ChunkOrder &o, int q) {  // q-th chunk of the walk -> row chunk
    if (o.boundary_chunks == 0) return q;
    if (q < o.boundary_chunks) {
        int left = q;
        for (int i = 0; i < o.count; ++i) {
            const int len = o.hi[i] - o.lo[i];
            if (left < len) return o.lo[i] + left;
            left -= len;
        }
        return q;
    }
    int chunk = q - o.boundary_chunks;
    for (int i = 0; i < o.count; ++i)
        if (chunk >= o.lo[i]) chunk += o.hi[i] - o.lo[i];
    return chunk;
}

struct Epilogue {                 // optional fused tail of the CSR stream / row kernels and the HLL row kernel
    const double *prev_sumsq = nullptr;  // divide every row by sqrt(*prev_sumsq)
    const double *inv_norm = nullptr;    // FLAT form: multiply every row by *inv_norm (1/|w_prev|, computed ONCE by the exchange
                                         // kernel: a square root and a division per thread cost a flat CTA a quarter of its time)
    double *partials = nullptr;   // partials[blockIdx.x] = sum of the squares of the rows this CTA produced
    int partials_total = 0;       // size of the caller's buffer (spmv_b200_csr_partials_count): CTA 0 zeroes the entries
                                  // [gridDim.x, partials_total) so that a caller may always sum the whole buffer
    spmv_b200_peers_t peers = {}; // rows mirrored into peer memory
    spmv_b200_mail_t mail = {};   // world > 0: |w|^2 travels through peer mailboxes instead of prev_sumsq (spmv_b200.h)
    ChunkOrder order;             // row kernels only: boundary chunks first (filled by boundary_first_order)
};

// the peers of a fused launch on M rows: a count in [0, SPMV_B200_MAX_PEERS] and row ranges 0 <= lo <= hi <= M (a range
// that reaches past the matrix would silently leave rows out of a neighbour's x); NULL = none (host side)
int check_peers(const spmv_b200_peers_t *peers, int M, const char *what);
// the union of the peers' row ranges in 256-row chunks, ascending and disjoint (host side; peers passed check_peers)
int boundary_first_order(const spmv_b200_peers_t &peers, int M, ChunkOrder &order);

// entries of the partials buffer that this launch does not write (the buffer is sized for the largest fused grid)
__device__ __forceinline__ void zero_partials_tail(const Epilogue &ep) {
    if (blockIdx.x == 0 && ep.partials != nullptr)
        for (int i = (int)gridDim.x + (int)threadIdx.x; i < ep.partials_total; i += (int)blockDim.x) ep.partials[i] = 0.0;
}

// ---- the fused tail of the iterated product, shared by csr_row_fused_kernel (csr.cu) and hll_row_fused_kernel (hll.cu):
// 256 threads per CTA, thread t of a CTA owns row chunk*256 + t of every chunk the CTA walks, so both formats produce
// the same per-CTA partial sums in the same order (bitwise equal |w|^2 for the same partition). ----
// start of a launch: 1/|w_prev| (from the mailbox, or from *prev_sumsq, or 1)
__device__ __forceinline__ double fused_inv_norm(const Epilogue &ep, bool &scaled, double *mail_total_smem) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    scaled = false;
    double prev_norm = 1.0;
    if (ep.inv_norm != nullptr) {
        scaled = true;
        zero_partials_tail(ep);
        return __ldg(ep.inv_norm);
    }
    if (ep.mail.world > 0) {
        if (ep.mail.iteration > 0) {
            if (warp == 0) {
                const double total = mail_wait_total(ep.mail, lane);
                if (lane == 0) *mail_total_smem = total;
            }
            __syncthreads();
            scaled = true;
            prev_norm = sqrt(*mail_total_smem);
        }
    } else if (ep.prev_sumsq != nullptr) {
        scaled = true;
        prev_norm = sqrt(*ep.prev_sumsq);
    }
    zero_partials_tail(ep);
    return 1.0 / prev_norm;  // one division per thread, one multiplication per row (1 ulp from a division)
}

// does any peer reference a row of the 256-row chunk that starts at chunk_lo?  (CTA-uniform)
__device__ __forceinline__ bool fused_chunk_is_boundary(const Epilogue &ep, long long chunk_lo) {
    bool boundary = false;
    for (int p = 0; p < ep.peers.count; ++p) boundary |= chunk_lo < ep.peers.hi[p] && chunk_lo + 256 > ep.peers.lo[p];
    return boundary;
}

__device__ __forceinline__ void fused_peer_store(const Epilogue &ep, long long row, double v) {
    for (int p = 0; p < ep.peers.count; ++p)
        if (row >= ep.peers.lo[p] && row < ep.peers.hi[p]) ep.peers.dst[p][row] = v;
}

// end of a launch: per-CTA partial of the squares (fixed order); with a mailbox the last CTA publishes the rank's sum
__device__ __forceinline__ void fused_finish(const Epilogue &ep, double sq, double *warp_sq_smem) {
    if (ep.partials == nullptr) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, off);
    if (lane == 0) warp_sq_smem[warp] = sq;
    __syncthreads();  // every row of this CTA (local and peer stores) is issued: a device-scope fence by thread 0 (cumulative
    if (warp == 0) {  // through the barrier) orders them before the counter and, through it, before the last CTA's sys release
        unsigned int arrived = 0;
        if (lane == 0) {
            double total = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) total += warp_sq_smem[w];
            ep.partials[blockIdx.x] = total;
            if (ep.mail.world > 0) {
                __threadfence();  // device scope; the system-scope fence is paid once, by the CTA that publishes (mail_publish)
                arrived = atomicAdd(ep.mail.counter, 1u);
            }
        }
        if (ep.mail.world > 0) {
            arrived = __shfl_sync(0xffffffffu, arrived, 0);
            if (arrived == gridDim.x - 1) mail_publish(ep.mail, ep.partials, (int)gridDim.x, lane);
        }
    }
}

constexpr int kBins = 7;  // rows binned by length: 1, 2, 4, 8, 16, 32 lanes per row, and "long" (split into fragments)

struct BinPlan {                 // csr.cu: row-binned vector kernel for skewed matrices (built on first use)
    int *rows = nullptr;         // device [M]: row ids sorted by bin, ascending inside a bin
    int offset[kBins + 1] = {};  // rows of bin b are rows[offset[b] .. offset[b+1])
    int block_start[kBins] = {}; // first CTA of bins 0..5 in the single launch; block_start[6] = total CTAs
    int num_long = 0;            // rows of the last bin
    int *frag_first = nullptr;   // device [num_long+1]
    int num_frag = 0;
    double *frag_partial = nullptr;
    bool built = false;
};

struct HostPipe;  // hostpath.cu: streams, events and the row-window plan of the *_spmv_host / *_spmm_host entry points
void host_pipe_free(HostPipe *p);

struct HllTile {      // tiles[t] = first hack of tile t and its first slot; tiles[num_tiles] = {num_hacks, slots}
    int hack;
    int pad;
    long long slot;
};


// Times launch(i) for candidates i = 0 .. n-1 on scratch vectors and returns the fastest index (plan time, large matrices)
// fastest_out (n entries, optional): each candidate's best time in ms, < 0 where it could not be timed
template <class Launch>
int tune_candidates(long long M, long long N, int n, int fallback, cudaStream_t stream, Launch launch,
                    float *fastest_out = nullptr) {
    // ROUNDS passes over all candidates, REPS launches each, the MINIMUM per candidate decides: a transient slowdown of the
    // GPU (power capping under sustained load shifts timings by 10 % for seconds) then cannot favour whichever candidate
    // happened to run in a quiet moment -- round 2 saw a one-pass tuner pick a 25 % slower kernel at the end of bench.py.
    constexpr int ROUNDS = 3, REPS = 3;
    double *x = nullptr, *y = nullptr;
    cudaEvent_t a = nullptr, b = nullptr;
    int best = fallback;
    for (int i = 0; fastest_out && i < n; ++i) fastest_out[i] = -1.0f;
    if (n > 0 && cudaMalloc(&x, (size_t)(N > 0 ? N : 1) * sizeof(double)) == cudaSuccess &&
        cudaMalloc(&y, (size_t)(M > 0 ? M : 1) * sizeof(double)) == cudaSuccess &&
        cudaMemsetAsync(x, 0, (size_t)(N > 0 ? N : 1) * sizeof(double), stream) == cudaSuccess &&
        cudaEventCreate(&a) == cudaSuccess && cudaEventCreate(&b) == cudaSuccess) {
        std::vector<float> fastest((size_t)n, -1.0f);
        bool ok = true;
        for (int round = 0; round < ROUNDS && ok; ++round) {
            for (int i = 0; i < n && ok; ++i) {
                if (round == 0) ok = launch(i, x, y) == SPMV_B200_OK;  // warm-up
                ok = ok && cudaEventRecord(a, stream) == cudaSuccess;
                for (int rep = 0; rep < REPS && ok; ++rep) ok = launch(i, x, y) == SPMV_B200_OK;
                ok = ok && cudaEventRecord(b, stream) == cudaSuccess && cudaEventSynchronize(b) == cudaSuccess;
                float ms = 0.0f;
                ok = ok && cudaEventElapsedTime(&ms, a, b) == cudaSuccess;
                if (ok && (fastest[i] < 0.0f || ms < fastest[i])) fastest[i] = ms;
            }
        }
        for (int i = 0; fastest_out && ok && i < n; ++i) fastest_out[i] = fastest[i];
        if (ok) {
            float best_ms = -1.0f;
            for (int i = 0; i < n; ++i)
                if (fastest[i] >= 0.0f && (best_ms < 0.0f || fastest[i] < best_ms)) {
                    best_ms = fastest[i];
                    best = i;
                }
        }
    }
    cudaGetLastError();
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
    cudaFree(x);
    cudaFree(y);
    return best;
}

struct CsrImage;  // image.cu: the private image of a CSR handle
}  // namespace spmv

struct spmv_b200_csr {
    int M = 0, N = 0;
    long long nnz = 0;
    int *row_ptr = nullptr;
    int *col_idx = nullptr;
    double *values = nullptr;
    float *values32 = nullptr;  // fp32 copy of the values (spmv_b200_csr_enable_f32): fp32 storage, fp64 arithmetic
    bool owns = false;
    // plan (shared by the tile kernel and the TMA stream kernel)
    int tile_items = spmv::kDefaultTileItems;
    int long_threshold = spmv::kDefaultLongThreshold;
    int forced_tpr = 0;
    int num_tiles = 0;
    int2 *tiles = nullptr;
    int num_long = 0;
    int *long_rows = nullptr;
    int *frag_first = nullptr;
    int num_frag = 0;
    double *frag_partial = nullptr;
    // spmv_b200_csr_spmm: num_frag x 32 partial sums of the long rows for one column tile, allocated by the first product
    // that needs it and freed with the plan (replan changes num_frag); like frag_partial it makes products on one handle
    // stream-ordered
    mutable double *spmm_partial = nullptr;
    spmv::BinPlan bins;
    int max_row = 0;     // longest row (plan time)
    int row_batch = 4;   // csr_row_kernel: column/value/gather batch per thread (tuned at plan time on large matrices)
    int row_batch32 = 4; // the same for fp32 storage (tuned by spmv_b200_csr_enable_f32)
    bool short_rows_stream = false;  // plan-time timing found the stream kernel faster than every row-kernel batch
    int fused_batch = 0;             // fused iterated product: 0 = fused stream kernel, else batch of the fused row kernel
    int flat_batch = 4;              // the FLAT fused row kernel (two-launch iterated product), timed at plan time
    // stream kernel launch shape
    int stages = spmv::kDefaultStages;
    int consumers = 12;
    int stream_grid = 0;
    // private image of the matrix (image.cu), column-major or patterns: held only when plan-time timing found it faster
    // (or set_image asked for it); owned arrays only, dropped by remap_columns
    spmv::CsrImage *image = nullptr;
    // staging vectors of the *_host entry points
    double *stage_x = nullptr;
    double *stage_y = nullptr;
    spmv::HostPipe *pipe = nullptr;
    spmv::HostPipe *spmm_pipe = nullptr;  // the *_spmm_host entry points: their own windows and staging (hostpath.cu)
};

namespace spmv {
// Runs of hacks of equal width (regular ELLPACK regions): hacks [begin[s], begin[s+1]) have `width[s]` columns and hack h
// of the run starts at slot base[s] + (h - begin[s]) * 32 * width[s] -- the offset by arithmetic, without the hack_off
// load (hll_rowu_kernel).  count = 0: the image has more than kMaxHllSegments runs, the kernel is not offered.
constexpr int kMaxHllSegments = 8;
struct HllSegments {
    int count = 0;
    int begin[kMaxHllSegments + 1] = {};
    int width[kMaxHllSegments] = {};
    long long base[kMaxHllSegments] = {};
};
}  // namespace spmv

struct spmv_b200_hll {
    int M = 0, N = 0, num_hacks = 0, max_width = 0;
    spmv::HllSegments segments;     // from host_off at plan time (hll_pick_row_batch)
    long long slots = 0, ref_slots = 0;
    long long *hack_off = nullptr;  // device [num_hacks+1]
    int *JA = nullptr;              // device [slots]
    double *AS = nullptr;           // device [slots]
    float *AS32 = nullptr;          // fp32 copy of AS (spmv_b200_hll_enable_f32)
    std::vector<long long> host_off;
    // stream kernel plan
    int tile_slots = spmv::kHllTileSlots;
    int wide_slots = spmv::kHllWideSlots;
    int stages = spmv::kDefaultStages;
    int consumers = 12;
    int num_tiles = 0;
    spmv::HllTile *tiles = nullptr;
    int stream_grid = 0;
    int row_batch = 4;   // hll_row_kernel batch (tuned at plan time on large matrices)
    int row_form = 0;    // fp64 row path: 0 = hll_row_kernel<row_batch>; 64 + b = hll_rowu_kernel<b> (regular images, timed at plan time)
    int row_batch32 = 4; // the same for fp32 storage (tuned by spmv_b200_hll_enable_f32)
    int fused_batch = 0; // hll_row_fused_kernel batch (tuned at plan time; 0 = row_batch)
    int flat_batch = 4;  // the FLAT form of hll_row_fused_kernel (two-launch iterated product)
    bool narrow_stream = false;  // plan-time timing found the stream kernel faster than every row-kernel batch
    double *stage_x = nullptr;
    double *stage_y = nullptr;
    spmv::HostPipe *pipe = nullptr;
    spmv::HostPipe *spmm_pipe = nullptr;  // the *_spmm_host entry points: their own windows and staging (hostpath.cu)
};

namespace spmv {
// stream.cu
int stream_prepare_csr(spmv_b200_csr *A);
// tile_count < 0: every tile; otherwise the tiles [tile_begin, tile_begin + tile_count) only
int stream_launch_csr(const spmv_b200_csr *A, const double *x, double *y, int accumulate, const Epilogue *ep,
                      cudaStream_t stream, int tile_begin = 0, int tile_count = -1);
int stream_plan_hll(spmv_b200_hll *H, cudaStream_t stream);
int stream_launch_hll(const spmv_b200_hll *H, const double *x, double *y, cudaStream_t stream, int tile_begin = 0,
                      int tile_count = -1);
// csr.cu / hll.cu: which kernel the automatic choice resolves to, and launches restricted to a window
enum CsrPath { kPathStream, kPathTile, kPathVector, kPathBinned, kPathRow, kPathImage };
constexpr int kRowKernelMaxLen = 12;  // AUTO: one thread per row when no row is longer than this (= kSerialRowMax: the
                                      // stream kernel then gives the same bits, so plan-time timing may pick either)
CsrPath csr_resolve(const spmv_b200_csr *A, int algo);
int csr_launch_window(const spmv_b200_csr *A, CsrPath path, int unit_begin, int unit_end, const double *x, double *y,
                      int accumulate, cudaStream_t stream);  // units: tiles (stream/tile paths) or rows (vector path)
enum HllPath { kHllSlice = 0, kHllStream = 1, kHllRows = 2 };
HllPath hll_resolve(const spmv_b200_hll *H);
int hll_launch_window(const spmv_b200_hll *H, HllPath path, int unit_begin, int unit_end, const double *x, double *y,
                      cudaStream_t stream);  // units: tiles (stream kernel) or hacks (slice and row kernels)
int env_int(const char *name, int fallback);
// hll.cu: the column-major layout, its fill and the masked kernels, for spmv_b200_hll_from_csr and the private image of a
// CSR handle (image.cu).  hll_layout: the hack widths of M rows, scanned into hack_off (device [num_hacks + 1], allocated
// here), its host copy, the widest hack and, unless narrow is NULL, whether every slot fits the image's narrow column
// field (col - row within 2^14, padding included).  The column field is JA, or JA16 (the narrow field) when that is not
// NULL.  hll_fill fills it and each value stream that is not NULL: fp64 (AS), 1-byte codes into table[K] (AC); masked: a
// padding slot is marked as such (always so in the narrow field).  hll_masked_launch: y = A x (or y += A x) over hacks
// [hack_begin, hack_end) by the masked hll_rowu_kernel<batch> (offset_free; regular layouts) or hll_row_kernel<batch>,
// on the codes when AC is not NULL (K >= 1), else on AS.
int hll_layout(int M, int N, const int *row_ptr, const int *col_idx, cudaStream_t stream, long long **hack_off,
               std::vector<long long> &host_off, int *max_width, bool *narrow);
HllSegments hll_find_segments(const std::vector<long long> &host_off, int num_hacks);
int hll_fill(int M, int N, const int *row_ptr, const int *col_idx, const double *values, int num_hacks,
             const long long *hack_off, int *JA, uint16_t *JA16, double *AS, uint8_t *AC, const double *table, int K,
             bool masked, cudaStream_t stream);
int hll_masked_launch(int hack_begin, int hack_end, int M, const long long *hack_off, const HllSegments &seg, const int *JA,
                      const uint16_t *JA16, long long slots, const double *AS, const uint8_t *AC, const double *table, int K,
                      int batch, bool offset_free, int accumulate, const double *x, double *y, cudaStream_t stream);
// image.cu: the private image of a CSR handle.  Plan time (A owns its arrays and has no long rows: the plan checks):
// image_candidates builds every form A qualifies for and returns their number (*out NULL when none),
// image_launch_candidate multiplies scratch vectors with candidate i (y = A x over all rows), and image_keep holds
// candidate i and frees every other stream -- or image_free frees them all (and sets img to NULL).
int image_candidates(const spmv_b200_csr *A, cudaStream_t stream, CsrImage **out);
int image_launch_candidate(const CsrImage *img, int i, const double *x, double *y, cudaStream_t stream);
void image_keep(CsrImage *img, int i);
void image_free(CsrImage *&img);
// spmv_b200_csr_set_image modes 1 (column-major, fp64 values), 2 (column-major, value codes) and 3 (patterns): replaces
// A->image by that form unless it holds it already; on failure (also: arrays not owned, long rows) A->image stays
int image_build(spmv_b200_csr *A, int mode, cudaStream_t stream);
// the held form over rows [row_begin, row_end): the column-major form runs whole hacks (row_begin a multiple of 32), the
// pattern form any row range (image_any_rows)
int image_launch(const CsrImage *img, int row_begin, int row_end, const double *x, double *y, int accumulate,
                 cudaStream_t stream);
bool image_any_rows(const CsrImage *img);
void image_info(const CsrImage *img, spmv_b200_csr_info_t *info);  // the image_* fields (all 0 for NULL)
int hll_row_forms();                                             // hll.cu: forms of hll_rowm_kernel (spmv_b200_row_forms)
int hll_row_form(int index, int *hacks, int *batch, int *ctas);  // 0 = ok
int fused_ctas_per_sm();  // csr.cu: CTAs per SM in the grid of the fused row kernels (CSR and HLL use the same value)

// ---- persisting-L2 window on x (csr.cu) -------------------------------------------------------------------------
// Gather-bound products (uniform 32/row, R-MAT) re-read x from DRAM because the once-read matrix stream keeps pushing
// it out of L2 (ncu, round 1: DRAM traffic 1.4-1.6x the algorithmic bytes).  The launches of the gather-bound kernels
// therefore carry a per-launch access-policy window over x (cudaLaunchAttributeAccessPolicyWindow): hits are
// "persisting", the rest of the window "streaming"; the device's persisting carve-out (cudaLimitPersistingL2CacheSize)
// is raised once per device to its maximum.  hitRatio = 1 when x fits the carve-out, else carve-out / bytes, so the
// persisting lines never thrash among themselves.  SPMV_B200_L2_PERSIST=0 switches it off (plain launches).
struct XPolicy {
    cudaLaunchAttribute attr[1];
    unsigned int count = 0;
};
XPolicy x_policy(const void *x, size_t bytes);
XPolicy matrix_policy(const void *head, size_t bytes);  // head of a matrix array held in L2 across products (csr.cu)

template <typename... Params, typename... Args>
inline cudaError_t launch_x(void (*kernel)(Params...), unsigned int grid, unsigned int block, size_t smem,
                            cudaStream_t stream, const XPolicy &policy, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cfg.attrs = const_cast<cudaLaunchAttribute *>(policy.attr);
    cfg.numAttrs = policy.count;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<Params>(args)...);
}
// Returns f(std::integral_constant<int, B>{}) for the B of Bs equal to batch, or for Default when none is: a launch site
// names the batches its kernel is instantiated for and the one that any other batch runs.
template <int Default, int B, int... Bs, class F>
auto with_batch(int batch, F &&f) {
    if (batch == B) return f(std::integral_constant<int, B>{});
    if constexpr (sizeof...(Bs) == 0) return f(std::integral_constant<int, Default>{});
    else return with_batch<Default, Bs...>(batch, f);
}
// Times launch(candidate) for candidate = first .. 7 on scratch vectors and returns the fastest (plan time, large
// matrices).  Candidates 2..7 are batches of the row kernels; 0 (first = 0 only, 1 is skipped) stands for the stream kernel.
template <class Launch>
int tune_batch(long long M, long long N, int fallback, cudaStream_t stream, Launch launch, int first = 2) {
    int ids[8], n = 0;
    for (int batch = first; batch <= 7; ++batch)
        if (batch != 1) ids[n++] = batch;
    int fallback_index = 0;
    for (int i = 0; i < n; ++i)
        if (ids[i] == fallback) fallback_index = i;
    const int pick = tune_candidates(M, N, n, fallback_index, stream, [&](int i, double *x, double *y) { return launch(ids[i], x, y); });
    return ids[pick] == fallback || pick != fallback_index ? ids[pick] : fallback;
}

// spmm.cu: the multi-vector launches of a window (V = double, or float on the enable_f32 copy; X and Y at row 0 of the
// matrix, arguments checked by check_spmm_args).  csr_spmm_rows: rows [r0, r1), leaving out the plan's long rows;
// csr_spmm_long: those long rows; hll_spmm_hacks: hacks [h0, h1).
int check_spmm_args(const char *what, const void *h, int k, const void *X, long long ldx, const void *Y, long long ldy);
template <typename V>
int csr_spmm_rows(const spmv_b200_csr *A, const V *values, long long r0, long long r1, int k, const V *d_X, long long ldx,
                  V *d_Y, long long ldy, int accumulate, cudaStream_t stream);
template <typename V>
int csr_spmm_long(const spmv_b200_csr *A, const V *values, int k, const V *d_X, long long ldx, V *d_Y, long long ldy,
                  int accumulate, cudaStream_t stream);
template <typename V>
int hll_spmm_hacks(const spmv_b200_hll *H, const V *AS, int h0, int h1, int k, const V *d_X, long long ldx, V *d_Y,
                   long long ldy, cudaStream_t stream);
}  // namespace spmv
