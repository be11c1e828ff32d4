// stream.cu -- persistent, warp-specialized, TMA-pipelined SpMV kernels for sm_100a (CSR and HLL).
//
// Why (profiles/r01a_ncu_full_summary.md): the first tile kernel moves exactly the algorithmic
// bytes but reaches only 49 % of DRAM throughput -- every CTA serialises
// "load stream -> gather x -> barrier -> reduce", so too few bytes are in flight.  Here the matrix
// stream is decoupled from the arithmetic:
//   * a persistent grid (2 CTAs per SM) walks the plan's tiles round-robin;
//   * each CTA owns a ring of `stages` shared-memory buffers.  ONE PRODUCER WARP refills them with
//     bulk asynchronous copies (cp.async.bulk global -> shared, the 1-D form of TMA, SASS UBLKCP)
//     that complete on a "full" mbarrier (complete_tx::bytes), with an L2 evict-first policy so the
//     once-read stream does not push x out of L2; it only waits for the stage's "empty" mbarrier;
//   * the CONSUMER WARPS never synchronise with each other: each takes 32-row chunks of the staged
//     tile (lane = row), reads values / columns / row offsets out of shared memory -- where the
//     row-strided access pattern costs nothing -- gathers x through the read-only path and writes y
//     coalesced; when a warp is done with a stage it arrives on the stage's "empty" mbarrier.
// Shared memory per stage: values (8 B) + columns (4 B) per element, plus the tile's slice of row_ptr
// for CSR.
//
// CSR rows are reduced by one lane each (left to right, mul and add kept separate: bit-identical
// to the reference's serial loop, reference src/csr_matrix.c:134-138) or by 2..32 lanes with an
// xor-shuffle tree when a tile holds longer rows.  HLL hacks are reduced by one warp each, lane = row,
// walking the column-major slots j*32 + lane (conflict-free), sequentially in j: bit-identical to the
// reference's spmv_hll_serial (reference src/hll_matrix.c:294-306).
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "handles.cuh"

namespace spmv {

constexpr int kDefaultCsrConsumers = 12;  // consumer warps per CTA (+ one producer warp); tools/tune.py sweep, profiles/r01b
constexpr int kDefaultHllConsumers = 16;

// ---- mbarrier / bulk-copy primitives (PTX) ------------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE;\n"
        "bra LAB_WAIT;\n"
        "LAB_DONE:\n"
        "}\n" ::"r"(smem_addr(bar)),
        "r"(parity)
        : "memory");
}

__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_addr(dst)),
        "l"(src), "r"(bytes), "r"(smem_addr(bar)), "l"(policy)
        : "memory");
}

// sum_{k = lo, lo+step, ... < hi} v[k] * x[c[k]] with values/columns staged in shared memory; U gathers
// in flight, products and sums rounded separately and added in index order.
template <int U>
__device__ __forceinline__ double dot_staged(const double *sv, const int *sc, int lo, int hi, int step,
                                             const double *__restrict__ x, double acc) {
    int k = lo;
    for (; k + (U - 1) * step < hi; k += U * step) {
        double v[U], xv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = sv[k + u * step];
#pragma unroll
        for (int u = 0; u < U; ++u) xv[u] = ldg_x(x, sc[k + u * step]);
#pragma unroll
        for (int u = 0; u < U; ++u) acc = __dadd_rn(acc, __dmul_rn(v[u], xv[u]));
    }
    for (; k < hi; k += step) acc = __dadd_rn(acc, __dmul_rn(sv[k], ldg_x(x, sc[k])));
    return acc;
}

// sv[k] <- sv[k] * x[sc[k]] for k = lo + first, lo + first + step, ... < hi (first = lane, step = 32 for one warp;
// first = thread, step = all consumer threads for a whole CTA): conflict-free shared-memory accesses and U
// independent gathers per lane, whatever the row lengths.
template <int U>
__device__ __forceinline__ void products_staged(double *sv, const int *sc, int lo, int hi, int first, int step,
                                                const double *__restrict__ x) {
    // guarded batches: every pass issues its U column reads, then its U gathers, then the U products -- also for the
    // last, partial pass (a scalar remainder loop would serialise one gather latency per element)
    for (int k = lo + first; k < hi; k += U * step) {
        int c[U];
        double v[U], xv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) c[u] = k + u * step < hi ? sc[k + u * step] : -1;
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = c[u] >= 0 ? sv[k + u * step] : 0.0;
#pragma unroll
        for (int u = 0; u < U; ++u) xv[u] = c[u] >= 0 ? ldg_x(x, c[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (c[u] >= 0) sv[k + u * step] = __dmul_rn(v[u], xv[u]);
    }
}

// Sum of one row of products parked in shared memory by G lanes (G a power of two, the same in the whole warp;
// every lane of the warp must call this).  Lane `sub` of the group adds the elements e = sub (mod G) of its row.
// When G divides the row length the walk starts at element (c * row_id) mod len, c = (G - len) mod 16, and wraps:
// rows of equal length then start len + c = G (mod 16) doubles apart, i.e. the groups of a half-warp fall into
// distinct banks.  Rows longer than kLaneRowMax elements per lane are summed by the whole warp, one after the other.
// Fixed order (partial sums, then an xor tree): deterministic.  The sum is returned in every lane of the group.
__device__ __forceinline__ double group_row_sum(const double *prod, int lo, int hi, int G, int lane, int row_id) {
    const int len = hi - lo, sub = lane & (G - 1);
    const bool wide = len > kLaneRowMax * G;
    double acc = 0.0;
    if (len <= kSerialRowMax) {
        // short rows keep the serial order whatever path their tile takes (bit-identical to the reference's loop and
        // independent of how the rows are partitioned over tiles and GPUs); the other lanes of the group add +0.0
        if (sub == 0)
            for (int k = lo; k < hi; ++k) acc = __dadd_rn(acc, prod[k]);
    } else if (!wide) {
        int st = 0;
        if ((len & (G - 1)) == 0) st = (((G - len) & 15) * row_id) % len;
        for (int k = lo + st + sub; k < hi; k += G) acc = __dadd_rn(acc, prod[k]);
        for (int k = lo + sub; k < lo + st; k += G) acc = __dadd_rn(acc, prod[k]);
    }
    for (int off = G >> 1; off > 0; off >>= 1) acc = __dadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, off));
    unsigned pending = __ballot_sync(0xffffffffu, wide && sub == 0);
    while (pending) {
        const int owner = __ffs(pending) - 1;
        pending &= pending - 1;
        const int wlo = __shfl_sync(0xffffffffu, lo, owner), whi = __shfl_sync(0xffffffffu, hi, owner);
        double part = 0.0;
        for (int k = wlo + lane; k < whi; k += 32) part = __dadd_rn(part, prod[k]);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) part = __dadd_rn(part, __shfl_xor_sync(0xffffffffu, part, off));
        if ((lane & ~(G - 1)) == owner) acc = part;
    }
    return acc;
}

__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }


// =================================================================================================
// CSR
// =================================================================================================
template <int kConsumerWarps, bool kFused>
__global__ void __launch_bounds__((kConsumerWarps + 1) * 32, (kConsumerWarps >= 24 ? 1 : 2))
csr_stream_kernel(const int2 *__restrict__ tiles, int num_tiles, const int *__restrict__ row_ptr,
                  const int *__restrict__ col_idx, const double *__restrict__ values, const double *__restrict__ x,
                  double *__restrict__ y, int M, int nnz_total, int stage_bytes, int stages, int long_threshold,
                  int forced_tpr, int accumulate, const Epilogue ep) {
    // a stage is one packed pool: [values: cnt x 8 B][columns: cnt x 4 B][row_ptr slice: rcnt x 4 B]
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)stages * stage_bytes);
    uint64_t *empty = full + stages;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nnz_bulk = nnz_total & ~3;  // bulk copies never touch a partial 16-byte group at the array end
    const int rp_bulk = (M + 1) & ~3;
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumerWarps);
        }
        fence_mbar_init();
    }
    __syncthreads();
    // before the producer warp leaves: zero_partials_tail strides over every thread of the CTA
    if constexpr (kFused) zero_partials_tail(ep);

    if (warp == kConsumerWarps) {
        // ---------------- producer: one elected lane streams the CTA's tiles into the ring ----------------
        if (lane == 0) {
            const uint64_t policy = policy_evict_first();
            int i = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++i) {
                const int s = i % stages;
                const int2 h = __ldg(&tiles[t]), tl = __ldg(&tiles[t + 1]);
                if (i >= stages) mbar_wait(&empty[s], (uint32_t)(i / stages - 1) & 1u);
                unsigned char *base = smem_raw + (size_t)s * stage_bytes;
                int cnt = 0, rcnt = 0;
                const int a0 = h.y & ~3, ra0 = h.x & ~3;
                if (!(tl.x - h.x == 1 && tl.y - h.y > long_threshold)) {
                    cnt = max(min((tl.y + 3) & ~3, nnz_bulk) - a0, 0);
                    rcnt = max(min((tl.x + 4) & ~3, rp_bulk) - ra0, 0);
                }
                mbar_arrive_expect_tx(&full[s], (uint32_t)(cnt * 12 + rcnt * 4));
                if (rcnt) bulk_g2s(base + (size_t)cnt * 12, row_ptr + ra0, (uint32_t)rcnt * 4u, &full[s], policy);
                if (cnt) {
                    bulk_g2s(base + (size_t)cnt * 8, col_idx + a0, (uint32_t)cnt * 4u, &full[s], policy);
                    bulk_g2s(base, values + a0, (uint32_t)cnt * 8u, &full[s], policy);
                }
            }
        }
        return;
    }

    // ---------------- consumers: independent warps, lane = row (or a slice of a row) ----------------
    __shared__ double warp_sq[kConsumerWarps];
    __shared__ double mail_total;
    bool scaled = false;
    double prev_norm = 1.0;
    if constexpr (kFused) {
        if (ep.mail.world > 0) {
            if (ep.mail.iteration > 0) {
                // wait for every rank's previous launch: its |w|^2 is in my mailbox and its boundary rows are in my x
                if (warp == 0) {
                    const double total = mail_wait_total(ep.mail, lane);
                    if (lane == 0) mail_total = total;
                }
                asm volatile("bar.sync 2, %0;" ::"n"(kConsumerWarps * 32) : "memory");
                scaled = true;
                prev_norm = sqrt(mail_total);
            }
        } else {
            scaled = ep.prev_sumsq != nullptr;
            prev_norm = scaled ? sqrt(*ep.prev_sumsq) : 1.0;
        }
    }
    const double inv_norm = 1.0 / prev_norm;  // one division per thread, one multiplication per row (1 ulp from a division)
    double sq = 0.0;  // sum of the squares of the rows this lane produced
    // y[row] = v; the fused instantiation scales it first, accumulates v^2 and mirrors boundary rows into the peers
    auto emit = [&](int row, double v) {
        if constexpr (kFused) {
            if (scaled) v *= inv_norm;
            sq = fma(v, v, sq);
            for (int p = 0; p < ep.peers.count; ++p)
                if (row >= ep.peers.lo[p] && row < ep.peers.hi[p]) ep.peers.dst[p][row] = v;
        }
        y[row] = v;
    };
    int2 head = make_int2(0, 0), tail = make_int2(0, 0);
    if ((int)blockIdx.x < num_tiles) {
        head = __ldg(&tiles[blockIdx.x]);
        tail = __ldg(&tiles[blockIdx.x + 1]);
    }
    int dealt = 0;  // chunks handed out so far, modulo the number of consumer warps (same in every warp)
    int i = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++i) {
        const int s = i % stages;
        const int r0 = head.x, rows = tail.x - head.x, n0 = head.y, n1 = tail.y;
        if (t + (int)gridDim.x < num_tiles) {  // descriptors of this CTA's next tile
            head = __ldg(&tiles[t + gridDim.x]);
            tail = __ldg(&tiles[t + gridDim.x + 1]);
        }
        unsigned char *base = smem_raw + (size_t)s * stage_bytes;
        const int a0 = n0 & ~3, ra0 = r0 & ~3;
        const int loaded = max(min((n1 + 3) & ~3, nnz_bulk) - a0, 0);
        const int rloaded = max(min((r0 + rows + 4) & ~3, rp_bulk) - ra0, 0);
        double *sv = reinterpret_cast<double *>(base);
        const int *sc = reinterpret_cast<const int *>(base + (size_t)loaded * 8);
        const int *srp = reinterpret_cast<const int *>(base + (size_t)loaded * 12);
        bool wrote = false;
        mbar_wait(&full[s], (uint32_t)(i / stages) & 1u);
        if (!(rows == 1 && n1 - n0 > long_threshold)) {  // long rows belong to the csr_long_* kernels
            auto rp = [&](int r) { return (r - ra0 < rloaded) ? srp[r - ra0] : __ldg(row_ptr + r); };
            const int nchunks = (rows + 31) >> 5;
            if (nchunks < kConsumerWarps && forced_tpr != 1 && n1 - a0 <= loaded) {
                // Few rows in the tile, i.e. longer rows: 32-row chunks would leave most warps without work.
                // (A) every consumer thread multiplies a strided share of the whole tile in place, (B) after a
                // consumer-only barrier the rows are summed by G lanes each, G chosen so that all lanes have a row.
                constexpr int kLanes = kConsumerWarps * 32;
                products_staged<8>(sv, sc, n0 - a0, n1 - a0, tid, kLanes, x);
                wrote = true;
                asm volatile("bar.sync 3, %0;" ::"n"(kLanes) : "memory");
                int G = 1;
                while (G < 32 && rows * (2 * G) <= kLanes) G <<= 1;
                const int per_pass = kLanes / G;
                for (int first = 0; first < rows; first += per_pass) {  // warp-uniform trip count
                    const int lr = first + tid / G;
                    const bool live = lr < rows;
                    int lo = 0, hi = 0;
                    if (live) {
                        lo = rp(r0 + lr) - a0;
                        hi = rp(r0 + lr + 1) - a0;
                    }
                    const double acc = group_row_sum(sv, lo, hi, G, lane, lr);
                    if (live && (lane & (G - 1)) == 0) emit(r0 + lr, accumulate ? __dadd_rn(y[r0 + lr], acc) : acc);
                }
            } else
            for (int c = (warp - dealt + kConsumerWarps) % kConsumerWarps; c < nchunks; c += kConsumerWarps) {
                const int lr = c * 32 + lane;
                const bool live = lr < rows;
                int lo = 0, hi = 0;
                if (live) {
                    lo = rp(r0 + lr) - a0;
                    hi = rp(r0 + lr + 1) - a0;
                }
                const int len = hi - lo;
                const int maxlen = __reduce_max_sync(0xffffffffu, len);
                const int chunk_hi = __reduce_max_sync(0xffffffffu, hi);  // offsets grow with the row index
                double acc = 0.0;
                const bool serial = forced_tpr == 1 || chunk_hi > loaded || (forced_tpr == 0 && maxlen <= kSerialRowMax);
                if (serial) {
                    // short rows: lane = row, left to right, mul and add rounded separately (the serial loop's order)
                    if (live && accumulate) acc = y[r0 + lr];
                    if (hi <= loaded) {
                        acc = dot_staged<4>(sv, sc, lo, hi, 1, x, acc);
                    } else {  // ragged end of the arrays (last tile only): the unstaged tail comes from HBM
                        for (int k = lo; k < hi; ++k) {
                            const double v = k < loaded ? sv[k] : values[(long long)a0 + k];
                            const int col = k < loaded ? sc[k] : col_idx[(long long)a0 + k];
                            acc = __dadd_rn(acc, __dmul_rn(v, ldg_x(x, col)));
                        }
                    }
                    if (live) emit(r0 + lr, acc);
                } else {
                    // longer rows: (A) products in place, lane-strided over the whole chunk; (B) row sums
                    const int chunk_lo = __shfl_sync(0xffffffffu, lo, 0);
                    products_staged<8>(sv, sc, chunk_lo, chunk_hi, lane, 32, x);
                    wrote = true;
                    __syncwarp();
                    acc = chunk_row_sum(sv, lo, hi, lane);
                    if (live) emit(r0 + lr, accumulate ? __dadd_rn(y[r0 + lr], acc) : acc);
                }
            }
            if (nchunks >= kConsumerWarps || forced_tpr == 1 || n1 - a0 > loaded) dealt = (dealt + nchunks) % kConsumerWarps;
        }
        if (wrote) fence_proxy_async();  // generic-proxy writes to the stage before the async proxy refills it
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
    }
    if (kFused && ep.partials != nullptr) {  // fixed-order CTA sum of squares (consumer warps only: the producer has left)
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, off);
        if (lane == 0) warp_sq[warp] = sq;
        asm volatile("bar.sync 2, %0;" ::"n"(kConsumerWarps * 32) : "memory");
        if (tid == 0) {
            double total = 0.0;
#pragma unroll
            for (int w = 0; w < kConsumerWarps; ++w) total += warp_sq[w];
            ep.partials[blockIdx.x] = total;
        }
        if (ep.mail.world > 0) {
            // every consumer's rows (local and peer stores) are issued before the barrier; a device-scope fence by
            // thread 0 (cumulative through the barrier) orders them before the counter; the CTA that completes the count
            // pays the one system-scope fence before it publishes the tag (mail_publish)
            asm volatile("bar.sync 2, %0;" ::"n"(kConsumerWarps * 32) : "memory");
            if (warp == 0) {
                unsigned int arrived = 0;
                if (lane == 0) {
                    __threadfence();
                    arrived = atomicAdd(ep.mail.counter, 1u);
                }
                arrived = __shfl_sync(0xffffffffu, arrived, 0);
                if (arrived == gridDim.x - 1) mail_publish(ep.mail, ep.partials, (int)gridDim.x, lane);  // last CTA of the launch
            }
        }
    }
}

// =================================================================================================
// HLL
// =================================================================================================
template <int kConsumerWarps>
__global__ void __launch_bounds__((kConsumerWarps + 1) * 32, (kConsumerWarps >= 24 ? 1 : 2))
hll_stream_kernel(const HllTile *__restrict__ tiles, int num_tiles, const long long *__restrict__ hack_off,
                  const int *__restrict__ JA, const double *__restrict__ AS, const double *__restrict__ x,
                  double *__restrict__ y, int M, int cap, int stages, int wide_slots) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ double wide_partial[kConsumerWarps][32];
    const size_t stage_bytes = (size_t)cap * 12;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + (size_t)stages * stage_bytes);
    uint64_t *empty = full + stages;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumerWarps);
        }
        fence_mbar_init();
    }
    __syncthreads();

    if (warp == kConsumerWarps) {
        if (lane == 0) {
            const uint64_t policy = policy_evict_first();
            int i = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++i) {
                const int s = i % stages;
                const HllTile h = tiles[t], tl = tiles[t + 1];
                if (i >= stages) mbar_wait(&empty[s], (uint32_t)(i / stages - 1) & 1u);
                unsigned char *base = smem_raw + (size_t)s * stage_bytes;
                long long cnt = tl.slot - h.slot;  // slots come in multiples of 32: always whole 16-byte groups
                if (tl.hack - h.hack == 1 && cnt > wide_slots) cnt = 0;  // wide hack: read straight from HBM
                mbar_arrive_expect_tx(&full[s], (uint32_t)(cnt * 12));
                if (cnt) {
                    bulk_g2s(base + (size_t)cap * 8, JA + h.slot, (uint32_t)cnt * 4u, &full[s], policy);
                    bulk_g2s(base, AS + h.slot, (uint32_t)cnt * 8u, &full[s], policy);
                }
            }
        }
        return;
    }

    HllTile head = {0, 0, 0}, tail = {0, 0, 0};
    if ((int)blockIdx.x < num_tiles) {
        head = tiles[blockIdx.x];
        tail = tiles[blockIdx.x + 1];
    }
    int dealt = 0;
    int i = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++i) {
        const int s = i % stages;
        const HllTile h = head, tl = tail;
        if (t + (int)gridDim.x < num_tiles) {
            head = tiles[t + gridDim.x];
            tail = tiles[t + gridDim.x + 1];
        }
        const int hacks = tl.hack - h.hack;
        const int span = (int)(tl.slot - h.slot);
        const unsigned char *base = smem_raw + (size_t)s * stage_bytes;
        const double *sv = reinterpret_cast<const double *>(base);
        const int *sc = reinterpret_cast<const int *>(base + (size_t)cap * 8);
        const int first = (warp - dealt + kConsumerWarps) % kConsumerWarps;
        long long o0 = 0, o1 = 0;  // slot range of this warp's first hack: requested before the wait
        if (first < hacks) {
            o0 = __ldg(hack_off + h.hack + first);
            o1 = __ldg(hack_off + h.hack + first + 1);
        }
        mbar_wait(&full[s], (uint32_t)(i / stages) & 1u);
        if (hacks == 1 && span > wide_slots) {
            // one very wide hack: the consumer warps split its columns (lane = row), fixed-order combine
            const int width = span >> 5;
            double acc = 0.0;
            for (int j = warp; j < width; j += kConsumerWarps) {
                const long long slot = h.slot + (long long)j * 32 + lane;
                acc = __dadd_rn(acc, __dmul_rn(ldg_stream_f64(AS + slot), ldg_x(x, ldg_stream_s32(JA + slot))));
            }
            wide_partial[warp][lane] = acc;
            asm volatile("bar.sync 1, %0;" ::"n"(kConsumerWarps * 32) : "memory");
            if (warp == 0) {
                double total = 0.0;
#pragma unroll
                for (int w = 0; w < kConsumerWarps; ++w) total = __dadd_rn(total, wide_partial[w][lane]);
                const long long row = (long long)h.hack * 32 + lane;
                if (row < M) y[row] = total;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(kConsumerWarps * 32) : "memory");
        } else {
            for (int lh = first; lh < hacks; lh += kConsumerWarps) {  // one warp per hack, lane = row
                if (lh != first) {
                    o0 = __ldg(hack_off + h.hack + lh);
                    o1 = __ldg(hack_off + h.hack + lh + 1);
                }
                const int rel = (int)(o0 - h.slot) + lane;
                const int hi = rel + (int)(o1 - o0);  // walk j*32 + lane: sequential in j, the serial order
                const double acc = dot_staged<8>(sv, sc, rel, hi, 32, x, 0.0);
                const long long row = (long long)(h.hack + lh) * 32 + lane;
                if (row < M) y[row] = acc;
            }
            dealt = (dealt + hacks) % kConsumerWarps;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
    }
}

// ---- HLL tile plan: bin hacks into windows of tile_slots merge items (slots + rows) -------------------
__global__ void hll_flag_kernel(int num_hacks, const long long *__restrict__ hack_off, int tile_slots, int wide_slots,
                                unsigned char *__restrict__ boundary) {
    const int hk = blockIdx.x * blockDim.x + threadIdx.x;
    if (hk >= num_hacks) return;
    const long long a = hack_off[hk], b = hack_off[hk + 1];
    bool open = hk == 0 || (b - a) > wide_slots;
    if (hk > 0) {
        const long long before = hack_off[hk - 1];
        open = open || (a - before) > wide_slots;
        open = open || (a + 32LL * hk) / tile_slots != (before + 32LL * (hk - 1)) / tile_slots;
    }
    boundary[hk] = open ? 1 : 0;
}

__global__ void hll_tiles_kernel(int num_tiles, int num_hacks, const int *__restrict__ first_hack,
                                 const long long *__restrict__ hack_off, HllTile *__restrict__ tiles) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > num_tiles) return;
    const int hk = t < num_tiles ? first_hack[t] : num_hacks;
    HllTile d;
    d.hack = hk;
    d.pad = 0;
    d.slot = hack_off[hk];
    tiles[t] = d;
}

// ---- host side ------------------------------------------------------------------------------------------
static int g_autotune = -1;  // -1: follow SPMV_B200_AUTOTUNE (default on)

int env_int(const char *name, int fallback) {
    if (g_autotune >= 0 && std::strcmp(name, "SPMV_B200_AUTOTUNE") == 0) return g_autotune;
    const char *v = std::getenv(name);
    if (!v || !*v) return fallback;
    return std::atoi(v);
}

static int round4(int v) { return (v + 3) & ~3; }

// bytes of one packed stage: 4 bytes per stream word of the window + the last row (<= L nonzeros) + alignment slack
static int csr_stage_bytes(const spmv_b200_csr *A) { return (4 * A->tile_items + 12 * A->long_threshold + 128 + 127) & ~127; }

static size_t csr_stream_smem(const spmv_b200_csr *A) {
    return (size_t)A->stages * (size_t)csr_stage_bytes(A) + (size_t)A->stages * 16 + 16;
}

constexpr int kMaxStreamSmem = 220 * 1024;  // the plans shrink their stage count until they fit below this

static int pick_grid(const void *kernel, int threads, size_t smem, int num_tiles, int &grid) {
    int dev = 0, sms = 0, per_sm = 0;
    SPMV_TRY_CUDA(cudaGetDevice(&dev));
    SPMV_TRY_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // the limit is per kernel and device, not per handle: always the largest size any plan may ask for, so that a second
    // handle planned with smaller stages can never lower it below what an older live handle passes at launch
    SPMV_TRY_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxStreamSmem));
    SPMV_TRY_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1) return fail(SPMV_B200_ERR_INVALID, "stream kernel does not fit: %zu bytes of shared memory per CTA", smem);
    const int want = env_int("SPMV_B200_CTAS_PER_SM", 0);
    if (want > 0) per_sm = std::min(per_sm, want);
    grid = std::max(1, std::min(num_tiles, sms * per_sm));
    return SPMV_B200_OK;
}

static int pick_consumers(int fallback) {
    const int c = env_int("SPMV_B200_CONSUMER_WARPS", fallback);
    return (c == 4 || c == 8 || c == 12 || c == 16 || c == 24) ? c : fallback;
}

#define STREAM_DISPATCH(consumers, KERNEL, EXPR)            \
    switch (consumers) {                                    \
        case 4: { auto kfn = KERNEL<4>; EXPR; } break;      \
        case 8: { auto kfn = KERNEL<8>; EXPR; } break;      \
        case 16: { auto kfn = KERNEL<16>; EXPR; } break;    \
        case 24: { auto kfn = KERNEL<24>; EXPR; } break;    \
        default: { auto kfn = KERNEL<12>; EXPR; } break;    \
    }

template <int C> constexpr auto csr_plain_kernel = csr_stream_kernel<C, false>;
template <int C> constexpr auto csr_fused_kernel = csr_stream_kernel<C, true>;

int stream_prepare_csr(spmv_b200_csr *A) {
    A->stages = std::max(1, std::min(env_int("SPMV_B200_STAGES", kDefaultStages), 8));
    A->stream_grid = 0;
    if (A->num_tiles == 0) return SPMV_B200_OK;
    size_t smem = csr_stream_smem(A);
    while (smem > 220 * 1024 && A->stages > 1) {
        A->stages--;
        smem = csr_stream_smem(A);
    }
    A->consumers = pick_consumers(kDefaultCsrConsumers);
    int rc = SPMV_B200_OK;
    STREAM_DISPATCH(A->consumers, csr_plain_kernel,
                    rc = pick_grid(reinterpret_cast<const void *>(kfn), (A->consumers + 1) * 32, smem, A->num_tiles, A->stream_grid));
    int fused_grid = 0;
    if (rc == SPMV_B200_OK)
        STREAM_DISPATCH(A->consumers, csr_fused_kernel,
                        rc = pick_grid(reinterpret_cast<const void *>(kfn), (A->consumers + 1) * 32, smem, A->num_tiles, fused_grid));
    if (rc == SPMV_B200_OK) A->stream_grid = std::min(A->stream_grid, fused_grid);
    return rc;
}

int stream_launch_csr(const spmv_b200_csr *A, const double *x, double *y, int accumulate, const Epilogue *ep,
                      cudaStream_t stream, int tile_begin, int tile_count) {
    if (tile_count < 0) {
        tile_begin = 0;
        tile_count = A->num_tiles;
    }
    if (tile_count == 0) return SPMV_B200_OK;
    const int2 *tiles = A->tiles + tile_begin;
    const int grid = std::min(A->stream_grid, tile_count);
    Epilogue none;
    const Epilogue e = ep ? *ep : none;
    const size_t smem = csr_stream_smem(A);
    if (ep) {
        STREAM_DISPATCH(A->consumers, csr_fused_kernel,
                        (kfn<<<grid, (A->consumers + 1) * 32, smem, stream>>>(
                            tiles, tile_count, A->row_ptr, A->col_idx, A->values, x, y, A->M, (int)A->nnz,
                            csr_stage_bytes(A), A->stages, A->long_threshold, A->forced_tpr, accumulate, e)));
    } else {
        STREAM_DISPATCH(A->consumers, csr_plain_kernel,
                        (kfn<<<grid, (A->consumers + 1) * 32, smem, stream>>>(
                            tiles, tile_count, A->row_ptr, A->col_idx, A->values, x, y, A->M, (int)A->nnz,
                            csr_stage_bytes(A), A->stages, A->long_threshold, A->forced_tpr, accumulate, e)));
    }
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

static size_t hll_stream_smem(const spmv_b200_hll *H, int &cap) {
    cap = round4(H->tile_slots + H->wide_slots + 32);
    return (size_t)H->stages * (size_t)cap * 12 + (size_t)H->stages * 16 + 16;
}

int stream_plan_hll(spmv_b200_hll *H, cudaStream_t stream) {
    cudaFree(H->tiles);
    H->tiles = nullptr;
    H->num_tiles = 0;
    H->stream_grid = 0;
    H->stages = std::max(1, std::min(env_int("SPMV_B200_STAGES", kDefaultStages), 8));
    H->tile_slots = std::max(64, env_int("SPMV_B200_HLL_TILE_SLOTS", kHllTileSlots));
    H->wide_slots = std::max(32, env_int("SPMV_B200_HLL_WIDE_SLOTS", kHllWideSlots));
    const int nb = H->num_hacks;
    if (nb == 0) return SPMV_B200_OK;
    unsigned char *boundary = nullptr;
    int *first = nullptr, *d_count = nullptr;
    void *temp = nullptr;
    auto body = [&]() -> int {
        SPMV_TRY_CUDA(cudaMalloc(&boundary, (size_t)nb));
        SPMV_TRY_CUDA(cudaMalloc(&first, (size_t)nb * sizeof(int)));
        SPMV_TRY_CUDA(cudaMalloc(&d_count, sizeof(int)));
        hll_flag_kernel<<<blocks_for(nb, 256), 256, 0, stream>>>(nb, H->hack_off, H->tile_slots, H->wide_slots, boundary);
        SPMV_TRY_CUDA(cudaGetLastError());
        thrust::counting_iterator<int> ids(0);
        size_t temp_bytes = 0;
        SPMV_TRY_CUDA(cub::DeviceSelect::Flagged(nullptr, temp_bytes, ids, boundary, first, d_count, nb, stream));
        SPMV_TRY_CUDA(cudaMalloc(&temp, temp_bytes ? temp_bytes : 1));
        SPMV_TRY_CUDA(cub::DeviceSelect::Flagged(temp, temp_bytes, ids, boundary, first, d_count, nb, stream));
        SPMV_TRY_CUDA(cudaMemcpyAsync(&H->num_tiles, d_count, sizeof(int), cudaMemcpyDeviceToHost, stream));
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
        SPMV_TRY_CUDA(cudaMalloc(&H->tiles, (size_t)(H->num_tiles + 1) * sizeof(HllTile)));
        hll_tiles_kernel<<<blocks_for(H->num_tiles + 1, 256), 256, 0, stream>>>(H->num_tiles, nb, first, H->hack_off, H->tiles);
        SPMV_TRY_CUDA(cudaGetLastError());
        SPMV_TRY_CUDA(cudaStreamSynchronize(stream));
        return SPMV_B200_OK;
    };
    int rc = body();
    cudaFree(boundary);
    cudaFree(first);
    cudaFree(d_count);
    cudaFree(temp);
    if (rc != SPMV_B200_OK) return rc;
    int cap;
    size_t smem = hll_stream_smem(H, cap);
    while (smem > 220 * 1024 && H->stages > 1) {
        H->stages--;
        smem = hll_stream_smem(H, cap);
    }
    H->consumers = pick_consumers(kDefaultHllConsumers);
    STREAM_DISPATCH(H->consumers, hll_stream_kernel,
                    rc = pick_grid(reinterpret_cast<const void *>(kfn), (H->consumers + 1) * 32, smem, H->num_tiles, H->stream_grid));
    return rc;
}

int stream_launch_hll(const spmv_b200_hll *H, const double *x, double *y, cudaStream_t stream, int tile_begin,
                      int tile_count) {
    if (tile_count < 0) {
        tile_begin = 0;
        tile_count = H->num_tiles;
    }
    if (tile_count == 0) return SPMV_B200_OK;
    int cap;
    const size_t smem = hll_stream_smem(H, cap);
    const int grid = std::min(H->stream_grid, tile_count);
    STREAM_DISPATCH(H->consumers, hll_stream_kernel,
                    (kfn<<<grid, (H->consumers + 1) * 32, smem, stream>>>(H->tiles + tile_begin, tile_count, H->hack_off, H->JA,
                                                                         H->AS, x, y, H->M, cap, H->stages, H->wide_slots)));
    SPMV_TRY_CUDA(cudaGetLastError());
    return SPMV_B200_OK;
}

}  // namespace spmv

extern "C" int spmv_b200_autotune(int enable) {
    const int before = spmv::env_int("SPMV_B200_AUTOTUNE", 1) ? 1 : 0;
    spmv::g_autotune = enable ? 1 : 0;
    return before;
}
