// common.cuh -- shared device helpers and host-side error plumbing for the sm_100a SpMV kernels.
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>

#include "spmv_b200.h"

namespace spmv {

// ---- per-thread error message (spmv_b200_last_error) -----------------------------------------
void set_error(const char *fmt, ...);
int fail(int code, const char *fmt, ...);

#define SPMV_TRY_CUDA(expr)                                                                      \
    do {                                                                                         \
        cudaError_t err__ = (expr);                                                              \
        if (err__ != cudaSuccess) {                                                              \
            const int code__ = (err__ == cudaErrorNoDevice || err__ == cudaErrorInsufficientDriver) \
                                   ? SPMV_B200_ERR_NO_DEVICE                                     \
                                   : (err__ == cudaErrorMemoryAllocation ? SPMV_B200_ERR_NOMEM   \
                                                                         : SPMV_B200_ERR_CUDA);  \
            return spmv::fail(code__, "%s: %s (%s:%d)", #expr, cudaGetErrorString(err__), __FILE__, __LINE__); \
        }                                                                                        \
    } while (0)

#define SPMV_TRY(expr)                   \
    do {                                 \
        int rc__ = (expr);               \
        if (rc__ != SPMV_B200_OK) return rc__; \
    } while (0)

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

inline unsigned int blocks_for(long long items, int per_block) {
    long long b = (items + per_block - 1) / per_block;
    return static_cast<unsigned int>(b > 0 ? b : 1);
}

// ---- streaming loads ---------------------------------------------------------------------------
// The matrix stream (values / column indices / HLL slots) is read exactly once per product: keep
// it out of L1 (no_allocate) and mark it evict-first in L2 so that x -- the only operand with
// reuse -- stays resident in the 126 MB L2.  sm_100 adds 256-bit global loads (LDG.E.256); the
// L2 eviction qualifier is only accepted on that form.
__device__ __forceinline__ void ldg_stream_f64x4(const double *p, double (&v)[4]) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3])
                 : "l"(p));
}

__device__ __forceinline__ int4 ldg_stream_s32x4(const int *p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ void ldg_stream_s32x8(const int *p, int (&c)[8]) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.s32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(c[0]), "=r"(c[1]), "=r"(c[2]), "=r"(c[3]), "=r"(c[4]), "=r"(c[5]), "=r"(c[6]), "=r"(c[7])
                 : "l"(p));
}

// SPMV_STREAM_EVICT_FIRST: the scalar stream loads also carry an L2 evict-first policy (createpolicy + cache_hint)
__device__ __forceinline__ unsigned long long policy_stream() {
    unsigned long long p;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));  // pure: hoisted out of loops
    return p;
}

__device__ __forceinline__ double ldg_stream_f64(const double *p) {
    double r;
#ifdef SPMV_STREAM_EVICT_FIRST
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(policy_stream()));
#else
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(r) : "l"(p));
#endif
    return r;
}

// float twins of the scalar loads (fp32 storage, fp64 arithmetic: SURVEY.md section 8(f).3); all return double
__device__ __forceinline__ double ldg_stream_f64(const float *p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return (double)r;
}

__device__ __forceinline__ int ldg_stream_s32(const int *p) {
    int r;
#ifdef SPMV_STREAM_EVICT_FIRST
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(policy_stream()));
#else
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
#endif
    return r;
}

// the 16-bit column field of a CSR handle's narrow private image (image.cu, hll.cu), zero-extended into 32 bits
__device__ __forceinline__ int ldg_stream_u16(const uint16_t *p) {
    unsigned int r;
#ifdef SPMV_STREAM_EVICT_FIRST
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u16 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(policy_stream()));
#else
    asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=r"(r) : "l"(p));
#endif
    return (int)r;
}

// a CSR handle's private image (image.cu, hll.cu): a 1-byte value code or pattern id, zero-extended into 32 bits
__device__ __forceinline__ int ldg_stream_u8(const uint8_t *p) {
    unsigned int r;
#ifdef SPMV_STREAM_EVICT_FIRST
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(policy_stream()));
#else
    asm volatile("ld.global.nc.L1::no_allocate.u8 %0, [%1];" : "=r"(r) : "l"(p));
#endif
    return (int)r;
}

// x is gathered through the read-only path (LDG.CONSTANT), allocating in L1: neighbouring rows of
// banded matrices hit the same lines -- and, more important, a gather that misses needs an L1 line while it is in
// flight: with L1::no_allocate the same kernels ran 3x slower on random columns (profiles/r01d_kernel_selection.md).
// SPMV_X_EVICT_LAST (off: measured +-1 %): the gathers also carry an L2 evict-last policy
// (createpolicy + ld.global.nc.L2::cache_hint), so that x outlives the once-read matrix stream in L2.
__device__ __forceinline__ unsigned long long policy_evict_last() {
    unsigned long long p;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));  // pure: hoisted out of loops
    return p;
}

__device__ __forceinline__ double ldg_x(const double *x, int col) {
#if defined(SPMV_X_EVICT_LAST)
    double r;
    asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(x + col), "l"(policy_evict_last()));
    return r;
#else
    return __ldg(x + col);
#endif
}

__device__ __forceinline__ double ldg_x(const float *x, int col) { return (double)__ldg(x + col); }

// ---- mailbox exchange of |w|^2 between ranks (spmv_b200_mail_t, include/spmv_b200.h): system-scope accesses to
// peer memory over NVLink.  Used by the fused stream kernel (stream.cu) and the fused row kernel (csr.cu). -------
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_relaxed_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

constexpr long long kMailSpinCycles = 4000000000LL;  // ~2 s at 1.9 GHz: a peer that has not answered by then is gone

// Launch k > 0, one whole warp: wait until every rank's slot of parity (k-1)&1 in MY mailbox carries tag k (launch k-1
// of that rank has finished: its |w|^2 is here and its boundary rows are in my x), then add the sums in rank order.
// Returns the total in every lane.
__device__ __forceinline__ double mail_wait_total(const spmv_b200_mail_t &m, int lane) {
    const unsigned long long want = m.iteration;
    const int parity = (int)((m.iteration - 1) & 1);
    double mine = 0.0;
    if (lane < m.world) {
        const unsigned long long *slot = m.box[m.rank] + 2 * (parity * m.world + lane);
        const long long t0 = clock64();
        while (ld_acquire_sys(slot + 1) != want) {
            if (clock64() - t0 > kMailSpinCycles) {
                *m.status = 1;
                break;
            }
            __nanosleep(40);
        }
        mine = __longlong_as_double((long long)ld_acquire_sys(slot));
    }
    double total = 0.0;
    for (int r = 0; r < m.world; ++r) total += __shfl_sync(0xffffffffu, mine, r);
    return total;
}

// Sum of count per-CTA partials by one warp, fixed order: lane l adds elements l, l+32, ... in order, then an xor tree.
// The loads of a group of 8 are issued together (they are independent; one by one they would cost an L2 round trip
// each on the critical path between two launches: 37 x 0.4 us for 1184 partials).
__device__ __forceinline__ double warp_sum_partials(const double *partials, int count, int lane) {
    double part = 0.0;
    for (int base = lane; base < count; base += 8 * 32) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = base + u * 32 < count ? __ldcg(partials + base + u * 32) : 0.0;
#pragma unroll
        for (int u = 0; u < 8; ++u) part += v[u];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
    return part;
}

// One whole warp of the LAST CTA of launch k (after a device-scope fence): add the per-CTA partials in a fixed order
// and write {sum, tag k+1} into slot [k&1][rank] of every rank's mailbox; reset the CTA counter for the next launch.
// Ordering: every CTA issued a device-scope fence + device-scope atomic after its rows (release pattern towards this CTA);
// this CTA's system-scope fence then orders all of them -- peer stores included -- before the st.release.sys of the tag
// (causality order is transitive across morally strong edges of different scopes).  One fence.sys per launch: a
// system-scope fence per CTA costs ~30 ns each, serialised (measured: 26-41 us per iteration on 2-8 GPUs).
__device__ __forceinline__ void mail_publish(const spmv_b200_mail_t &m, const double *partials, int count, int lane) {
    __threadfence_system();
    const double part = warp_sum_partials(partials, count, lane);
    if (lane < m.world) {
        unsigned long long *slot = m.box[lane] + 2 * ((int)(m.iteration & 1) * m.world + m.rank);
        st_relaxed_sys(slot, (unsigned long long)__double_as_longlong(part));
        st_release_sys(slot + 1, m.iteration + 1);
    }
    if (lane == 0) *m.counter = 0;
}

// ---- per-row sums of products parked in shared memory, one warp per chunk of 32 rows ---------------
constexpr int kSerialRowMax = 12;  // rows up to this length are always summed by ONE lane, left to right: the stream and
                                   // tile kernels reproduce the reference's serial loop bit for bit on such rows, whatever
                                   // tile, path or GPU partition they fall into
constexpr int kLaneRowMax = 64;  // rows up to this length are summed by their own lane, longer ones by the whole warp

// Lane = row [lo, hi) of prod[].  Short rows start at a lane-dependent element and wrap around, so equally long
// rows (stride = row length) do not pile up on one shared-memory bank; rows longer than kLaneRowMax are summed
// by all 32 lanes followed by a fixed xor tree.  Every lane of the warp must call this (it shuffles).
__device__ __forceinline__ double chunk_row_sum(const double *prod, int lo, int hi, int lane) {
    const int len = hi - lo;
    double acc = 0.0;
    if (len <= kLaneRowMax && len > 0) {
        const int start = len <= kSerialRowMax ? lo : lo + lane % len;
        for (int k = start; k < hi; ++k) acc = __dadd_rn(acc, prod[k]);
        for (int k = lo; k < start; ++k) acc = __dadd_rn(acc, prod[k]);
    }
    unsigned wide = __ballot_sync(0xffffffffu, len > kLaneRowMax);
    while (wide) {
        const int owner = __ffs(wide) - 1;
        wide &= wide - 1;
        const int wlo = __shfl_sync(0xffffffffu, lo, owner), whi = __shfl_sync(0xffffffffu, hi, owner);
        double part = 0.0;
        for (int k = wlo + lane; k < whi; k += 32) part = __dadd_rn(part, prod[k]);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) part = __dadd_rn(part, __shfl_xor_sync(0xffffffffu, part, off));
        if (lane == owner) acc = part;
    }
    return acc;
}

// ---- counter-based hash shared by the device generators and their numpy twins -----------------
__host__ __device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

__host__ __device__ __forceinline__ unsigned long long hash3(unsigned long long seed, unsigned long long a,
                                                             unsigned long long b) {
    return mix64(seed + a * 0x9E3779B97F4A7C15ULL + b * 0xD1B54A32D192ED03ULL);
}

// uniform in (0, 1]: 53 random bits
__host__ __device__ __forceinline__ double unit_interval(unsigned long long h) {
    return (double)((h >> 11) + 1ULL) * (1.0 / 9007199254740992.0);
}

}  // namespace spmv
