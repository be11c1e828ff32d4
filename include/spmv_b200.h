/*
 * spmv_b200.h -- thin C-ABI over the hand-written sm_100a SpMV kernels.
 *
 * This is the layer the reference's CUDA driver binds instead of launching its own
 * __global__ kernels.  Each entry point cites the reference interface it replaces
 * (paths relative to the reference repository):
 *
 *   reference main_cuda.cu:135-145   cudaMalloc + cudaMemcpy of row_ptr/col_idx/values
 *                                    -> spmv_b200_csr_upload / spmv_b200_csr_wrap_device
 *   reference main_cuda.cu:166,238,317  spmv_csr_{naive,warp,warp_shared_memory}_kernel<<<>>>
 *       (cuda_libs/csr_matrix_cuda.cuh:26-49)      -> spmv_b200_csr_spmv
 *   reference main_cuda.cu:183,255,336  cudaMemcpy(y, D2H) after every product
 *                                    -> spmv_b200_csr_spmv_host (H2D x, product, D2H y)
 *   reference main_cuda.cu:369-402   per-block cudaMalloc/cudaMemcpy of ELLPACKBlock.JA/AS
 *                                    -> spmv_b200_hll_upload (one column-major arena)
 *   reference main_cuda.cu:454,568,637  spmv_hll_{warp_shared_v1,naive,warp}_kernel<<<>>>
 *       (cuda_libs/hll_matrix.cuh:40-51)           -> spmv_b200_hll_spmv
 *   reference main_cuda.cu:471,585,653  cudaMemcpy(y, D2H)   -> spmv_b200_hll_spmv_host
 *
 * Conventions: plain C types only; every function returns 0 (SPMV_B200_OK) or a negative
 * status and never calls exit() (the reference aborts through checkCudaErrors,
 * cuda_libs/helper_cuda.h:582-595); spmv_b200_last_error() returns a per-thread message.
 * "d_" pointers are device pointers on the CURRENT CUDA device, "stream" is a cudaStream_t
 * passed as void* (NULL = default stream).  All arithmetic is fp64, indices are int32 as in
 * the reference (libs/csr_matrix.h:8-16); nnz and slot counts are 64-bit where they may
 * exceed 2^31 in bytes.  There is no CPU fallback: without a CUDA device every compute entry
 * point fails with SPMV_B200_ERR_NO_DEVICE.
 */
#ifndef SPMV_B200_H
#define SPMV_B200_H

#include "hll_matrix.h" /* ELLPACKBlock / HLLMatrix / HACK_SIZE (drop-in host structs) */

#ifdef __cplusplus
extern "C" {
#endif

#define SPMV_B200_OK 0
#define SPMV_B200_ERR_INVALID (-1)
#define SPMV_B200_ERR_CUDA (-2)
#define SPMV_B200_ERR_NO_DEVICE (-3)
#define SPMV_B200_ERR_NOMEM (-4)

/* CSR kernel selection for spmv_b200_csr_spmv */
#define SPMV_B200_ALGO_AUTO 0     /* ROW, STREAM or ROW_IMAGE (timed at plan time, same bits) when no row exceeds 12 nonzeros;
                                     STREAM for <= 12 nnz/row on average; else VECTOR (even rows) or BINNED (skewed rows) */
#define SPMV_B200_ALGO_VECTOR 1   /* plain vector-per-row kernel with shuffle reduction      */
#define SPMV_B200_ALGO_TILE 2     /* retired (round 2): accepted for compatibility, runs STREAM */
#define SPMV_B200_ALGO_STREAM 3   /* persistent row-binned kernel, TMA bulk-copy pipeline    */
#define SPMV_B200_ALGO_BINNED 4   /* rows binned by length: 1..32 lanes per row, longest rows split */
#define SPMV_B200_ALGO_ROW 5      /* one thread per row, serial order (bit-identical to the reference loop) */
#define SPMV_B200_ALGO_ROW_IMAGE 6 /* one lane per row on the handle's private image, column-major or patterns (spmv_b200_csr_set_image);
                                      the same bits as ROW.  SPMV_B200_ERR_INVALID when the handle holds no image */

/* synthetic CSR generators (BASELINE.json configs 2, 3, 5) */
#define SPMV_B200_SYNTH_LAP2D 1   /* p0 = n   : 5-point Laplacian on an n x n grid           */
#define SPMV_B200_SYNTH_LAP3D 2   /* p0 = n   : 7-point Laplacian on an n^3 grid             */
#define SPMV_B200_SYNTH_UNIFORM 3 /* p0 = M, p1 = N, p2 = nnz per row (stratified columns)   */

typedef struct spmv_b200_csr spmv_b200_csr; /* opaque: resident CSR matrix + kernel plan    */
typedef struct spmv_b200_hll spmv_b200_hll; /* opaque: resident column-major HLL image      */

typedef struct {
    int M, N;
    long long nnz;
    int num_tiles;       /* row-binned tiles of the adaptive kernel                          */
    int num_long_rows;   /* rows split over several CTAs (deterministic two-phase combine)   */
    int num_fragments;   /* fragments of those rows                                          */
    int threads_per_row; /* width of the in-tile shuffle reduction (1 = one thread per row)  */
    int tile_items;      /* D: rows+nnz per tile                                             */
    int long_threshold;  /* L: rows longer than this are "long"                              */
    long long algorithmic_bytes; /* nnz*12 + 4*(M+1) + 8*M + 8*N  (SURVEY.md section 8(d))   */
    int max_row_nnz;     /* longest row                                                      */
    int auto_algo;       /* the SPMV_B200_ALGO_* that SPMV_B200_ALGO_AUTO resolves to        */
    int row_batch;       /* batch of the thread-per-row kernel (tuned at plan time)          */
    int fused_batch;     /* fused iterated product: 0 = fused stream kernel, else batch of the fused row kernel */
    int flat_batch;      /* batch of the FLAT fused row kernel of the two-launch iterated product (plan-time choice) */
    int flat_chunks;     /* always 1: the FLAT kernel runs one CTA per 256 rows (kept for the layout of this struct) */
    long long image_bytes; /* size of the private image at 12 bytes per slot, as defined in version 102, whatever the
                              width of its column field (0: none, see spmv_b200_csr_set_image); image_device_bytes
                              is what it occupies */
    int image_form;      /* its kernel: 64 + B hll_rowu_kernel<B,double,true>, B hll_row_kernel<B,double,true>, 0 none
                            (on the value codes when image_value_bytes is 1) */
    int image_index_bytes; /* bytes of its column field: 2 (col - row; every column within 2^14 of its row), 4, 0 none */
    long long image_device_bytes; /* device bytes of its columns, values and value table:
                                     (image_index_bytes + image_value_bytes) per slot, plus 8 per table entry */
    int image_value_bytes; /* bytes of its value field: 8 (fp64), 1 (a code into a table of at most 256 doubles), 0 none */
    int image_patterns;  /* the pattern form (set_image mode 3; spmv_b200_version() >= 106): the number of distinct row
                            patterns in its dictionary, 0 for the other forms or none.  For this form image_form is
                            256 + W (csr_pattern_kernel<W>, W the longest row), image_bytes and image_device_bytes are
                            M (one byte per row) plus the dictionary's 12 * W + 4 bytes per pattern, and
                            image_index_bytes and image_value_bytes are 0 */
    int image_windows;   /* the pattern form (spmv_b200_version() >= 107): the windows of x a tile of 1024 rows stages
                            in shared memory -- one per cluster of the patterns' col - row, at most min(W, 3) of them --
                            or 0 when its kernel gathers x from global memory (scattered col - row); 0 for the other
                            forms.  The bytes of the image do not change with it */
} spmv_b200_csr_info_t;

typedef struct {
    int M, N;
    int num_hacks;          /* = ceil(M/32), reference src/hll_matrix.c:49                   */
    int max_maxnz;
    long long slots;        /* sum_b 32*MAXNZ_b (device image: rows padded to 32)            */
    long long nnz_reference_slots; /* sum_b rows_b*MAXNZ_b (reference host layout)           */
    long long algorithmic_bytes;   /* slots*12 + 8*(num_hacks+1) + 8*M + 8*N                 */
    int auto_kernel;        /* automatic choice: 0 slice, 1 stream, 2 rows                   */
    int row_batch;          /* batch of the lane-per-row kernel (tuned at plan time)         */
    int fused_batch, flat_batch; /* plan-time choices of the fused iterated product (grid-stride / FLAT) */
    int flat_chunks;        /* always 1: the FLAT kernel runs one CTA per 8 hacks (kept for the layout of this struct) */
} spmv_b200_hll_info_t;

/* ---- library / device ---------------------------------------------------------------- */
const char *spmv_b200_last_error(void);
/* forget the calling thread's message: the void drop-in products (csr_matrix_vector_mult, spmv_hll, ...) report a
 * failure by filling y with NaN and leaving a message here, so a caller that wants to tell "failed" from "x held a
 * NaN" clears the message first and looks at it afterwards */
void spmv_b200_clear_error(void);
int spmv_b200_version(void);
int spmv_b200_device_count(int *count);
/* name[len], sm count, L2 bytes, total global memory of the current device */
int spmv_b200_device_info(char *name, int len, int *sm_count, long long *l2_bytes, long long *mem_bytes);

/* ---- resident cache of the drop-in host API (off by default) -------------------------------------------------------
 * The reference's product signatures (csr_matrix_vector_mult, spvm_csr_parallel, spmv_hll, ...) carry raw arrays and no
 * state, so the drop-in versions upload the matrix on every call.  The reference's drivers call them 100 times on the
 * same arrays (main.c:105-362): with the cache on, the device copy of the last CSR and of the last HLL matrix is kept
 * and reused while the array POINTERS, sizes and a sampled fingerprint of the contents are unchanged; free_csr_matrix /
 * free_hll_matrix drop it.  Contract: do not modify the arrays in place between calls without calling
 * spmv_b200_resident_drop() (a sampled fingerprint cannot see every change).  Also switched on by the environment
 * variable SPMV_B200_RESIDENT=1.  enable = 2 (SPMV_B200_RESIDENT=2) is the strict mode: every element of the index and
 * value arrays is hashed on every call (one parallel pass over the host arrays), so no in-place change and no free +
 * malloc at the same addresses can go unnoticed. */
int spmv_b200_resident_cache(int enable); /* 0 off, 1 sampled, 2 strict; returns the previous setting */
void spmv_b200_resident_drop(void);       /* forget every cached device copy */
/* Plan-time timing of kernel candidates (a few products on scratch vectors when a large matrix is uploaded; only
 * candidates that give the same bits compete).  On by default; SPMV_B200_AUTOTUNE=0 or this switch turns it off, e.g. for
 * a matrix that is used once.  Returns the previous setting. */
int spmv_b200_autotune(int enable);

/* ---- CSR ----------------------------------------------------------------------------- */
/* host arrays (reference CSRMatrix fields, libs/csr_matrix.h:8-16) -> resident device copy */
int spmv_b200_csr_upload(int M, int N, long long nnz, const int *row_ptr, const int *col_idx,
                         const double *values, spmv_b200_csr **out);
/* arrays already on the device (not copied, not owned), e.g. the reference driver's own
 * cudaMalloc'ed d_row_ptr / d_col_idx / d_values (main_cuda.cu:135-145) */
int spmv_b200_csr_wrap_device(int M, int N, long long nnz, const int *d_row_ptr,
                              const int *d_col_idx, const double *d_values, void *stream,
                              spmv_b200_csr **out);
/* COO -> resident CSR built on the device (one stable radix sort of (row, column) keys).  I / J / val as PreMatrix
 * holds them (0-based; reference libs/matrix_parser.h:6-14).  Identical to convert_in_csr + upload for matrices
 * without repeated coordinates; repeated coordinates keep their input order (the reference's order inside such a
 * row is whatever its quicksort leaves, src/utility.c:38-91).  Replaces reference src/csr_matrix.c:63-126 for data
 * that is generated or already resident on the GPU. */
int spmv_b200_csr_from_coo(int M, int N, long long nz, const int *I, const int *J, const double *val,
                           spmv_b200_csr **out);
int spmv_b200_csr_from_coo_device(int M, int N, long long nz, const int *d_I, const int *d_J, const double *d_val,
                                  void *stream, spmv_b200_csr **out);
/* tuning knobs for the plan (0 keeps the default); rebuilds the plan */
int spmv_b200_csr_replan(spmv_b200_csr *A, int tile_items, int long_threshold, int threads_per_row,
                         void *stream);
int spmv_b200_csr_info(const spmv_b200_csr *A, spmv_b200_csr_info_t *info);
/* The arrays of the handle, READ-ONLY: a handle that owns its arrays may hold a private image of them (below), which a
 * write through these pointers would leave stale. */
int spmv_b200_csr_device_arrays(const spmv_b200_csr *A, const int **d_row_ptr, const int **d_col_idx,
                                const double **d_values);
int spmv_b200_csr_download(const spmv_b200_csr *A, int *row_ptr, int *col_idx, double *values);
/* y = A x  (accumulate != 0: y += A x, the reference's serial semantics, src/csr_matrix.c:136) */
int spmv_b200_csr_spmv(const spmv_b200_csr *A, const double *d_x, double *d_y, int accumulate,
                       int algo, void *stream);
/* host x[N] -> device, product, device -> host y[M]; one synchronous call.  Inside, the rows are cut into up to 16
 * windows and the upload of x, the products and the download of y overlap on three streams (hostpath.cu); pinned or
 * cudaHostRegister'ed buffers give the overlap, pageable ones work but serialise. */
int spmv_b200_csr_spmv_host(spmv_b200_csr *A, const double *x, double *y, int accumulate, int algo);
/* ---- fused iterated product (BASELINE config 5; no reference counterpart: the reference only repeats
 * the same product, main_cuda.cu:159-200).  One launch computes
 *     y[r] = (A x)[r] / sqrt(*d_prev_sumsq)            (d_prev_sumsq == NULL: no scaling)
 * writes y, mirrors the rows [lo,hi) listed in `peers` into the peers' buffers (NVLink peer memory obtained
 * with spmv_b200_ipc_open), and leaves per-CTA partial sums of y[r]^2 in d_partials
 * (spmv_b200_csr_partials_count doubles; NULL: skipped).  Matrices with long rows are rejected
 * (SPMV_B200_ERR_INVALID): use spmv_b200_csr_spmv + the vec helpers for those. */
#define SPMV_B200_MAX_PEERS 7
typedef struct {
    int count;
    double *dst[SPMV_B200_MAX_PEERS]; /* peer pointer that corresponds to local row 0 of y            */
    int lo[SPMV_B200_MAX_PEERS];      /* local row range [lo,hi) the peer needs, 0 <= lo <= hi <= M   */
    int hi[SPMV_B200_MAX_PEERS];
} spmv_b200_peers_t;
int spmv_b200_csr_partials_count(const spmv_b200_csr *A);
int spmv_b200_csr_spmv_fused(const spmv_b200_csr *A, const double *d_x, double *d_y, const double *d_prev_sumsq,
                             double *d_partials, const spmv_b200_peers_t *peers, void *stream);

/* The same launch with the exchange of |w|^2 folded in as well -- no collective library call in the loop.
 * Every rank owns a "mailbox" in peer-mappable memory (spmv_b200_ipc_alloc, SPMV_B200_MAILBOX_BYTES, zeroed):
 * 2 parities x world slots of {sum, tag}.  Launch k (mail->iteration = k, 0-based):
 *   start: if k > 0, waits until all `world` slots of parity (k-1)&1 in its OWN mailbox carry tag k (i.e. every rank,
 *          itself included, has finished launch k-1 and its boundary rows have landed here), adds the sums in rank
 *          order and divides every row by the square root;
 *   end:   the last CTA to finish adds the per-CTA partials in a fixed order and writes {sum, tag k+1} into slot
 *          [k&1][rank] of EVERY rank's mailbox (box[r], NVLink peer stores, release at system scope).
 * counter: one zeroed unsigned int in local memory (self-resetting).  status: one int in local memory, set to 1 if a
 * wait gave up after ~2 s (a peer died): results are then invalid, but the kernel never hangs.
 * Launches of one rank must be stream ordered; ranks must not share a GPU (a launch waits for its peers' previous
 * launch). */
#define SPMV_B200_MAX_RANKS 8
#define SPMV_B200_MAILBOX_BYTES (2 * SPMV_B200_MAX_RANKS * 16)
typedef struct {
    int world, rank;
    unsigned long long iteration;
    unsigned long long *box[SPMV_B200_MAX_RANKS]; /* box[r] = rank r's mailbox as mapped HERE; box[rank] is local */
    unsigned int *counter;
    int *status;
} spmv_b200_mail_t;
int spmv_b200_csr_spmv_fused_mail(const spmv_b200_csr *A, const double *d_x, double *d_y, double *d_partials,
                                  const spmv_b200_peers_t *peers, const spmv_b200_mail_t *mail, void *stream);

/* The iterated product as TWO launches per iteration (round 2) -- the fastest form measured:
 *   spmv_b200_csr_spmv_fused_flat   the fused product on a grid as large as the matrix (C consecutive 256-row chunks per
 *       CTA, batch and C timed at plan time): y = (A x) * (*d_inv_norm) (NULL: no scaling), boundary rows mirrored
 *       into `peers`, one partial sum of y^2 per CTA in d_partials (spmv_b200_csr_flat_partials_count doubles).  It
 *       never waits for anything, so the block scheduler balances the SMs as it does for the plain product.  Rows of
 *       up to 12 nonzeros only (one thread per row, the reference's summation order).
 *   spmv_b200_mail_exchange         one CTA: adds the partials in a fixed order, publishes {sum, tag k+1} into slot
 *       [k&1][rank] of every rank's mailbox (mail->iteration = k; same mailbox layout and tag numbering as
 *       spmv_b200_csr_spmv_fused_mail), waits for the tags of all ranks in its own mailbox -- which also proves their
 *       boundary rows have landed -- and leaves {|w_k|^2, 1/|w_k|} (ranks added in rank order) in d_sumsq_out[0..1]; the
 *       next product launch takes d_inv_norm = d_sumsq_out + 1 (the square root and the division are paid once, not once
 *       per thread).  Above 8192 partials the sum is spread over up to 64 CTAs (the last one to finish carries on with
 *       the exchange): d_partials is then CONSUMED (a few entries are overwritten with chunk sums) and mail->counter must
 *       point to one zeroed unsigned int (self-resetting); with mail->counter == NULL one CTA does all of it.  Launches of
 *       one rank must be stream ordered.
 * The HLL twins: spmv_b200_hll_spmv_fused_flat / spmv_b200_hll_flat_partials_count. */
int spmv_b200_csr_flat_partials_count(const spmv_b200_csr *A);
int spmv_b200_csr_spmv_fused_flat(const spmv_b200_csr *A, const double *d_x, double *d_y, const double *d_inv_norm,
                                  double *d_partials, const spmv_b200_peers_t *peers, void *stream);
int spmv_b200_mail_exchange(double *d_partials, int count, const spmv_b200_mail_t *mail, double *d_sumsq_out, void *stream);

/* The asynchronous form of the fused iterated product: no rank ever waits for the CURRENT launch of another rank.
 *   - x lives in a ring of THREE buffers (launch k reads ring[k%3], writes ring[(k+1)%3], own rows locally and the
 *     boundary rows into the neighbours' ring[(k+1)%3]); the caller passes d_x, d_y and peers->dst accordingly;
 *   - the rows a neighbour references are computed FIRST; as soon as they are stored the launch raises a per-neighbour
 *     "halo" tag (k+1) in that neighbour's mailbox, long before the launch ends;
 *   - the scale factor lags one launch: launch k multiplies by 1/sqrt(S[k-2]) (S[j] = |output of launch j|^2 over all
 *     ranks, published by the last CTA of launch j as in the mailbox form; no scaling for k < 2).  The iterate keeps
 *     its direction and stays bounded; lambda = sqrt(S[K-1] S[K-3] / S[K-2]) and v = x / sqrt(S[K-1]) after K launches;
 *   - launch k starts by checking the sums of launch k-2 (4-slot ring) and the halo tags >= k of the ranks it receives
 *     from -- both normally long satisfied.
 * Mailbox layout (SPMV_B200_ASYNC_MAILBOX_BYTES, zeroed, spmv_b200_ipc_alloc): 4 x world slots {sum, tag}, then
 * SPMV_B200_MAX_RANKS halo tags.  counter / bcounter: zeroed unsigned ints in local memory.  Thread-per-row kernel only
 * (matrices whose rows hold at most 12 nonzeros); peers->lo/hi must be chunk-friendly contiguous row ranges. */
#define SPMV_B200_ASYNC_MAILBOX_BYTES (4 * SPMV_B200_MAX_RANKS * 16 + SPMV_B200_MAX_RANKS * 8)
typedef struct {
    int world, rank;
    unsigned long long iteration;
    unsigned long long *box[SPMV_B200_MAX_RANKS]; /* box[r] = rank r's mailbox as mapped HERE; box[rank] is local */
    int num_recv;
    int recv_from[SPMV_B200_MAX_PEERS];           /* ranks whose boundary rows this rank reads */
    int send_to[SPMV_B200_MAX_PEERS];             /* rank behind peers->dst[i] */
    unsigned int *counter, *bcounter;
    int *status;
} spmv_b200_async_t;
int spmv_b200_csr_spmv_fused_async(const spmv_b200_csr *A, const double *d_x, double *d_y, double *d_partials,
                                   const spmv_b200_peers_t *peers, const spmv_b200_async_t *async, void *stream);

/* product restricted to rows [row_begin,row_end) (the reference's per-thread row ranges,
 * src/csr_matrix.c:294-313); other rows of y are left untouched.  Vector kernel; one thread per row when no row holds
 * more than 12 nonzeros, on the pattern form of the private image when the handle holds it (same bits). */
int spmv_b200_csr_spmv_rows(const spmv_b200_csr *A, int row_begin, int row_end, const double *d_x,
                            double *d_y, void *stream);
/* ---- support for the literal "NCCL allgather of x" refresh (BASELINE config 5; no reference counterpart).  One
 * ncclAllGather needs equal slices, the nnz-balanced row ranges differ by a few rows: x is therefore kept in a PADDED
 * rank-major layout, part p's entries at [p*stride, p*stride + rows_p), and the column indices of the resident matrix
 * are rewritten once: c in [starts[p], starts[p+1]) -> p*stride + (c - starts[p]) (monotonic, rows stay sorted).  The
 * matrix must own its arrays (upload / synth / from_coo); N becomes nparts*stride (the kernel plan does not depend on
 * column ids and stays; a private image is dropped). */
int spmv_b200_csr_remap_columns(spmv_b200_csr *A, int nparts, const long long *starts, long long stride, void *stream);
/* largest contiguous row range around the middle row whose columns all lie in [col_lo, col_hi): the rows a rank can
 * multiply BEFORE the refresh of x has landed (their columns are its own slice), overlapping the collective */
int spmv_b200_csr_interior_rows(const spmv_b200_csr *A, long long col_lo, long long col_hi, int *row_lo, int *row_hi,
                                void *stream);
/* Private image.  A handle that owns its arrays (upload, synth, from_coo[_device]; never wrap_device), whose rows hold at
 * most 12 nonzeros and that is large enough for plan-time timing, may keep a second copy of the matrix in HLL layout
 * (hacks of 32 rows, column-major; padding slots marked and skipped, so the products are bit for bit
 * SPMV_B200_ALGO_ROW for every x, accumulate included).  When every slot's column lies within 2^14 of its row
 * (col - row in [-16384, 16383]: banded matrices, 2-D stencils up to a 16383-wide grid) the column field is 2 bytes,
 * col - row with bit 15 marking padding, and the image takes 10 bytes per slot; otherwise it is the column itself with
 * bit 31 marking padding, 12 bytes per slot.  The width follows from the matrix (image_index_bytes).  The values are
 * fp64, or -- when the matrix holds at most 256 distinct 64-bit value patterns (stencils, FEM assembly, unit-weight
 * graphs; +0.0 and -0.0, and NaNs of different payloads, count apart) -- 1-byte codes into a table of those patterns,
 * sorted as uint64; the kernels multiply by the stored double itself in the same order, so y keeps its bits
 * (image_value_bytes 8 or 1) -- except that where two different NaNs meet in one row's sum (a NaN value or x entry and
 * an invalid product such as 0 * Inf) the NaN that results may carry the other payload or sign.  Its kernels need no row_ptr load and find a hack's first slot by arithmetic, which makes them faster on stencils
 * (lap2d 4096^2: DESIGN.md section 3).  The plan times the image with either value field and keeps it only when one
 * times faster than every other candidate and its padding adds at most a quarter to nnz; then AUTO uses it.  Cost, on
 * top of the CSR arrays, per slot: 2 or 4 bytes of column field plus 8 (fp64) or 1 (codes) -- +252 MB on lap2d 4096^2,
 * narrow and coded; +839 MB with fp64 values.
 * Pattern form (spmv_b200_version() >= 106): when the rows hold at most 256 distinct patterns -- a pattern is the row's
 * length, then col - row of each nonzero, then the 64-bit pattern of each value (+0.0 and -0.0, and NaN payloads, count
 * apart) -- and the dictionary of those patterns takes at most 24 KB at 12 bytes per pattern and slot of the longest
 * row, the image may instead be one byte per row naming its pattern (csr_pattern_kernel: lap2d 4096^2, 9 patterns:
 * +16.8 MB; DESIGN.md section 3).  The same bits as ROW, with the same NaN-payload exception as the value codes.  The
 * plan builds it alongside the column-major image under the same padding rule (M times the longest row at most 5/4 of
 * nnz), times both and keeps one of them at most.
 * mode 0 drops the image (AUTO falls back to the plan's choice among ROW / STREAM); mode 1 builds it with fp64 values
 * whenever the matrix is eligible in structure (owned arrays, no row above 12 nonzeros, no long rows), whatever its size
 * or timing, narrow when the matrix qualifies, replacing a coded one, and returns SPMV_B200_ERR_INVALID otherwise; mode 2
 * does the same with the value codes, and returns SPMV_B200_ERR_INVALID, leaving the handle as it was, on a matrix of
 * more than 256 distinct value patterns; mode 3 builds the pattern form, replacing a column-major image, and returns
 * SPMV_B200_ERR_INVALID, leaving the handle as it was, on a matrix that does not qualify for it.  replan decides again;
 * remap_columns drops it.  The fp32, SpMM, fused and host-buffer products do not use it, nor does the row-range product
 * (spmv_b200_csr_spmv_rows) use the column-major image. */
int spmv_b200_csr_set_image(spmv_b200_csr *A, int mode, void *stream);
void spmv_b200_csr_free(spmv_b200_csr *A);

/* plan-free launch on raw device arrays: drop-in for
 * spmv_csr_warp_kernel<<<grid,block>>>(M,row_ptr,col_idx,values,x,y) (main_cuda.cu:238).
 * threads_per_row in {0 (auto from nnz/M),1,2,4,8,16,32}. */
int spmv_b200_csr_spmv_raw(int M, long long nnz, const int *d_row_ptr, const int *d_col_idx,
                           const double *d_values, const double *d_x, double *d_y,
                           int threads_per_row, void *stream);

/* ---- HLL ----------------------------------------------------------------------------- */
/* host HLLMatrix exactly as convert_to_hll builds it (row-major blocks, last block short,
 * NULL arrays for empty blocks; src/hll_matrix.c:37-257) -> column-major device image */
int spmv_b200_hll_upload(const HLLMatrix *hll, int M, int N, spmv_b200_hll **out);
/* device-side conversion of a resident CSR matrix whose rows are column-sorted; identical to
 * convert_to_hll + upload for duplicate-free rows */
int spmv_b200_hll_from_csr(const spmv_b200_csr *A, void *stream, spmv_b200_hll **out);
int spmv_b200_hll_info(const spmv_b200_hll *H, spmv_b200_hll_info_t *info);
/* the column-major device image: hack b owns slots [d_hack_off[b], d_hack_off[b+1]) of d_JA / d_AS, slot(b, r, j) =
 * d_hack_off[b] + 32 j + r (replaces the reference's array of per-block device pointers, main_cuda.cu:369-402) */
int spmv_b200_hll_device_arrays(const spmv_b200_hll *H, const long long **d_hack_off, const int **d_JA, const double **d_AS);
/* device image -> freshly malloc'ed host HLLMatrix in the reference layout (free it with
 * free_hll_matrix); round trip of spmv_b200_hll_upload */
int spmv_b200_hll_download(const spmv_b200_hll *H, HLLMatrix *out);
int spmv_b200_hll_spmv(const spmv_b200_hll *H, const double *d_x, double *d_y, void *stream);
/* spmv_b200_hll_spmv picks between the two kernels below from the mean hack width */
/* one-warp-per-hack slice kernel, 128/256-bit loads straight from HBM */
int spmv_b200_hll_spmv_slice(const spmv_b200_hll *H, const double *d_x, double *d_y, void *stream);
/* one warp per hack, lane = row, in the order of spmv_hll_serial (bit-identical), no shared memory */
int spmv_b200_hll_spmv_rows(const spmv_b200_hll *H, const double *d_x, double *d_y, void *stream);
/* persistent TMA bulk-copy pipeline (shared-memory staging) */
int spmv_b200_hll_spmv_stream(const spmv_b200_hll *H, const double *d_x, double *d_y, void *stream);
int spmv_b200_hll_spmv_host(spmv_b200_hll *H, const double *x, double *y);
/* product restricted to hacks [hack_begin,hack_end) (reference per-thread block ranges,
 * src/hll_matrix.c:376-408) */
int spmv_b200_hll_spmv_hacks(const spmv_b200_hll *H, int hack_begin, int hack_end, const double *d_x,
                             double *d_y, void *stream);
/* ---- fused iterated product on the HLL image: the twins of spmv_b200_csr_spmv_fused / _fused_mail (same Epilogue:
 * y = (A x) / sqrt(*d_prev_sumsq) or the mailbox sum, per-CTA partials of y^2 in d_partials, boundary rows mirrored into
 * `peers`, last CTA publishes |w|^2).  The reference splits HLL work by block ranges (src/hll_matrix.c:376-408,471-498):
 * a rank owns a contiguous range of hacks, so its local row 0 is a multiple of 32 rows of the global matrix.  For the
 * same row partition the results are bitwise those of the CSR iteration. ---- */
int spmv_b200_hll_partials_count(const spmv_b200_hll *H);
int spmv_b200_hll_spmv_fused(const spmv_b200_hll *H, const double *d_x, double *d_y, const double *d_prev_sumsq,
                             double *d_partials, const spmv_b200_peers_t *peers, void *stream);
int spmv_b200_hll_spmv_fused_mail(const spmv_b200_hll *H, const double *d_x, double *d_y, double *d_partials,
                                  const spmv_b200_peers_t *peers, const spmv_b200_mail_t *mail, void *stream);
/* the two-launch form (see spmv_b200_csr_spmv_fused_flat; the exchange kernel spmv_b200_mail_exchange is shared) */
int spmv_b200_hll_flat_partials_count(const spmv_b200_hll *H);
int spmv_b200_hll_spmv_fused_flat(const spmv_b200_hll *H, const double *d_x, double *d_y, const double *d_inv_norm,
                                  double *d_partials, const spmv_b200_peers_t *peers, void *stream);
void spmv_b200_hll_free(spmv_b200_hll *H);

/* ---- multi-vector products Y = A X (SpMM), fp64, device arrays (spmv_b200_version() >= 101) ----------------------------
 * X is N x k and Y is M x k, both row-major with leading dimensions ldx >= k and ldy >= k counted in elements: element
 * (i, c) is at i*ld + c (64-bit offsets).  One call streams the matrix once for all k columns.  Only rows < M and columns
 * < k of Y are written; the elements between k and ldy are never touched.  X and Y must not overlap.
 *   CSR, rows of at most info.long_threshold nonzeros: column c of Y is bit for bit the serial loop csr_matrix_vector_mult
 *     on column c of X (one lane per (row, column), index order, mul and add rounded separately), i.e. the bits of
 *     spmv_b200_csr_spmv(..., SPMV_B200_ALGO_ROW) on that column; accumulate != 0 starts each sum from Y's value.
 *   CSR, longer rows (the plan's long rows, in fragments of 8192 nonzeros): each fragment is summed as 32 fixed
 *     index-ordered sub-ranges and a fixed tree, the fragments are added in order; no atomics.  Within
 *     (len + 2) 2^-53 sum_j |a_ij x_jc| of the exact sum, identical bits from call to call, and the bits of a column do not
 *     depend on k, ldx, ldy or the column's position in X.
 *   HLL: column c is bit for bit spmv_hll_serial on column c, padding slots (x 0.0) included -- the bits of
 *     spmv_b200_hll_spmv_rows.  No accumulate flag (as spmv_b200_hll_spmv).
 * k = 0 and M = 0 are no-ops; with nnz = 0, Y becomes zero (or is left as it is with accumulate).  A negative k, ldx < k,
 * ldy < k, or a NULL handle or array with k > 0 returns SPMV_B200_ERR_INVALID and launches nothing.  The CSR product
 * on a matrix with long rows keeps num_fragments x 32 partial sums on the handle (allocated by the first such call, freed
 * with the plan): as with spmv_b200_csr_spmv, products on one handle must be stream-ordered. */
int spmv_b200_csr_spmm(const spmv_b200_csr *A, int k, const double *d_X, long long ldx, double *d_Y, long long ldy,
                       int accumulate, void *stream);
int spmv_b200_hll_spmm(const spmv_b200_hll *H, int k, const double *d_X, long long ldx, double *d_Y, long long ldy,
                       void *stream);
/* Host-buffer twins (spmv_b200_version() >= 108): host X -> device, Y = A X (or Y += A X), device -> host Y; one
 * synchronous call, with the conventions of spmv_b200_csr_spmm / spmv_b200_hll_spmm above (row-major, ldx >= k and
 * ldy >= k, 64-bit offsets, only rows < M and columns < k of Y written -- the elements between k and ldy are never
 * touched, not even by a zero-copy store -- no overlap of X and Y, k = 0 and M = 0 no-ops, nnz = 0 gives zero or leaves
 * Y with accumulate, bad k, ld or a NULL pointer SPMV_B200_ERR_INVALID before anything is launched, accumulate on CSR
 * only).  Every column of Y has the bits spmv_b200_{csr,hll}_spmm gives on the same handle for the same X, whatever k,
 * ldx, ldy, the window count or column-block width, pinned or pageable buffers, zero-copy or staged Y, long rows or not.
 * As spmv_b200_csr_spmv_host does for one vector, the call cuts the rows into up to 16 windows (rows for CSR, hacks for
 * HLL) and overlaps the upload of X in pieces, the products of the windows and the download of Y on three streams
 * (hostpath.cu); the long rows of a CSR plan run after the last piece.  Y is stored by the kernels straight into a
 * pinned or cudaHostRegister'ed buffer when ldy > k or a row of Y holds at most 16 bytes (measured, DESIGN.md section
 * 3, "Host buffers"); it is staged and downloaded otherwise, and always with accumulate.  SPMV_B200_HOST_ZEROCOPY=0 forces staging.  Pinned buffers give the overlap; pageable ones work but
 * serialise.
 * Device memory: the handle keeps a staging buffer for N x kc elements of X (plus M x kc of Y when Y is staged), kc = k
 * when that fits half of the free device memory, else column blocks of the largest kc that does; it is reused and grown
 * by later calls and freed with the handle (spmv_b200_csr_free / spmv_b200_hll_free), as are the window plan, streams
 * and events of these calls, made by the first one. */
int spmv_b200_csr_spmm_host(spmv_b200_csr *A, int k, const double *X, long long ldx, double *Y, long long ldy, int accumulate);
int spmv_b200_hll_spmm_host(spmv_b200_hll *H, int k, const double *X, long long ldx, double *Y, long long ldy);

/* ---- fp32 storage with fp64 arithmetic (BASELINE.json: y within 1e-5 relative of the serial fp64 product).  The value
 * stream, x and y are float (algorithmic bytes 8 nnz + 4 (M+1) + 4 M + 4 N instead of 12 nnz + ...); every product is
 * formed and summed in double and rounded once on the store.  enable_f32 adds a float copy of the values to the
 * resident matrix (the indices, plans and the fp64 values stay).  CSR algo: AUTO, ROW, VECTOR or BINNED. ---- */
int spmv_b200_csr_enable_f32(spmv_b200_csr *A, void *stream);
int spmv_b200_csr_spmv_f32(const spmv_b200_csr *A, const float *d_x, float *d_y, int accumulate, int algo, void *stream);
int spmv_b200_csr_spmv_host_f32(spmv_b200_csr *A, const float *x, float *y);
int spmv_b200_hll_enable_f32(spmv_b200_hll *H, void *stream);
int spmv_b200_hll_spmv_f32(const spmv_b200_hll *H, const float *d_x, float *d_y, void *stream);
int spmv_b200_hll_spmv_host_f32(spmv_b200_hll *H, const float *x, float *y);
/* Multi-vector products on the float copy (spmv_b200_version() >= 105): X, Y and the values are float, the conventions
 * those of spmv_b200_csr_spmm / spmv_b200_hll_spmm (row-major, ld >= k, 64-bit offsets, only rows < M and columns < k of
 * Y written, no overlap, k = 0 and M = 0 no-ops, nnz = 0 gives zero or leaves Y with accumulate).  A widened float times
 * a widened float is exact in double (24 + 24 significand bits), so the only roundings are the adds and the final store:
 *   CSR, rows of at most info.long_threshold nonzeros: column c of Y is bit for bit spmv_b200_csr_spmv_f32(...,
 *     SPMV_B200_ALGO_ROW) on column c of X -- the serial fp64 loop over the widened values and x, rounded once to float;
 *     accumulate != 0 starts each sum from (double)Y[i,c].
 *   CSR, longer rows: each fragment summed as the same fixed sub-ranges and tree as the fp64 product, in double, the
 *     fragments added in order and rounded once; within ulp32(y) + (len + 2) 2^-53 sum_j |a_ij x_jc| of the exact sum,
 *     identical bits from call to call, and the bits of a column do not depend on k, ldx, ldy or its position in X.
 *   HLL, every row (hacks of any width): serial in j with the padding slots included, rounded once -- the bits of the
 *     lane-per-row kernel hll_row_kernel<B,float>.  No accumulate flag.
 * Without spmv_b200_{csr,hll}_enable_f32 on the handle they return SPMV_B200_ERR_INVALID and launch nothing; bad k, ld or
 * NULL arguments are rejected as by the fp64 forms.  The CSR form shares the fp64 form's partials buffer. */
int spmv_b200_csr_spmm_f32(const spmv_b200_csr *A, int k, const float *d_X, long long ldx, float *d_Y, long long ldy,
                           int accumulate, void *stream);
int spmv_b200_hll_spmm_f32(const spmv_b200_hll *H, int k, const float *d_X, long long ldx, float *d_Y, long long ldy,
                           void *stream);
/* Host-buffer twins of the two above (spmv_b200_version() >= 108), as spmv_b200_csr_spmm_host / _hll_spmm_host: the
 * bits of spmv_b200_{csr,hll}_spmm_f32 on the same handle.  They call spmv_b200_{csr,hll}_enable_f32 themselves. */
int spmv_b200_csr_spmm_host_f32(spmv_b200_csr *A, int k, const float *X, long long ldx, float *Y, long long ldy, int accumulate);
int spmv_b200_hll_spmm_host_f32(spmv_b200_hll *H, int k, const float *X, long long ldx, float *Y, long long ldy);
/* Which form of the row kernel enable_f32 timed fastest for this matrix: 1..8 = csr_row_kernel / hll_row_kernel with that
 * many loads in flight per row; >= 16 = form (id - 16) of csr_rowm_kernel / hll_rowm_kernel (index-only predicates, so
 * that every load of a step is issued ahead of the first multiply; rows per thread, loads in flight per row and CTAs
 * per SM from spmv_b200_row_form_describe); HLL only, 64 + b = hll_rowu_kernel with b loads in flight (regular images:
 * hack offsets by arithmetic, no offset load); 0 before enable_f32.  The environment variable SPMV_B200_ROW_MULTI=k
 * (k >= 1) sends every row-kernel launch, fp64 included, through form k - 1: all forms give the same bits, which is
 * what the parity tests use it for. */
int spmv_b200_csr_row_form_f32(const spmv_b200_csr *A);
int spmv_b200_hll_row_form_f32(const spmv_b200_hll *H);
/* the same for the fp64 lane-per-row kernel of an HLL image: 1..8 = hll_row_kernel with that batch, 64 + b = hll_rowu_kernel */
int spmv_b200_hll_row_form(const spmv_b200_hll *H);
/* number of multi-row forms of a format (SPMV_B200_FORMAT_CSR / _HLL), and what form `index` is */
int spmv_b200_row_forms(int format);
int spmv_b200_row_form_describe(int format, int index, int *rows_per_thread, int *batch, int *ctas_per_sm);

/* ---- timing harness on a resident matrix: the reference driver's protocol (main_cuda.cu:159-200: cudaEvents around
 * every product, the first `warmup` iterations not counted, mean over the rest) behind one call, so that a C
 * driver needs no CUDA runtime of its own.  x: host vector, uploaded once (as main_cuda.cu:145); y: host result of
 * the last product (may be NULL).  kernel for HLL: 0 automatic, 1 slice kernel, 2 stream kernel, 3 lane-per-row kernel. ---- */
int spmv_b200_csr_time(spmv_b200_csr *A, const double *x, double *y, int algo, int warmup, int iters,
                       double *mean_seconds, double *min_seconds);
int spmv_b200_hll_time(spmv_b200_hll *H, const double *x, double *y, int kernel, int warmup, int iters,
                       double *mean_seconds, double *min_seconds);

/* ---- synthetic matrices generated on the device (rows [row_begin,row_end) of the global
 * matrix, global column ids, local row_ptr starting at 0); see SURVEY.md section 8(d) ---- */
int spmv_b200_synth_csr(int kind, long long p0, long long p1, int p2, unsigned long long seed,
                        long long row_begin, long long row_end, void *stream, spmv_b200_csr **out);
/* number of nonzeros in rows [0,row) of a synthetic matrix (closed form; no device needed) */
long long spmv_b200_synth_row_offset(int kind, long long p0, long long p1, int p2, long long row);
/* x_i = (hash(seed,i) in (0,1]) */
int spmv_b200_synth_vector(double *d_x, long long n, unsigned long long seed, void *stream);

/* ---- dense vector helpers for the iterated product (power method, BASELINE config 5) ---- */
int spmv_b200_vec_fill(double *d_v, long long n, double value, void *stream);
/* *d_out = sum v_i^2, deterministic two-stage tree (independent of n's partition into CTAs
 * only through a fixed CTA count); d_ws must hold spmv_b200_vec_ws_doubles() doubles */
int spmv_b200_vec_ws_doubles(void);
int spmv_b200_vec_sumsq(const double *d_v, long long n, double *d_ws, double *d_out, void *stream);
/* d_dst[i] = d_src[i] / sqrt(*d_sumsq)   (no host round trip) */
/* *d_out = sum of n doubles, one CTA, fixed tree (n is small: the per-CTA partials above) */
int spmv_b200_vec_sum(const double *d_in, int n, double *d_out, void *stream);
int spmv_b200_vec_scale_by_inv_norm(double *d_dst, const double *d_src, long long n,
                                    const double *d_sumsq, void *stream);

/* d_peer_dst[p][i] = d_src[i] for p < npeers, i < n: a slice of x pushed into the replicas of the other ranks with NVLink
 * peer stores (the all-gather of the "allgather_peer" exchange written against peer memory; `ctas` = grid size, 0 = two
 * CTAs per SM).  256-bit loads / 256-bit peer stores when the source and every target share their offset within 32
 * bytes (the same row range of equally aligned replicas), scalar otherwise.  d_peer_dst is a HOST array of device
 * pointers.  No ordering is implied towards the peers: follow it with spmv_b200_mail_exchange (tag after fence). */
int spmv_b200_vec_push(const double *d_src, long long n, int npeers, double *const *d_peer_dst, int ctas, void *stream);

/* ---- peer memory for the fused exchange: device buffers that other ranks (processes) on the same NVLink
 * domain can map.  handle is an opaque 64-byte token (cudaIpcMemHandle_t) to ship to the peers. ---- */
int spmv_b200_ipc_alloc(long long bytes, void **d_ptr, unsigned char handle[64]);
int spmv_b200_ipc_open(const unsigned char handle[64], void **d_peer_ptr);
int spmv_b200_ipc_close(void *d_peer_ptr);
int spmv_b200_ipc_free(void *d_ptr);

/* ---- 1..8 GPUs of one box from plain C: the row-partitioned product and the iterated product (power method, BASELINE
 * config 5).  ONE process, one host thread, peer access between the devices (multi.cu); devices 0 .. ngpus-1.  The
 * reference has no multi-GPU path (main_cuda.cu:128-200 drives device 0 only); the partition is its own rule for OpenMP
 * threads -- contiguous row ranges balanced by nnz (src/csr_matrix.c:167-266), cut on 32-row block boundaries for HLL
 * (src/hll_matrix.c:471-498) -- with GPUs in the role of threads (fewer GPUs are used when the rule yields fewer
 * non-empty ranges).  Every GPU holds its rows and a replica of x in a padded rank-major layout (part p at
 * [p*stride, p*stride + rows_p)); the column indices are rewritten once on the device.
 *   spmv_b200_multi_iterate(ctx, iters, exchange, &lambda, &ms): iters times  y = A x; lambda = |y|_2; x = y / lambda
 *     SPMV_B200_EXCHANGE_MAILBOX    ONE fused launch per GPU per iteration, boundary rows and |w|^2 travel through NVLink
 *                                   peer stores and mailboxes (spmv_b200_csr_spmv_fused_mail / _hll_), no collective
 *     SPMV_B200_EXCHANGE_ALLGATHER  product, |y|^2, 1-double ncclAllReduce, scale, ONE in-place ncclAllGather of x
 *                                   (NCCL resolved with dlopen at first use; works for skewed matrices too)
 *     SPMV_B200_EXCHANGE_ALLGATHER_PEER  the same iteration without NCCL: |y|^2 through the peer mailboxes
 *                                   (spmv_b200_mail_exchange), then every GPU copies its slice into the replicas of all
 *                                   the others over NVLink (one cudaMemcpyPeerAsync per peer: the copy engines drive
 *                                   the links, 750 GB/s per direction measured against NCCL's 500-600); any matrix
 *   ms = device time per iteration, cudaEvents on every GPU's stream, maximum over the GPUs.  lambda = |A v_{k-1}| of
 *   the last iteration.  The iterate continues across calls; spmv_b200_multi_reset starts again from x0 (NULL: ones)
 *   and is required before switching the exchange mode. ---- */
#define SPMV_B200_FORMAT_CSR 0
#define SPMV_B200_FORMAT_HLL 1
#define SPMV_B200_EXCHANGE_MAILBOX 0
#define SPMV_B200_EXCHANGE_ALLGATHER 1
#define SPMV_B200_EXCHANGE_ALLGATHER_PEER 2
typedef struct spmv_b200_multi spmv_b200_multi;
typedef struct {
    int ngpus, format;
    long long M, N, nnz;
    long long stride;                               /* slot size of the padded x                                   */
    int fused_ok;                                   /* 0: rows above the long-row threshold, MAILBOX is refused     */
    long long row_begin[SPMV_B200_MAX_RANKS], row_end[SPMV_B200_MAX_RANKS], nnz_part[SPMV_B200_MAX_RANKS];
    long long halo_doubles[SPMV_B200_MAX_RANKS];    /* doubles a GPU receives from its neighbours per iteration     */
} spmv_b200_multi_info_t;
/* synthetic matrix generated on the devices (kinds and parameters of spmv_b200_synth_csr) */
int spmv_b200_multi_init_synth(int ngpus, int format, int kind, long long p0, long long p1, int p2, unsigned long long seed,
                               spmv_b200_multi **out);
/* host CSR arrays (reference CSRMatrix fields); partitioned with prepare_thread_distribution, uploaded slice by slice */
int spmv_b200_multi_init_csr(int ngpus, int format, int M, int N, long long nnz, const int *row_ptr, const int *col_idx,
                             const double *values, spmv_b200_multi **out);
int spmv_b200_multi_info(const spmv_b200_multi *ctx, spmv_b200_multi_info_t *info);
int spmv_b200_multi_reset(spmv_b200_multi *ctx, const double *x0);
int spmv_b200_multi_iterate(spmv_b200_multi *ctx, int iters, int exchange, double *lambda, double *ms_per_iteration);
/* the normalised iterate v_k (host, N doubles, original numbering) */
int spmv_b200_multi_get_x(spmv_b200_multi *ctx, double *x_host);
/* one row-partitioned product y = A x on host vectors (x: N doubles, y: M doubles) */
int spmv_b200_multi_spmv(spmv_b200_multi *ctx, const double *x_host, double *y_host);
void spmv_b200_multi_free(spmv_b200_multi *ctx);

#ifdef __cplusplus
}
#endif
#endif /* SPMV_B200_H */
