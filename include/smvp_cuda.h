/*
 * include/smvp_cuda.h -- C ABI of libsmvp_cuda, the B200 (sm_100a) engine behind the CSR and TJDS
 * hot path of circletile/smvp-toolkit.
 *
 * The reference has no plugin / FFI layer: the path is two functions called straight from main(),
 *
 *     double *smvp_csr_compute (MMRawData *coo, int rows,           int nnz, int iters, struct _time_data_ *t);   main-cli.c:325  (call site :1457)
 *     double *smvp_tjds_compute(MMRawData *coo, int rows, int cols, int nnz, int iters, struct _time_data_ *t);   main-cli.c:734  (call site :1469)
 *
 * Each of them does "build the format" + "repeat the multiply `iters` times, timing each pass".
 * This header splits exactly those two steps per format (names fixed by the project brief):
 *
 *     smvp_csr_build   replaces main-cli.c:336-365   (qsort by (row,col) + CSR fill)
 *     smvp_csr_mult    replaces main-cli.c:402-456   (the timed multiply loop + per-iteration ms)
 *     smvp_tjds_build  replaces main-cli.c:755-967   (TJDS conversion, incl. the x permutation table)
 *     smvp_tjds_mult   replaces main-cli.c:1004-1024 (+ :1120-1148 timing)
 *     smvp_time_stats  replaces main-cli.c:428-456 / calcStDevDouble :114-130
 *
 * Plain C: pointers and sizes only.  All indices int32, all values IEEE fp64 (the reference's types).
 * Errors are returned (0 = ok, negative = SMVP_E_*); the library never calls exit() and never falls
 * back to a CPU implementation: without a CUDA device every entry point returns SMVP_E_CUDA.
 *
 * Ownership: the caller owns every host buffer and every device buffer it passes in; the library
 * owns the device memory behind a handle until smvp_*_free.  `coo` is const (the reference sorts the
 * caller's array in place, main-cli.c:340/:766; callers of this ABI keep their array untouched so
 * --all-algs can build both formats from one load).
 *
 * Input contract: 0 <= row < rows, 0 <= col < cols (violations -> SMVP_E_RANGE); (row, col) pairs
 * unique -- duplicates are undefined in the reference too (its qsort order is unspecified and its TJDS
 * rank code reads uninitialised memory, main-cli.c:820-824).
 */
#ifndef SMVP_CUDA_H
#define SMVP_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#pragma GCC visibility push(default)

#define SMVP_OK 0
#define SMVP_E_ARG (-1)         /* null pointer / negative size / bad enum                   */
#define SMVP_E_ALLOC (-2)       /* host or device allocation failed                          */
#define SMVP_E_CUDA (-3)        /* CUDA runtime error (no device, launch failure, ...)       */
#define SMVP_E_RANGE (-4)       /* a coordinate lies outside [0,rows) x [0,cols)             */
#define SMVP_E_TOOBIG (-5)      /* nnz does not fit the format's int32 offsets               */
#define SMVP_E_PATTERN (-6)     /* a (row, col) pair the handle does not store               */

/* == MMRawData (main-cli.c:42-47): 16 bytes, no padding.  0-based coordinates. */
typedef struct smvp_coo
{
    int32_t row;
    int32_t col;
    double val;
} smvp_coo;

typedef struct smvp_csr smvp_csr;   /* opaque: CSRData  (main-cli.c:61-66) resident in HBM */
typedef struct smvp_tjds smvp_tjds; /* opaque: TJDSData (main-cli.c:70-75) resident in HBM */

/* CSR multiply variants */
#define SMVP_CSR_AUTO 0   /* pick from the row-length distribution measured at build time        */
#define SMVP_CSR_VECTOR 1 /* sub-warp per row, 128-bit loads, __shfl_xor_sync reduction           */
#define SMVP_CSR_MERGE 2  /* merge-path over cp.async.bulk (TMA) staged tiles, skew-proof         */

/* TJDS multiply variants */
#define SMVP_TJDS_ATOMIC 0        /* coalesced jagged-diagonal streaming, fp64 atomicAdd scatter into y */
#define SMVP_TJDS_DETERMINISTIC 1 /* order-independent INTEGER accumulation in fixed point, scaled per row by a bound known
                                     before the multiply, one final rounding; bit-identical run to run (and between the
                                     straight and the skewed walk, with and without row relabelling).  Exactly:
                                       e(v) = ilogb(v) + 1 (so |v| < 2^e(v)),
                                       T_r  = max e(a_rj) over the nonzero entries of row r
                                              + ceil(log2 count_r) (every stored entry, explicit zeros included)
                                              + max e(x_c) over the nonzero x_c of the columns that hold entries
                                              (x entries of empty columns are never read and change nothing),
                                       p_j  = fl(a_rj * x_j),
                                       y_r  = RN( sum_j trunc0(p_j * 2^(94 - T_r)) * 2^(T_r - 94) )
                                     with trunc0 toward zero, the sum exact (integers) and RN ONE round-to-nearest-even
                                     to fp64, subnormal results included; a row without a nonzero product is +0.0.
                                     y_r is the CORRECTLY ROUNDED row sum whenever every product is a multiple of
                                     2^(T_r - 94), e.g. |p_j| >= 2^(T_r - 42) for all j (products within 2^-42 of the
                                     row bound).  Otherwise |y_r - sum_j p_j| <= ulp(y_r) / 2 + count_r * 2^(T_r - 94):
                                     a row whose products sit far below its bound (cancellation, or a column of x much
                                     larger than the ones the row reads) loses the digits under 2^(T_r - 94).        */
#define SMVP_TJDS_DETERMINISTIC_FAST 2 /* the same with 2^(62 - T_r) in place of 2^(94 - T_r): one 64-bit word per product
                                     instead of two.  Just as reproducible (integer sums), one reduction per run and
                                     half the accumulator traffic; |y_r - sum_j p_j| <= ulp(y_r) / 2 +
                                     count_r * 2^(T_r - 62), exact only for products that are multiples of 2^(T_r - 62)
                                     (|p_j| >= 2^(T_r - 10)).  The bound is NORMWISE -- 2^-9 of what one fp64 addition at
                                     magnitude 2^T_r rounds away -- not relative to |y_r|: an x whose entries span many
                                     orders of magnitude can cost a row with small products digits that the two-word
                                     variant keeps.                                                                  */

/* ---- statistics of the per-iteration times: struct _time_data_ (main-cli.c:87-95), same field order */
typedef struct smvp_time_stats_t
{
    double time_total;
    double time_avg;
    double time_stdev; /* population stdev, sqrt(sum((t-mean)^2)/n)  (main-cli.c:129) */
    double time_min;
    double time_max;
} smvp_time_stats_t;

int smvp_time_stats(const double *ms_each, int n, smvp_time_stats_t *out);

/* ---- format builders: host COO (array of smvp_coo == MMRawData) -> format arrays in HBM ---- */
int smvp_csr_build(const smvp_coo *coo, int32_t rows, int32_t cols, int64_t nnz, smvp_csr **out);
int smvp_tjds_build(const smvp_coo *coo, int32_t rows, int32_t cols, int64_t nnz, smvp_tjds **out);

/* ---- multiply loops, host vectors: x_host[cols] -> y_host[rows], repeated `iters` times.
 * ms_each (may be NULL) receives `iters` per-iteration device times in milliseconds, taken with CUDA
 * events around the multiply only; the zero-fill of y is outside the bracket, as in the reference
 * (main-cli.c:405 vs :408/:419).  x is copied to the device once and y copied back once per call
 * (the reference reports the last iteration's y).  For vectors of millions of entries smvp_csr_mult overlaps
 * both copies with the first / last pass, and uploads only the part of x between the smallest and the largest
 * column index the matrix holds (the rest is never read) -- when BOTH vectors are page-locked (smvp_host_alloc,
 * cudaHostAlloc, cudaHostRegister); pageable buffers are served by plain copies (an asynchronous copy from pageable
 * memory blocks the host, which would serialise the pieces).  ms_each of such a pass is the sum of the device
 * brackets of its tile ranges (short launches: more GPU time than one whole-matrix launch).
 * Small matrices (rows + cols + nnz < 2^22): the loop runs batched -- one untimed pass, one pass timed exactly, the
 * others replayed from CUDA graphs 50 at a time (a pass is charged its batch's time / 50); SMVP_EXACT_ITER_TIMES=1
 * restores one event pair and one synchronisation per iteration.
 * smvp_tjds_mult: diag_limit <= 0 walks every jagged diagonal.  diag_limit = k > 0 walks only the
 * first k (and, like the shipped loop, skips a final diagonal that holds a single element): with
 * k = smvp_tjds_info().ref_diag_limit this reproduces the reference's golden TJDS report files,
 * which contain a truncated product (main-cli.c:865 evaluated before the sort at :868).        */
int smvp_csr_mult(smvp_csr *A, const double *x_host, double *y_host, int iters, double *ms_each, int variant);
int smvp_tjds_mult(smvp_tjds *A, const double *x_host, double *y_host, int iters, double *ms_each, int variant,
                   int32_t diag_limit);

/* ---- device-resident entry points (synthetic matrices that never exist on the host, benchmarks,
 * multi-GPU shards).  All pointers are device pointers of the current device; `stream` is a
 * cudaStream_t passed as void* (NULL = default stream).  Calls are asynchronous on `stream` unless
 * noted.  COO here is structure-of-arrays.                                                        */
int smvp_csr_build_device(const int32_t *d_row, const int32_t *d_col, const double *d_val, int32_t rows,
                          int32_t cols, int64_t nnz, smvp_csr **out); /* synchronous */
int smvp_tjds_build_device(const int32_t *d_row, const int32_t *d_col, const double *d_val, int32_t rows,
                           int32_t cols, int64_t nnz, smvp_tjds **out); /* synchronous */
/* Declares the x of the following passes (the reference multiplies the SAME x `-n` times, main-cli.c:368-369 /
 * :402-420).  Handles whose multiply plan relabels the column space by popularity (power-law matrices whose x
 * exceeds L2, see smvp_csr_info_t.x_relabel) form their permuted copy of x here, once, the way the reference
 * permutes x once for TJDS (main-cli.c:907-923); for all other handles the call only records the pointer.
 * d_x stays owned by the caller and must remain valid and unchanged while passes with d_x == NULL run.
 * The first call on a handle may synchronise (it decides and builds the plan).                              */
int smvp_csr_set_x_device(smvp_csr *A, const double *d_x, void *stream);
/* one pass y = A x.  d_x == NULL: the x last given to smvp_csr_set_x_device.  d_x != NULL is always
 * correct too; on a relabelled handle it costs one extra permutation pass over x per call.             */
int smvp_csr_mult_device(smvp_csr *A, const double *d_x, double *d_y, int variant, void *stream);
/* The merge-path kernel runs as a persistent grid that fills every SM; `ctas_per_sm` > 0 makes it leave room for that
 * many CTAs of ANOTHER kernel per SM (default 0).  A caller that runs a small kernel beside the multiply -- the
 * multi-GPU path pushes the previous pass's rows to its peers while the next pass multiplies -- sets 1: without the
 * room part of the persistent grid starts only when the co-runner retires and the pass ends that much later. */
int smvp_csr_set_corunner_headroom(smvp_csr *A, int ctas_per_sm);
/* one pass y = A x with the result stored into n_out (<= 8) destinations at once: d_y_list[k][r] = y[r] for
 * every row r of A and every k.  The destinations may be peer-mapped buffers of other GPUs (NVLink symmetric
 * memory): this is how the row-partitioned multi-GPU path fuses the "allgather of y" into the SpMV epilogue.
 * d_y_list is a HOST array of device pointers; the destinations are write-only for the library.             */
int smvp_csr_mult_device_fanout(smvp_csr *A, const double *d_x, double *const *d_y_list, int n_out, int variant,
                                void *stream);
/* x_perm[p] = x[perm[p]] into the handle (the reference permutes x once, at build time, main-cli.c:907-923) */
int smvp_tjds_set_x_device(smvp_tjds *A, const double *d_x, void *stream);
/* one pass y = A x with the x last given to smvp_tjds_set_x_device; zero-fills y first */
int smvp_tjds_mult_device(smvp_tjds *A, double *d_y, int variant, int32_t diag_limit, void *stream);

/* ---- transposed product y = A^T x (BiCG, QMR, LSQR and CGNE need it once per iteration; pull-direction graph walks
 * multiply by A^T).  Two routes, one per format:
 *   CSR   a second handle holds A^T; every CSR plan (row patterns, relabelling, pipelined host call, fan-out) serves it
 *         through the ordinary smvp_csr_mult* calls.
 *   TJDS  the handle itself: TJDS stores A by column, so A^T x is a gather along each column -- no atomics, no second
 *         copy of the matrix.                                                                                         */
/* A^T as a new, independent CSR handle, built on the device from A's arrays (A is not modified; free the two in any
 * order).  Row c of the result lists A's column c in ascending row order, i.e. its arrays are bit-identical to what
 * smvp_csr_build makes from the COO with rows and columns swapped.  Synchronous, like the builders.  The new handle
 * starts with every plan undecided and no co-runner headroom.  It holds as much HBM as A, and its build takes about as
 * much temporary HBM as a build of A from a device COO.                                                            */
int smvp_csr_transpose(const smvp_csr *A, smvp_csr **out);
/* one pass y = A^T x: d_x has A->rows entries, d_y A->cols.  Every entry of d_y is written (+0.0 for an empty column).
 * Deterministic, no atomics.  Column c's terms val * x[row] are taken in ascending row order: columns of at most 32
 * entries are summed left to right from +0.0 (bit-identical to the sequential transposed loop); longer columns in
 * chunks of 32 entries, each summed left to right from +0.0, the chunk sums then added left to right from +0.0 -- the
 * order is a function of the matrix alone.  The first call on a handle may synchronise (plan + scratch: one double per
 * chunk of a column longer than 32 entries, counted in smvp_tjds_info_t.device_bytes).  A pass is one launch when no
 * column holds more than 32 entries, two otherwise.  Independent of smvp_tjds_set_x_device and of the row relabelling
 * of A x; the handle's x and plans stay as they are.                                                              */
int smvp_tjds_mult_transpose_device(smvp_tjds *A, const double *d_x, double *d_y, void *stream);
/* the same with host vectors x_host[rows] -> y_host[cols], `iters` timed passes: the -n loop of smvp_tjds_mult (x copied
 * to the device once and y back once per call; ms_each as there, exact or batched for small matrices)             */
int smvp_tjds_mult_transpose(smvp_tjds *A, const double *x_host, double *y_host, int iters, double *ms_each);

/* ---- scaled, accumulating multiply y = alpha * A x + beta * y (and alpha * A^T x + beta * y): the update Krylov solvers
 * repeat -- a residual r = b - A x is alpha = -1, beta = 1 with y = b; LSQR's u <- A v - a u and v <- A^T u - b v.  The
 * update is fused into the store of the multiply: one read of y instead of a temporary and a second vector pass.
 *
 * For every row r let s_r be what the plain call (same handle, variant, plan and diag_limit) stores into y[r], bit for
 * bit.  These calls store
 *     beta != 0:  y[r] = fl( fl(alpha * s_r) + fl(beta * y[r]) )   (each product and the sum rounded separately, no FMA)
 *     beta == 0:  y[r] = fl(alpha * s_r), and y is NEVER READ (uninitialised or NaN-filled y is fine, as in BLAS; -0.0
 *                 counts as 0)
 * alpha = 0 does not skip the matrix: the formula holds as written, so an Inf or NaN in A x still propagates.
 * alpha = 1, beta = 0 is the plain call: the same kernels and launches, the same bits.
 * Exception, inherited from the plain pass: SMVP_TJDS_ATOMIC (and the deterministic variants routed to it,
 * det_route = -1): s_r is the atomic pass's value, which is not reproducible run to run.  The deterministic variants are
 * bit-exact.
 * Aliasing: d_y may not be the x the kernels read -- for CSR d_x, or the x of smvp_csr_set_x_device when d_x == NULL;
 * for the TJDS transposed call d_x.  Those calls return SMVP_E_ARG; a partial overlap is undefined.  TJDS A x reads the
 * handle's own permuted copy of x, so there d_y may be the caller's x.
 * Device vectors only, asynchronous on `stream`.  As with the plain calls, the first call on a handle may synchronise
 * (plans, scratch); later calls only enqueue work and can be captured in a CUDA graph.  Launches per pass: those of the
 * plain call, except SMVP_TJDS_ATOMIC on a handle with y_relabel = -1, which takes one more (its sums land in a scratch
 * of `rows` doubles, allocated at the first such call and counted in device_bytes, and a per-row pass applies the
 * formula).  A TJDS handle without entries: the transposed call stores fl(alpha * 0) + fl(beta * y) with one launch.
 * Bytes added to a pass: 8 * rows (the read of y) when beta != 0; TJDS atomic in natural order 16 * rows more.       */
int smvp_csr_mult_device_axpby(smvp_csr *A, double alpha, const double *d_x, double beta, double *d_y, int variant,
                               void *stream); /* d_x == NULL: the x of smvp_csr_set_x_device */
int smvp_tjds_mult_device_axpby(smvp_tjds *A, double alpha, double beta, double *d_y, int variant, int32_t diag_limit,
                                void *stream); /* the x of smvp_tjds_set_x_device, as smvp_tjds_mult_device */
int smvp_tjds_mult_transpose_device_axpby(smvp_tjds *A, double alpha, const double *d_x, double beta, double *d_y,
                                          void *stream); /* d_x: rows entries, d_y: cols */

/* ---- the same update with an inner product of the new y fused into it: CG's p^T (A p), a residual's ||b - A x||^2,
 * BiCG's and LSQR's products with A^T -- without a second kernel that reads y (and w) again.
 *
 * y: bit for bit what the matching *_axpby call (same handle, variant, plan, diag_limit and arguments, (1, 0) included)
 *    stores, with its exception unchanged (TJDS atomic).
 * *d_dot = sum over every row r of y of fl(w[r] * y_new[r]) -- for the transposed call the `cols` entries of y.
 *    d_w == NULL means w = y_new (||y_new||^2); d_w may be the x the kernels read (CG's p^T A p).  d_dot is ONE device
 *    double, overwritten (never accumulated), written on `stream`.  When every term is zero (no rows; a handle without
 *    entries and beta = 0) it is +0.0.  Inf and NaN propagate as IEEE arithmetic says.
 * Order of the sum: each product is rounded once (no FMA).  The kernel that stores y adds the products of a WORK UNIT, a
 *    fixed set of rows of the handle's plan, into one partial:
 *        CSR row-pattern plan         a tile of 32 rows                       products added in a pairwise tree    d = 5
 *        CSR merge-path plan          a warp tile (its row ends, lane by lane, then a pairwise tree over the lanes) plus
 *                                     the fix-up's first row of the tile                                            d = 20
 *        CSR vector variant           the rows of one 256-thread CTA, pairwise tree over the threads               d = 8
 *        TJDS A x (every variant)     a block of 256 rows of y, pairwise tree                                       d = 8
 *        TJDS A^T x                   one CTA of the gather (its empty columns, then its short column) or of the
 *                                     combine kernel, pairwise tree over the threads      d = 9 + ceil((cols - nslots) /
 *                                     (256 * gather CTAs)), nslots the columns that hold entries; no entries: 256-entry
 *                                     blocks, d = 8
 *    The P partials are then summed in a tree that depends on P alone (at most 48 + ceil(P / 2^21) additions deep).
 *    With k = 1 + d + 48 + ceil(P / 2^21) and u = 2^-53:  |dot - sum_r w_r y_r| <= k u / (1 - k u) * sum_r |w_r y_r|.
 *    The bits are a function of the handle, its plan, the variant and the vectors -- never of the grid, the SM count,
 *    smvp_csr_set_corunner_headroom or timing: wherever y is reproducible the dot is bit-identical run to run (TJDS atomic
 *    and inputs routed to it, det_route = -1, are not).
 * Arguments: SMVP_E_ARG when d_dot is NULL, d_w == d_y (pass NULL for the new y), d_dot equals d_x, d_y or d_w, or a rule
 *    of the *_axpby call is broken.
 * Launches: those of the *_axpby call with (alpha, beta) != (1, 0) on the handle, plus one reduction -- a dot pass always
 *    runs the epilogue, so TJDS atomic on a handle with y_relabel = -1 uses the scratch y and the per-row pass even for
 *    (1, 0).  Bytes added to the *_axpby pass: 8 * rows for w when d_w != NULL, plus 16 bytes per work unit.  The
 *    per-handle scratch of the partials -- 8 * (U + ceil(U / 8192) + 1) bytes, U the most units the handle can use (CSR:
 *    any variant or plan; TJDS: A x, and A^T x once its plan exists) -- is allocated at the first dot call, which may
 *    synchronise, and counted in device_bytes; later calls only enqueue work.  The one exception: a TJDS handle whose
 *    first transposed dot call comes after an A x one grows it then, synchronising once.  Only one dot pass may be in
 *    flight per handle.                                                                                              */
int smvp_csr_mult_device_axpby_dot(smvp_csr *A, double alpha, const double *d_x, double beta, double *d_y,
                                   const double *d_w, double *d_dot, int variant, void *stream);
int smvp_tjds_mult_device_axpby_dot(smvp_tjds *A, double alpha, double beta, double *d_y, const double *d_w,
                                    double *d_dot, int variant, int32_t diag_limit, void *stream);
int smvp_tjds_mult_transpose_device_axpby_dot(smvp_tjds *A, double alpha, const double *d_x, double beta, double *d_y,
                                              const double *d_w, double *d_dot, void *stream);

/* ---- new values on the stored entries (Newton steps, implicit time steps, continuation, shifted systems A - sigma I: the
 * sparsity stays, the values change) without a new build.
 *
 * Input: a COO list of n entries in the form the builders take -- the host variant an smvp_coo array (copied to the
 *    device as smvp_csr_build does), the device variant structure-of-arrays device pointers.  Every (row, col) of the list
 *    must be an entry the handle stores; its value is replaced.  Entries not in the list keep their values.  Any order,
 *    any subset (only the diagonal, for A - sigma I, is fine).  n = 0 is a no-op.  A pair listed twice: one of its values
 *    lands, which one is unspecified (the handle stays consistent: its plans are decided from the values that landed).
 * Structure never changes: a value set to 0 stays stored as an explicit zero (TJDS's count_r still counts it).  To add or
 *    remove entries, build a new handle.  A handle made by smvp_csr_transpose is updated with the same list with rows and
 *    columns swapped.
 * Errors that leave the handle untouched, bit for bit (the whole list is checked before anything is written):
 *    SMVP_E_ARG a NULL handle, n < 0, or NULL arrays with n > 0; SMVP_E_RANGE a coordinate outside [0,rows) x [0,cols);
 *    SMVP_E_PATTERN a pair the handle does not store (any pair, on a handle without entries).
 * Errors after the write (SMVP_E_CUDA, SMVP_E_ALLOC): the handle holds the new values; its value-dependent plans are back
 *    to "not decided" and the next pass decides them as on a new handle.
 * Result: the handle behaves exactly like smvp_*_build run on the updated matrix once both have decided the same plans --
 *    the same smvp_*_export arrays, the same y bits from every pass (plain, *_axpby, *_axpby_dot and its dot, transposed,
 *    host -n loop, fan-out; SMVP_TJDS_ATOMIC as reproducible as between two runs), the same smvp_*_info except
 *    input_order (how the handle was built) and device_bytes (the scratch allocated so far).
 * Kept, not recomputed: row_ptr / col_ind, TJDS perm / start_pos / row_ind; the merge tiles, the row patterns, the
 *    relabelling, the TJDS walk and segment table, the pipelined host plan, the transposed and dot scratch, the co-runner
 *    headroom, and the x declared with smvp_*_set_x_device (it stays in effect).  val is rewritten in place: the pointers
 *    of smvp_csr_arrays_device stay valid.
 * Decided again for the new values: CSR with row_patterns > 0 -- value_bytes and its narrow copy (device_bytes follows
 *    the width); TJDS once a deterministic pass has run -- the row bounds and matrix flags, and det_route goes back to 0
 *    so that the next pass routes the current x again (Inf / NaN, the short split loop).  A plan still undecided stays so.
 * Synchronous, like the builders: ordered on `stream` after the work enqueued there, returns when the update is complete.
 *    No pass on the handle may be in flight on another stream (the rule of smvp_*_free).  A CUDA graph captured before an
 *    update must be captured again: kernel choices baked into it (value width, TJDS short split) may no longer hold.
 * Cost: no sort, no structural plan work; a fixed number of launches whatever n and nnz (CSR: 2, plus 2 with the row
 *    patterns; TJDS: 3, plus 2 with the deterministic state; the host variants 1 more to unzip the list).  One thread per
 *    entry binary-searches its row (CSR) or its column (TJDS), twice: once to check the whole list, once to write.
 *    Temporaries: O(rows + cols) (TJDS: the slot of every column, and the row counts of the bound pass), never O(nnz) or
 *    O(n); the host variants stage the list on the device as the builders do (32 bytes per entry).
 *    Measured (DESIGN.md §5.8): faster than a rebuild for a CSR list in row order and for short lists (the diagonal); a
 *    full list in random order, and a full TJDS list in any order, cost about a rebuild or more.                      */
int smvp_csr_update_values(smvp_csr *A, const smvp_coo *coo, int64_t n);
int smvp_csr_update_values_device(smvp_csr *A, const int32_t *d_row, const int32_t *d_col, const double *d_val, int64_t n,
                                  void *stream);
int smvp_tjds_update_values(smvp_tjds *A, const smvp_coo *coo, int64_t n);
int smvp_tjds_update_values_device(smvp_tjds *A, const int32_t *d_row, const int32_t *d_col, const double *d_val, int64_t n,
                                   void *stream);

/* ---- introspection ---- */
typedef struct smvp_csr_info_t
{
    int32_t rows, cols;
    int64_t nnz;
    int32_t max_row_nnz;
    int32_t auto_variant;     /* what SMVP_CSR_AUTO resolves to for this matrix               */
    int32_t input_order;      /* 0 unsorted, 1 arrived (row,col)-sorted, 2 arrived (col,row)-sorted */
    int64_t bytes_per_mult;   /* algorithmic bytes of one pass: 12 nnz + 4 (rows+1) + 8 cols + 8 rows */
    int64_t device_bytes;     /* HBM held by the handle                                        */
    int32_t launches_per_mult[3]; /* kernels one pass launches, indexed by variant (0 = AUTO)   */
    int32_t x_relabel;        /* multiply plan: 1 = the kernels read popularity-relabelled column indices
                                 and a permuted copy of x (row sums keep their order: y is bit-identical),
                                 -1 = natural order kept, 0 = not decided yet (decided at the first pass) */
    int32_t row_patterns;     /* multiply plan: P > 0 = every row's column offsets (col - row) are one of P lists of at most
                                 32 entries (stencils, banded matrices); the merge variant then streams a one-byte pattern id
                                 per row instead of col_ind and sums each row in the reference's order (y bit-identical to
                                 main-cli.c:410-416); -1 = not used (more than 256 lists, a longer row, a relabelled handle,
                                 or SMVP_CSR_PATTERN=0); 0 = not decided yet (decided at the first pass)              */
    int32_t value_bytes;      /* with row_patterns > 0: the width the pattern kernel streams the values at -- 2 (fp16) or
                                 4 (fp32) when EVERY value converts to that type and back with the same 64 bits (pattern
                                 and integer matrices, constant-coefficient stencils; a copy at that width is held and
                                 counted in device_bytes, y stays bit-identical), else 8; 0 = not decided yet.
                                 Meaningless when row_patterns <= 0.                                                  */
} smvp_csr_info_t;

typedef struct smvp_tjds_info_t
{
    int32_t rows, cols;
    int64_t nnz;
    int32_t ndiag;            /* number of jagged diagonals = largest column count             */
    int32_t ref_diag_limit;   /* diagonals the SHIPPED reference loop walks: count(col 0) + 1  */
    int32_t input_order;
    int64_t bytes_per_mult;   /* 12 nnz + 4 (ndiag+1) + 8 cols + 8 rows                         */
    int64_t device_bytes;
    int32_t launches_per_mult[3]; /* indexed by variant; includes the zero-fill of y            */
    int32_t y_relabel;        /* multiply plan: 1 = the kernels scatter through popularity-relabelled row
                                 indices and a last pass restores the row order of y, -1 = natural order,
                                 0 = not decided yet (decided at the first pass)                  */
    int32_t skewed_walk;      /* multiply plan: 1 = the kernels walk the (slot, diagonal) plane along anti-diagonals and
                                 merge runs of equal rows in registers before reducing into y (banded matrices),
                                 -1 = straight walk, 0 = not decided yet                              */
    int32_t det_route;        /* SMVP_TJDS_DETERMINISTIC with the current x: 1 = exact integer accumulation,
                                 -1 = served by the atomic kernel because x or the matrix holds Inf / NaN or the
                                 exponents may overflow (results then follow IEEE propagation, not run-to-run
                                 bit identity), 0 = not decided yet                                   */
} smvp_tjds_info_t;

int smvp_csr_info(const smvp_csr *A, smvp_csr_info_t *out);
int smvp_tjds_info(const smvp_tjds *A, smvp_tjds_info_t *out);

/* ---- parity accessors: copy the device-built arrays back for bit-exact checks (any pointer may be NULL).
 * row_ptr[rows+1], col_ind[nnz], val[nnz];  perm[cols], start_pos[ndiag+1], row_ind[nnz], val[nnz] */
int smvp_csr_export(const smvp_csr *A, int32_t *row_ptr, int32_t *col_ind, double *val);
int smvp_tjds_export(const smvp_tjds *A, int32_t *perm, int32_t *start_pos, int32_t *row_ind, double *val);
/* device views of the same arrays (owned by the handle; valid until free) */
int smvp_csr_arrays_device(const smvp_csr *A, const int32_t **d_row_ptr, const int32_t **d_col_ind,
                           const double **d_val);

void smvp_csr_free(smvp_csr *A);
void smvp_tjds_free(smvp_tjds *A);

/* page-locked host memory for the x / y vectors of the host entry points (NULL on failure).  smvp_csr_mult overlaps
 * its PCIe transfers with the multiply only when both vectors are page-locked; pageable buffers (malloc) are served by
 * plain copies -- same result, no overlap. */
void *smvp_host_alloc(int64_t bytes);
void smvp_host_free(void *p);

const char *smvp_strerror(int code);
/* text of the last CUDA error seen by this thread's last failing call ("" if none) */
const char *smvp_last_cuda_error(void);
/* number of CUDA devices visible, or SMVP_E_CUDA */
int smvp_device_count(void);
/* kernels launched by this library since load (every launch is counted) */
int64_t smvp_launch_count(void);

#pragma GCC visibility pop
#ifdef __cplusplus
}
#endif
#endif /* SMVP_CUDA_H */
