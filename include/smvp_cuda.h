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
#define SMVP_TJDS_DETERMINISTIC 1 /* order-independent exact INTEGER accumulation: every product is split exactly into two
                                     64-bit fixed-point words scaled per row by a bound known before the multiply
                                     (row_exp + exponent of max|x|), the words are added with integer atomics, one final
                                     rounding: y is the CORRECTLY ROUNDED row sum, bit-identical run to run (and between
                                     the straight and the skewed walk, with and without row relabelling).            */
#define SMVP_TJDS_DETERMINISTIC_FAST 2 /* the same with the high word only: a product is truncated toward zero at 2^-62 of
                                     its row's bound B_r = 2^ceil(log2(max|a_rj| * max|x| * count_r)).  Just as
                                     reproducible (integer sums), one reduction per run and half the accumulator traffic;
                                     the error is bounded NORMWISE, |err_r| <= count_r * 2^-62 * B_r -- 2^-9 of what one
                                     fp64 addition at magnitude B_r rounds away -- not relative to |y_r|: an x whose
                                     entries span many orders of magnitude can cost a row with small products digits
                                     that the exact variant keeps.                                                  */

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
    int32_t x_split;          /* multiply plan of a relabelled handle: 1 = the merge-path multiply runs in two passes, the
                                 entries whose column is among the 4 Mi most popular (their part of x stays in L2) and
                                 the others (y += ...): a row sum is then taken in two parts -- within 1e-12, not
                                 bit-identical to the one-pass order; -1 = one pass (the default: the split is an
                                 opt-in experiment, SMVP_CSR_SPLIT=1, that loses on R-MAT); 0 = not decided yet   */
    int32_t row_patterns;     /* multiply plan: P > 0 = every row's column offsets (col - row) are one of P lists of at most
                                 32 entries (stencils, banded matrices); the merge variant then streams a one-byte pattern id
                                 per row instead of col_ind and sums each row in the reference's order (y bit-identical to
                                 main-cli.c:410-416); -1 = not used (more than 256 lists, a longer row, a relabelled handle,
                                 or SMVP_CSR_PATTERN=0); 0 = not decided yet (decided at the first pass)              */
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
