// common.cuh -- shared declarations of libsmvp_cuda (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <cstdlib>
#include <functional>
#include <new>

#include "../../include/smvp_cuda.h"

namespace smvp
{

// ---------------------------------------------------------------- errors / bookkeeping
extern thread_local char g_last_cuda_error[256];
extern std::atomic<long long> g_launches;

int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define SMVP_CUDA(expr)                                                   \
    do                                                                    \
    {                                                                     \
        cudaError_t e__ = (expr);                                         \
        if (e__ != cudaSuccess)                                           \
            return ::smvp::cuda_fail(e__, #expr, __FILE__, __LINE__);     \
    } while (0)

#define SMVP_TRY(expr)        \
    do                        \
    {                         \
        int rc__ = (expr);    \
        if (rc__ != SMVP_OK)  \
            return rc__;      \
    } while (0)

// every kernel launch goes through this so that smvp_launch_count() is a true count
#define SMVP_LAUNCH(kernel, grid, block, smem, stream, ...)                       \
    do                                                                            \
    {                                                                             \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);               \
        ::smvp::g_launches.fetch_add(1, std::memory_order_relaxed);               \
    } while (0)

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// device allocation padded so that 16-byte vector / bulk copies may over-read the tail
template <typename T>
static inline cudaError_t dev_alloc(T **p, int64_t n)
{
    size_t bytes = (size_t)(n > 0 ? n : 0) * sizeof(T);
    bytes = ((bytes + 255) & ~(size_t)255) + 256;
    return cudaMalloc((void **)p, bytes);
}

// a device temporary that is released on every exit path (error returns included)
struct DevTmp
{
    void *p = nullptr;
    DevTmp() = default;
    DevTmp(const DevTmp &) = delete;
    DevTmp &operator=(const DevTmp &) = delete;
    ~DevTmp() { cudaFree(p); }
    template <typename T>
    cudaError_t alloc(int64_t n)
    {
        cudaFree(p);
        p = nullptr;
        T *q = nullptr;
        const cudaError_t e = dev_alloc(&q, n);
        p = q;
        return e;
    }
    template <typename T>
    T *as() const { return static_cast<T *>(p); }
};

// The `-n` loop of the host entry points (main-cli.c:402-420 / :1004-1024): `iters` passes, per-iteration
// milliseconds into ms_each (may be NULL).  `pass(stream)` enqueues ONE pass.
//   exact mode   CUDA events around every pass and a synchronisation per iteration (what round 1 did everywhere);
//   batched mode for matrices whose pass is shorter than the launch + synchronisation latency that exact mode adds
//                (~10 us): the first pass is timed exactly, the others are captured `batch` at a time in a CUDA graph
//                and replayed back to back; a pass is charged its batch's time / batch.  SMVP_EXACT_ITER_TIMES=1
//                forces exact mode, SMVP_LOOP_BATCH sets the batch (default 50).
constexpr int64_t SMVP_SMALL_LOOP_ITEMS = 1 << 22; // rows + cols + nnz below this: batched mode
//                `multi(stream, n)`, when given, enqueues n passes as ONE launch (tiny matrices: a single CTA loops
//                over the passes, csr_tiny_loop_kernel) and replaces the graph.
int timed_loop(int iters, double *ms_each, bool batched, const std::function<int(cudaStream_t)> &pass,
               const std::function<int(cudaStream_t, int)> &multi = nullptr);

struct DeviceProps
{
    int sms;
    int max_smem_optin;
};
const DeviceProps &device_props();

// ---------------------------------------------------------------- primitives (scan_sort.cu)
// exclusive prefix sum of n uint32 -> out[0..n) (out may alias in); *d_total (device, may be null) = sum
int exclusive_scan_u32(const uint32_t *d_in, uint32_t *d_out, int64_t n, uint32_t *d_total, cudaStream_t s);
// histogram: counts[key[i]]++  (counts pre-zeroed by the callee), keys in [0,nbins)
int histogram_i32(const int32_t *d_keys, int64_t n, uint32_t *d_counts, int64_t nbins, cudaStream_t s);
// stable LSD radix sort of (key, payload) pairs over the bit ranges given; returns pointers to result
// buffers through *out_keys/*out_vals (one of the two ping-pong buffers).
template <typename KeyT>
int radix_sort_pairs(KeyT *keys_a, uint32_t *vals_a, KeyT *keys_b, uint32_t *vals_b, int64_t n,
                     const int *bit_lo, const int *bit_hi, int nranges, KeyT **out_keys, uint32_t **out_vals,
                     cudaStream_t s);
int max_u32(const uint32_t *d_in, int64_t n, uint32_t *d_out, cudaStream_t s);

// ---------------------------------------------------------------- COO order detection (coo_common.cu)
enum InputOrder
{
    ORDER_NONE = 0,
    ORDER_ROW_COL = 1,
    ORDER_COL_ROW = 2
};
// validates coordinates (SMVP_E_RANGE) and reports the arrival order
int coo_inspect(const int32_t *d_row, const int32_t *d_col, int64_t nnz, int32_t rows, int32_t cols, int *order,
                cudaStream_t s);
// AoS (smvp_coo, 16 B) -> SoA
int coo_unzip(const smvp_coo *d_aos, int64_t nnz, int32_t *d_row, int32_t *d_col, double *d_val, cudaStream_t s);
// sorting permutation of the COO: major/minor lexicographic, using the arrival order to skip work.
// On return *d_idx (device, nnz uint32, owned by caller via cudaFree) lists source positions in sorted
// order, or is NULL when the input already is in the requested order.
int coo_sort_index(const int32_t *d_major, const int32_t *d_minor, int64_t nnz, int32_t n_major, int32_t n_minor,
                   bool already_sorted, bool sorted_transposed, uint32_t **d_idx, cudaStream_t s);
static inline int bits_for(uint32_t n) // bits needed to represent values in [0, n)
{
    int b = 0;
    while (b < 32 && (n == 0 ? 0u : (uint32_t)(n - 1)) >> b)
        b++;
    return b;
}

constexpr int32_t EXP_NONE = (int32_t)0x80808080; // memset(0x80) pattern: "no exponent seen", below any real one

// row-pattern plan (pattern.cu): at most PAT_MAX distinct column-offset lists (ids are one byte), none longer than PAT_LMAX
constexpr int PAT_MAX = 256;
constexpr int PAT_LMAX = 32;

} // namespace smvp

// ---------------------------------------------------------------- handles
struct smvp_csr
{
    int32_t rows, cols;
    int64_t nnz;
    int32_t *row_ptr; // [rows+1]
    int32_t *col_ind; // [nnz]
    double *val;      // [nnz]
    int32_t max_row_nnz;
    int32_t input_order;
    int32_t auto_variant;
    int64_t device_bytes;
    // merge-path plan (csr_mult.cu), built lazily
    int32_t merge_headroom; // CTAs per SM the persistent merge-path grid leaves free for a co-running kernel (default 0)
    int32_t merge_cfg;      // which template instantiation the plan was made for (-1 none)
    int32_t merge_tiles;
    int32_t *tile_row;      // [merge_tiles+1] rows consumed before each tile
    double *head_val;       // [merge_tiles] partial of the first row that ends in the tile
    double *carry_val;      // [merge_tiles] partial of the row that continues past the tile
    // scratch for the host-vector entry point
    double *d_x, *d_y;
    // plan of the pipelined host-vector pass (csr_mult.cu): tile ranges, the rows each completes and how much of x
    // (a leading part, x arrives front to back) each reads.  Host-side copies; pipe_cfg = tile size they were cut for.
    int32_t pipe_ramp;                       // 1: the ranges were cut with the ramped piece profile (SMVP_PIPE_PROFILE)
    int32_t pipe_cfg, pipe_ranges, pipe_xlo; // pipe_xlo: first entry of x any nonzero reads (rounded down to 64)
    int32_t pipe_tile[65], pipe_row[65], pipe_xneed[64];
    void *pipe_res; // streams and events of that pass, created on first use (csr_mult.cu)
    // popularity relabelling of the column space (relabel.cu): 0 undecided, 1 in use, -1 not worth it
    int32_t relabel_state;
    int32_t *col_rel;    // [nnz]  rank of col_ind[j]; what the kernels read instead of col_ind when in use
    int32_t *x_order;    // [cols] column with rank p
    double *x_rel;       // [cols] x in rank order
    const double *x_set; // the x last given to smvp_csr_set_x_device (caller-owned)
    // hot / cold split of a relabelled handle (relabel.cu): two CSR matrices over the SAME rank-ordered column space,
    // `hot` holding the entries whose column rank is below the L2-resident prefix of x_rel, `cold` the others.  The
    // merge-path multiply runs hot (every gather an L2 hit) then cold (+=).  0 undecided, 1 in use, -1 not used.
    int32_t split_state;
    int32_t ranked_cols; // 1: col_ind already holds popularity ranks (a hot / cold part): the ranked gather hints apply
    smvp_csr *hot, *cold;
    // row-pattern plan (pattern.cu): 0 undecided, 1 in use, -1 not used.  Row r's k-th nonzero sits in column
    // r + pat_off[pat_id[r] * PAT_LMAX + k]; the multiply reads pat_id instead of col_ind.
    int32_t pattern_state;
    int32_t pattern_count, pattern_maxlen; // distinct patterns, longest pattern
    uint8_t *pat_id;                       // [rows]
    int32_t *pat_off;                      // [pattern_count * PAT_LMAX]
    int32_t *pat_len;                      // [pattern_count]
};
namespace smvp
{
void csr_pipe_release(smvp_csr *A);                                // csr_mult.cu
int csr_relabel_plan(smvp_csr *A, cudaStream_t s);                 // relabel.cu
int csr_relabel_x(smvp_csr *A, const double *d_x, cudaStream_t s); // relabel.cu
void csr_relabel_release(smvp_csr *A);                             // relabel.cu
int csr_split_plan(smvp_csr *A, cudaStream_t s);                   // relabel.cu: after csr_relabel_plan
int csr_pattern_plan(smvp_csr *A, cudaStream_t s);                // pattern.cu: decides the relabelling first
void csr_pattern_release(smvp_csr *A);                             // pattern.cu
void csr_release(smvp_csr *A);                                     // csr_build.cu
int csr_build_impl(const int32_t *d_row, const int32_t *d_col, const double *d_val, int32_t rows, int32_t cols, int64_t nnz,
                   smvp_csr *A, cudaStream_t s);                   // csr_build.cu
// row_of[j] = row of nonzero j, from row_ptr[rows+1] (asynchronous on s)
int csr_expand_rows(const int32_t *row_ptr, int32_t rows, int64_t nnz, int32_t *row_of, cudaStream_t s); // csr_build.cu
} // namespace smvp

struct smvp_tjds
{
    int32_t rows, cols;
    int64_t nnz;
    int32_t ndiag;
    int32_t ref_diag_limit;
    int32_t input_order;
    int32_t nslots;      // columns with at least one entry (= length of diagonal 0)
    int32_t last_diag_len; // entries in the last jagged diagonal
    int32_t *perm;       // [cols]   slot -> original column
    int32_t *slot_len;   // [cols]   entries in the column at slot p (descending)
    int32_t *start_pos;  // [ndiag+1]
    int32_t *row_ind;    // [nnz]
    double *val;         // [nnz]
    double *x_perm;      // [cols]
    int2 *seg_blocks;    // [num_seg_blocks] {segment, first slot}: work plan of the multiply (tjds_mult.cu)
    int32_t num_seg_blocks;
    int64_t device_bytes;
    // deterministic variant: exact fixed-point accumulation (tjds_mult.cu)
    int32_t *row_exp;        // [rows] ea_r + cb_r: |a_rj| < 2^ea_r, row holds <= 2^cb_r entries (aux, built lazily)
    long long *acc;          // [2*rows] hi/lo integer accumulators
    int32_t *x_exp;          // [1] exponent bound of max |x|
    double *d_x, *d_y;
    // popularity relabelling of the ROW space (relabel.cu): 0 undecided, 1 in use, -1 not worth it
    int32_t skew;            // walk of the multiply kernels: 0 undecided, 1 skewed (runs of equal rows), -1 straight
    int32_t det_flags[5];    // host copy: [0] bit 0 = the matrix holds Inf/NaN, bit 1 = a row has entries but only zeros;
                             // [1] / [2] = largest / smallest row_exp (EXP_NONE / EXP_LOW_NONE if none);
                             // [3] / [4] = first / last row (of the index space the kernels use) that holds an entry
    int32_t *x_exp_host;     // pinned: x_exp as of the last smvp_tjds_set_x_device, valid once x_exp_event has passed
    cudaEvent_t x_exp_event;
    int32_t x_exp_pending;   // 1: x_exp_host has not been looked at since the last set_x
    int32_t det_fast;        // for the current x: 1 every row bound is in the range of the short split loop, -1 not
    int32_t det_route;       // for the current x: 1 exact integer kernel, -1 atomic kernel (non-finite / overflowing input)
    int32_t relabel_state;
    int32_t *row_rel;        // [nnz]  rank of row_ind[j]; what the kernels scatter through when in use
    int32_t *row_rank;       // [rows] rank of row r
    double *y_rel;           // [rows] y in rank order (atomic variant)
    // transposed product y = A^T x (tjds_mult.cu), scratch built at its first call.  Columns longer than TJDS_SEG
    // (slots [0, tr_nlong)) are summed per segment into tr_part, then combined; tr_nwide of them are longer than
    // TJDS_SEG^2 entries and are combined by a whole warp.
    int32_t tr_ready;        // 1 once the scratch below exists
    int32_t tr_nlong, tr_nwide;
    uint32_t *tr_seg_off;    // [nseg] first partial of segment g; slot q of segment g writes tr_part[tr_seg_off[g] + q]
    double *tr_part;         // one partial per (segment, slot) pair of the long columns
    double *d_xt, *d_yt;     // [rows] / [cols]: scratch of the host-vector entry point
};
namespace smvp
{
int tjds_relabel_plan(smvp_tjds *A, cudaStream_t s); // relabel.cu
void tjds_relabel_release(smvp_tjds *A);             // relabel.cu
} // namespace smvp
