// common.cuh -- shared declarations of libsmvp_cuda (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <cstdlib>
#include <functional>
#include <memory>
#include <new>
#include <type_traits>

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

// Owners of the library's CUDA resources: device memory, pinned host memory, events, streams and graphs are each held by
// one of these, so every return path releases them.  cudaFree synchronises the device implicitly, and wherever an owner
// may go out of scope while a stream still uses its memory, the code synchronises that stream first.
struct DevFree
{
    void operator()(void *p) const { cudaFree(p); }
};
struct PinnedFree
{
    void operator()(void *p) const { cudaFreeHost(p); }
};
struct CudaDestroy
{
    void operator()(cudaEvent_t e) const { cudaEventDestroy(e); }
    void operator()(cudaStream_t s) const { cudaStreamDestroy(s); }
    void operator()(cudaGraph_t g) const { cudaGraphDestroy(g); }
    void operator()(cudaGraphExec_t g) const { cudaGraphExecDestroy(g); }
};
template <typename T>
using DevPtr = std::unique_ptr<T, DevFree>;
template <typename T>
using PinnedPtr = std::unique_ptr<T, PinnedFree>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, CudaDestroy>;
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, CudaDestroy>;
using Graph = std::unique_ptr<std::remove_pointer_t<cudaGraph_t>, CudaDestroy>;
using GraphExec = std::unique_ptr<std::remove_pointer_t<cudaGraphExec_t>, CudaDestroy>;

// out(owner): the handle pointer a creating call writes to (cudaEventCreate(out(ev))); the owner takes the new handle
// at the end of the full expression, before SMVP_CUDA looks at the result
template <typename P>
struct OutPtr
{
    P &owner;
    typename P::pointer raw = nullptr;
    ~OutPtr() { owner.reset(raw); }
    operator typename P::pointer *() { return &raw; }
};
template <typename P>
static inline OutPtr<P> out(P &owner)
{
    return OutPtr<P>{owner};
}

// device allocation padded so that 16-byte vector / bulk copies may over-read the tail
template <typename T>
static inline cudaError_t dev_alloc(DevPtr<T> &p, int64_t n)
{
    size_t bytes = (size_t)(n > 0 ? n : 0) * sizeof(T);
    bytes = ((bytes + 255) & ~(size_t)255) + 256;
    return cudaMalloc((void **)(T **)out(p), bytes);
}

// Lifts a run-time flag into a template argument: f(std::true_type()) or f(std::false_type()), so that a launcher names
// each kernel instantiation once.
template <typename F>
static inline int with_flag(bool b, F &&f)
{
    return b ? f(std::true_type()) : f(std::false_type());
}

// The store of the scaled, accumulating multiply y = alpha * A x + beta * y (the *_axpby entry points): s is what the plain
// pass stores for the row, y0 the row's old value.  Products and the sum are rounded separately (no FMA).  beta == 0:
// fl(alpha * s) and y0 is not used -- callers then never load it.
struct Axpby
{
    double alpha, beta;
    bool plain() const { return alpha == 1.0 && beta == 0.0; } // fl(1 * s) = s: the plain kernels store exactly this
};
__device__ __forceinline__ double axpby(double alpha, double s, double beta, double y0)
{
    return beta != 0.0 ? __dadd_rn(__dmul_rn(alpha, s), __dmul_rn(beta, y0)) : __dmul_rn(alpha, s);
}

// The inner product fused into the store (the *_axpby_dot entry points, DESIGN.md §5.7).  The kernel that stores row r of
// y also forms dot_term = fl(w[r] * y_new[r]) (w == NULL: y_new[r] itself) and sums the terms of its WORK UNIT -- a fixed
// set of rows the plan defines -- into part[unit].  dot_reduce then sums the partials in a fixed tree that depends on
// their number only, so the bits never depend on the grid, the SM count or timing.
struct DotOut
{
    const double *w; // NULL: w = y_new
    double *part;    // one partial per work unit
};
__device__ __forceinline__ double dot_term(const double *w, int64_t r, double v) { return __dmul_rn(w ? __ldg(w + r) : v, v); }

// Multi GPU (row blocks, SURVEY.md 8e): every rank must end with the whole y, so the CSR multiply kernels store each
// finished row straight into every peer's copy of y over NVLink (peer-mapped symmetric memory): the "allgather" is fused
// into the SpMV epilogue and overlaps the streaming of the matrix instead of following it.
constexpr int SMVP_MAX_FANOUT = 8;
struct YFan
{
    double *p[SMVP_MAX_FANOUT];
    int n;
};

// How a kernel stores a finished row s of y.  Every kernel that stores y takes the mode as a template parameter, so each
// instantiation stores one way:
//   Plain   y[r] = s
//   Fanout  s into every copy of y in a YFan; y is only ever written, never read, so it may be a write-only mapping
//   Axpby   y[r] = fl(alpha * s) + fl(beta * y[r])   (the *_axpby entry points)
//   Dot     Axpby, and the row's dot term goes to the kernel's work-unit partial   (the *_axpby_dot entry points)
enum class YStore
{
    Plain,
    Fanout,
    Axpby,
    Dot
};
__host__ __device__ constexpr bool reads_y(YStore m) { return m == YStore::Axpby || m == YStore::Dot; } // only when beta != 0
// the mode of a pass: a dot pass runs the epilogue and never fans out; the fan-out only serves y = A x
static inline YStore store_mode(bool dot, bool fan, const Axpby &ab)
{
    return dot ? YStore::Dot : fan ? YStore::Fanout : ab.plain() ? YStore::Plain : YStore::Axpby;
}
// Lifts a run-time store mode into a template argument, like with_flag: f(std::integral_constant<YStore, m>()) for the
// modes Ms a kernel family is instantiated with (the launcher lists them), so that each launcher names every
// instantiation once.  Store modes are picked by store_mode, so m is always one of Ms.
template <YStore... Ms, typename F>
static inline int with_store(YStore m, F &&f)
{
    int rc = SMVP_E_ARG;
    (void)((m == Ms && ((rc = f(std::integral_constant<YStore, Ms>())), true)) || ...);
    return rc;
}
// The store of row r in mode M (fan: the copies of a Fanout store).  Returns the row's dot term in Dot mode, +0.0 otherwise.
// Every row has exactly one writer in a pass, so the read-modify-write of Axpby and Dot is safe; beta == 0 never loads y.
template <YStore M>
__device__ __forceinline__ double store_row(double *__restrict__ y, int64_t r, double s, double alpha, double beta,
                                            const double *__restrict__ w, const YFan *fan = nullptr)
{
    if constexpr (M == YStore::Plain)
        y[r] = s;
    else if constexpr (M == YStore::Fanout)
    {
        for (int k = 0; k < fan->n; k++)
            fan->p[k][r] = s;
    }
    else
    {
        const double v = axpby(alpha, s, beta, beta != 0.0 ? y[r] : 0.0);
        y[r] = v;
        if constexpr (M == YStore::Dot)
            return dot_term(w, r, v);
    }
    return 0.0;
}
// pairwise tree over the 32 lanes in lane order (a butterfly: every lane ends with the same bits)
__device__ __forceinline__ double warp_tree_sum(double v)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
        v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// pairwise tree over the THREADS threads of a CTA in thread order; the sum is valid in thread 0.  Every thread calls it.
template <int THREADS>
__device__ __forceinline__ double cta_tree_sum(double v)
{
    constexpr int W = THREADS / 32;
    static_assert(W >= 1 && W <= 32 && (W & (W - 1)) == 0, "a power of two of warps");
    __shared__ double s_w[W];
    v = warp_tree_sum(v);
    if (W == 1)
        return v;
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    if (lane == 0)
        s_w[wi] = v;
    __syncthreads();
    if (wi == 0)
    {
        v = lane < W ? s_w[lane] : 0.0;
#pragma unroll
        for (int o = 1; o < W; o <<= 1)
            v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    }
    return v;
}
// Per-handle scratch of a dot pass (dot.cu): the partials of `units` work units, the reduction's CTA sums and its counter.
// Grows *buf (counted in *device_bytes) when the plan needs more room; may synchronise then.
int dot_scratch(DevPtr<double> *buf, int64_t *cap, int64_t *device_bytes, int64_t units, cudaStream_t s);
// one launch: *out = the partials buf[0, units) summed in the fixed tree (DESIGN.md §5.7)
int dot_reduce(double *buf, int64_t cap, int64_t units, double *out, cudaStream_t s);

// ---------------------------------------------------------------- environment (api.cu)
// The library's only reader of the environment: every SMVP_* switch goes through these (table in INTEGRATION.md).
const char *env_str(const char *name);                   // the value; NULL when unset or empty
bool env_set(const char *name);                          // set at all, even to ""
int env_int(const char *name, int dflt, int lo, int hi); // decimal integer clamped to [lo, hi]; dflt when unset or empty
int env_tristate(const char *name);                      // 1 for "1...", -1 for "0...", 0 otherwise

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
// On return *d_idx (device, nnz uint32) lists source positions in sorted order, or is empty when the input already
// is in the requested order.
int coo_sort_index(const int32_t *d_major, const int32_t *d_minor, int64_t nnz, int32_t n_major, int32_t n_minor,
                   bool already_sorted, bool sorted_transposed, DevPtr<uint32_t> *d_idx, cudaStream_t s);
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
// Value widths of that plan: fp64 (double), fp32 (float) or fp16 held as its 16 bits (uint16_t).  pattern.cu keeps a
// narrow width only where narrow_value then widen_value gives back the same 64 bits for EVERY value, and the pattern
// kernel widens with the same instruction, so its products see exactly the fp64 operands.
__device__ __forceinline__ double widen_value(double v) { return v; }
__device__ __forceinline__ double widen_value(float v)
{
    double d;
    asm("cvt.f64.f32 %0, %1;" : "=d"(d) : "f"(v));
    return d;
}
__device__ __forceinline__ double widen_value(uint16_t v)
{
    double d;
    asm("cvt.f64.f16 %0, %1;" : "=d"(d) : "h"(v));
    return d;
}
template <typename V>
__device__ __forceinline__ V narrow_value(double v)
{
    static_assert(std::is_same<V, float>::value || std::is_same<V, uint16_t>::value, "fp32 or fp16");
    V n;
    if constexpr (std::is_same<V, float>::value)
        asm("cvt.rn.f32.f64 %0, %1;" : "=f"(n) : "d"(v));
    else
        asm("cvt.rn.f16.f64 %0, %1;" : "=h"(n) : "d"(v));
    return n;
}

// streams and events of the pipelined host-vector pass (csr_mult.cu), created on its first use.  One stream per direction:
// pieces on two or three streams per direction only share the link and finish later (10.15 ms per call with one, 11.9
// with two, 13.2 with three; profiles/r01_logs/e2e_sweep.log).
constexpr int PIPE_MAX_RANGES = 64;
constexpr int PIPE_MAX_XCHUNKS = 64;
struct PipeResources
{
    Stream up, down, compute;
    Event begin, x_ready[PIPE_MAX_XCHUNKS], done[PIPE_MAX_RANGES], down_done[PIPE_MAX_RANGES], t0[PIPE_MAX_RANGES],
        t1[PIPE_MAX_RANGES];
};

} // namespace smvp

// ---------------------------------------------------------------- handles
// Created value-initialised (new (std::nothrow) smvp_csr()), so every scalar starts at zero; the owners free everything
// the handle holds when it is deleted.
struct smvp_csr
{
    int32_t rows, cols;
    int64_t nnz;
    smvp::DevPtr<int32_t> row_ptr; // [rows+1]
    smvp::DevPtr<int32_t> col_ind; // [nnz]
    smvp::DevPtr<double> val;      // [nnz]
    int32_t max_row_nnz;
    int32_t input_order;
    int32_t auto_variant;
    int64_t device_bytes;
    // merge-path plan (csr_mult.cu), built lazily
    int32_t merge_headroom; // CTAs per SM the persistent merge-path grid leaves free for a co-running kernel (default 0)
    int32_t merge_cfg;      // which template instantiation the plan was made for (-1 none)
    int32_t merge_tiles;
    smvp::DevPtr<int32_t> tile_row; // [merge_tiles+1] rows consumed before each tile
    smvp::DevPtr<double> head_val;  // [merge_tiles] partial of the first row that ends in the tile
    smvp::DevPtr<double> carry_val; // [merge_tiles] partial of the row that continues past the tile
    // scratch for the host-vector entry point
    smvp::DevPtr<double> d_x, d_y;
    // plan of the pipelined host-vector pass (csr_mult.cu): tile ranges, the rows each completes and how much of x
    // (a leading part, x arrives front to back) each reads.  Host-side copies; pipe_cfg = tile size they were cut for.
    int32_t pipe_cfg, pipe_ranges, pipe_xlo; // pipe_xlo: first entry of x any nonzero reads (rounded down to 64)
    int32_t pipe_tile[smvp::PIPE_MAX_RANGES + 1], pipe_row[smvp::PIPE_MAX_RANGES + 1], pipe_xneed[smvp::PIPE_MAX_RANGES];
    std::unique_ptr<smvp::PipeResources> pipe_res;
    // popularity relabelling of the column space (relabel.cu): 0 undecided, 1 in use, -1 not worth it
    int32_t relabel_state;
    smvp::DevPtr<int32_t> col_rel; // [nnz]  rank of col_ind[j]; what the kernels read instead of col_ind when in use
    smvp::DevPtr<int32_t> x_order; // [cols] column with rank p
    smvp::DevPtr<double> x_rel;    // [cols] x in rank order
    const double *x_set;           // the x last given to smvp_csr_set_x_device (caller-owned)
    // row-pattern plan (pattern.cu): 0 undecided, 1 in use, -1 not used.  Row r's k-th nonzero sits in column
    // r + pat_off[pat_id[r] * PAT_LMAX + k]; the multiply reads pat_id instead of col_ind.
    int32_t pattern_state;
    int32_t pattern_count, pattern_maxlen; // distinct patterns, longest pattern
    smvp::DevPtr<uint8_t> pat_id;          // [rows]
    smvp::DevPtr<int32_t> pat_off;         // [pattern_count * PAT_LMAX]
    smvp::DevPtr<int32_t> pat_len;         // [pattern_count]
    // the values the pattern kernel streams: val itself (pat_vbytes 8) or, when every value converts to fp32 / fp16 and
    // back with the same 64 bits, a copy at that width (pat_vbytes 4 / 2).  0 = not decided.  val stays for every other path.
    int32_t pat_vbytes;
    smvp::DevPtr<char> pat_val; // [nnz * pat_vbytes] narrow copy (empty at width 8)
    // scratch of the fused inner product (*_axpby_dot, dot.cu): unit partials, reduction sums and counter; built at first use
    smvp::DevPtr<double> dot_buf;
    int64_t dot_cap;
};
namespace smvp
{
int csr_relabel_plan(smvp_csr *A, cudaStream_t s);                 // relabel.cu
int csr_relabel_x(smvp_csr *A, const double *d_x, cudaStream_t s); // relabel.cu
int csr_pattern_plan(smvp_csr *A, cudaStream_t s);                // pattern.cu: decides the relabelling first
int csr_pattern_values(smvp_csr *A, cudaStream_t s);              // pattern.cu: the value width of an accepted plan
} // namespace smvp

struct smvp_tjds
{
    int32_t rows, cols;
    int64_t nnz;
    int32_t ndiag;
    int32_t ref_diag_limit;
    int32_t input_order;
    int32_t nslots;                  // columns with at least one entry (= length of diagonal 0)
    int32_t last_diag_len;           // entries in the last jagged diagonal
    smvp::DevPtr<int32_t> perm;      // [cols]   slot -> original column
    smvp::DevPtr<int32_t> slot_len;  // [cols]   entries in the column at slot p (descending)
    smvp::DevPtr<int32_t> start_pos; // [ndiag+1]
    smvp::DevPtr<int32_t> row_ind;   // [nnz]
    smvp::DevPtr<double> val;        // [nnz]
    smvp::DevPtr<double> x_perm;     // [cols]
    smvp::DevPtr<int2> seg_blocks;   // [num_seg_blocks] {segment, first slot}: work plan of the multiply (tjds_mult.cu)
    int32_t num_seg_blocks;
    int64_t device_bytes;
    // deterministic variant: exact fixed-point accumulation (tjds_mult.cu)
    smvp::DevPtr<int32_t> row_exp; // [rows] ea_r + cb_r: |a_rj| < 2^ea_r, row holds <= 2^cb_r entries (aux, built lazily)
    smvp::DevPtr<long long> acc;   // [2*rows] hi/lo integer accumulators
    smvp::DevPtr<int32_t> x_exp;   // [1] exponent bound of max |x|
    smvp::DevPtr<double> d_x, d_y;
    // popularity relabelling of the ROW space (relabel.cu): 0 undecided, 1 in use, -1 not worth it
    int32_t skew;            // walk of the multiply kernels: 0 undecided, 1 skewed (runs of equal rows), -1 straight
    int32_t det_flags[5];    // host copy: [0] bit 0 = the matrix holds Inf/NaN, bit 1 = a row has entries but only zeros;
                             // [1] / [2] = largest / smallest row_exp (EXP_NONE / EXP_LOW_NONE if none);
                             // [3] / [4] = first / last row (of the index space the kernels use) that holds an entry
    smvp::PinnedPtr<int32_t> x_exp_host; // x_exp as of the last smvp_tjds_set_x_device, valid once x_exp_event has passed
    smvp::Event x_exp_event;
    int32_t x_exp_pending;   // 1: x_exp_host has not been looked at since the last set_x
    int32_t det_fast;        // for the current x: 1 every row bound is in the range of the short split loop, -1 not
    int32_t det_route;       // for the current x: 1 exact integer kernel, -1 atomic kernel (non-finite / overflowing input)
    int32_t relabel_state;
    smvp::DevPtr<int32_t> row_rel;  // [nnz]  rank of row_ind[j]; what the kernels scatter through when in use
    smvp::DevPtr<int32_t> row_rank; // [rows] rank of row r
    smvp::DevPtr<double> y_rel;     // [rows] y in rank order (atomic variant)
    smvp::DevPtr<double> y_sum;     // [rows] atomic sums of a natural-order handle under the epilogue (*_axpby), built at first use
    // transposed product y = A^T x (tjds_mult.cu), scratch built at its first call.  Columns longer than TJDS_SEG
    // (slots [0, tr_nlong)) are summed per segment into tr_part, then combined; tr_nwide of them are longer than
    // TJDS_SEG^2 entries and are combined by a whole warp.
    int32_t tr_ready;        // 1 once the scratch below exists
    int32_t tr_nlong, tr_nwide;
    smvp::DevPtr<uint32_t> tr_seg_off; // [nseg] first partial of segment g; slot q of segment g writes tr_part[tr_seg_off[g] + q]
    smvp::DevPtr<double> tr_part;      // one partial per (segment, slot) pair of the long columns
    smvp::DevPtr<double> d_xt, d_yt;   // [rows] / [cols]: scratch of the host-vector entry point
    smvp::DevPtr<double> dot_buf;      // scratch of the fused inner product (*_axpby_dot, dot.cu), built at first use
    int64_t dot_cap;
};
namespace smvp
{
int tjds_relabel_plan(smvp_tjds *A, cudaStream_t s); // relabel.cu
int tjds_update_det(smvp_tjds *A, cudaStream_t s);   // tjds_mult.cu: the row bounds again after a value update
} // namespace smvp
