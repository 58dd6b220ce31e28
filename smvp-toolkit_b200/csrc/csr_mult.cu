// csr_mult.cu -- y = A x in CSR on sm_100a.  Replaces the loop at main-cli.c:410-416
//
//     for row: for j in row_ptr[row] .. row_ptr[row+1]:  y[row] += val[j] * x[col_ind[j]]
//
// Two hand-written kernels, picked from the row-length distribution measured at build time:
//
//  VECTOR  one sub-warp (2..32 lanes) per row.  Each lane pulls 4 consecutive entries per step with
//          128-bit loads (one int4 of col_ind, two double2 of val) from a 16-byte-aligned position,
//          gathers x through the read-only path, and the sub-warp folds with __shfl_xor_sync.
//          Right for long regular rows and for matrices so small that launch latency is the cost.
//
//  MERGE   merge-path (Merrill & Garland): the list of row ends and the list of nonzeros are merged
//          conceptually and cut into equal tiles of 32*IPT items, so no row-length skew can
//          unbalance a warp or a lane.  Persistent, WARP-AUTONOMOUS: every warp owns a shared-memory
//          stage and an mbarrier, stages the val / col_ind / row_end slices of its tile with its own
//          TMA bulk copies (cp.async.bulk, evict-first in L2) and never meets a block-wide barrier.
//          Each lane owns IPT consecutive merge items: it first issues all its x gathers (independent,
//          IPT loads in flight per lane), then walks its items sequentially.  Lanes IPT items apart
//          sit on neighbouring rows at the same stencil position, which is what makes the x gather of
//          a banded matrix coalesce (2-3 sectors per request instead of ~22 for the vector kernel).
//          Rows cut by a lane boundary are stitched with a segmented warp scan, rows cut by a tile
//          boundary by a small fix-up kernel -- fixed order, no atomics: the kernel is deterministic.
//
// Arithmetic: products and sums are separate roundings (__dmul_rn/__dadd_rn), like the reference's
// mulsd+addsd; a row that lies inside one thread is summed in exactly the reference's order.
#include "common.cuh"

namespace smvp
{

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ int4 ld_stream_v4i(const int32_t *p)
{
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ double2 ld_stream_v2d(const double *p)
{
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile("{\n\t"
                 ".reg .pred p;\n\t"
                 "WAIT_%=:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE_%=;\n\t"
                 "bra WAIT_%=;\n\t"
                 "DONE_%=:\n\t"
                 "}" ::"r"(smem_u32(bar)),
                 "r"(parity)
                 : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_last_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// x gather of a popularity-relabelled matrix (relabel.cu): the column index IS the popularity rank, so the
// load can say how long the line deserves to live.  rank < hot_l1: keep in L1; rank < hot_l2: keep in L2
// (evict-last) while the matrix streams and the cold gathers pass through evict-first and do not allocate in L1.
// Every other L1 / L2 size measured on R-MAT scale 26 lost (DESIGN.md §5.4).
constexpr int32_t HOT_L1_ENTRIES = 8192;    // 64 KB of x
constexpr int32_t HOT_L2_ENTRIES = 4 << 20; // 32 MB of x
__device__ __forceinline__ double ldg_x_ranked(const double *x, int32_t c, int32_t hot_l1, int32_t hot_l2, uint64_t pol_last,
                                               uint64_t pol_first)
{
    double v;
    const uint64_t pol = c < hot_l2 ? pol_last : pol_first;
    // (one instruction per asm: a two-instruction block is not if-converted and every gather ends up in its own branch)
    if (c < hot_l1)
        asm volatile("ld.global.nc.L1::evict_last.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(x + c), "l"(pol));
    else
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(x + c), "l"(pol));
    return v;
}
// x[c] through the read-only path; the address is formed inside the asm (one IMAD.WIDE -- left to the compiler, the
// predicated index select turns it into a four-instruction sign-extend / shift sequence) and the load keeps its place
__device__ __forceinline__ double ldg_x_pinned(const double *x, int32_t c)
{
    double v;
    asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.s32 a, %2, 8, %1;\n\tld.global.nc.f64 %0, [a];\n\t}" : "=d"(v) : "l"(x), "r"(c));
    return v;
}
__device__ __forceinline__ uint64_t l2_evict_first_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}

// Variants A/B-tested on B200 and dropped from the source (profiles/r01_logs/ab_variants.log, stencil 369^3, ms per
// SpMV): all off 2.995 | explicit 32-bit ld.shared 2.984 | + warp-uniform fast path for regular tiles 3.13 |
//   + clamped (unpredicated) gathers 3.20 | + early-exit stitch scan 3.26 | all on 3.22
// i.e. every extra vote / branch costs more than the instructions it saves.  Only the explicit ld.shared is kept:
//   early-exit stitch scan (an __any_sync vote per step of the lane-boundary scan): removed.
//   x gathers with an L2 evict-last policy: measured 1 % on the stencil, 0 % on R-MAT: removed.

// explicit shared-window loads with 32-bit addresses (one register per view instead of a 64-bit generic pointer)
__device__ __forceinline__ double lds_f64(uint32_t a)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ int32_t lds_s32(uint32_t a)
{
    int32_t v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// ------------------------------------------------------------------ where y goes
// The kernels below store y in one of the modes of common.cuh (YStore, store_row).  Under Axpby and Dot the lane that ends
// a row, or the fix-up kernel for rows cut by tile boundaries, is the row's one writer.

// y[r] for the epilogue, loaded ahead of its store: through the coherent path (y is written by the same kernel) and
// issued where it stands (volatile: not sunk to its use)
__device__ __forceinline__ double ld_y_early(const double *p)
{
    double v;
    asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
// w[r] for the dot, loaded ahead of its use like ld_y_early (read-only: w is never y)
__device__ __forceinline__ double ld_w_early(const double *p)
{
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

// =====================================================================================  VECTOR
// LPR >= 16 (WIDE): each lane pulls 4 consecutive entries per step with 128-bit loads (long rows).
// LPR < 16: lane l takes entries l, l+LPR, ... with 8/4-byte loads (short rows).  With only a few rows per warp
//           the lanes of one request then sit on consecutive entries of consecutive rows, so the x gather of a
//           banded matrix touches far fewer sectors per request -- the vector kernel is L1-bound on such rows.
// Dot: the work unit is the CTA -- the rows its sub-warps end, in thread order.  It runs at 6 CTAs per SM: at the default
// bound ptxas keeps 32 registers and spills in the 128-bit configurations.
template <YStore M>
__host__ __device__ constexpr int vector_min_ctas() { return M == YStore::Dot ? 6 : 0; }
template <int LPR, YStore M>
__global__ void __launch_bounds__(256, vector_min_ctas<M>())
    csr_vector_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col_ind, const double *__restrict__ val,
                      const double *__restrict__ x, double *__restrict__ y, int32_t rows, const __grid_constant__ YFan fan, double alpha,
                      double beta, const double *__restrict__ w, double *__restrict__ part)
{
    constexpr bool WIDE = LPR >= 16;
    const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t row = gt / LPR;
    const int lane = (int)(gt % LPR);
    double sum = 0.0;
    if (row < rows && !WIDE)
    {
        const int32_t start = row_ptr[row], end = row_ptr[row + 1];
        int32_t j = start + lane;
        // two steps per trip: 4 independent loads and 2 gathers in flight per lane
        for (; j + LPR < end; j += 2 * LPR)
        {
            const int32_t c0 = __ldg(col_ind + j), c1 = __ldg(col_ind + j + LPR);
            const double v0 = __ldg(val + j), v1 = __ldg(val + j + LPR);
            const double x0 = __ldg(x + c0), x1 = __ldg(x + c1);
            sum = __dadd_rn(sum, __dmul_rn(v0, x0));
            sum = __dadd_rn(sum, __dmul_rn(v1, x1));
        }
        if (j < end)
            sum = __dadd_rn(sum, __dmul_rn(__ldg(val + j), __ldg(x + __ldg(col_ind + j))));
    }
    if (row < rows && WIDE)
    {
        const int32_t start = row_ptr[row], end = row_ptr[row + 1];
        for (int32_t j = (start & ~3) + 4 * lane; j < end; j += 4 * LPR)
        {
            const int4 c = ld_stream_v4i(col_ind + j);
            const double2 v0 = ld_stream_v2d(val + j);
            const double2 v1 = ld_stream_v2d(val + j + 2);
            double x0 = 0.0, x1 = 0.0, x2 = 0.0, x3 = 0.0;
            const bool p0 = j >= start, p1 = j + 1 >= start && j + 1 < end, p2 = j + 2 >= start && j + 2 < end,
                       p3 = j + 3 < end;
            if (p0)
                x0 = __ldg(x + c.x);
            if (p1)
                x1 = __ldg(x + c.y);
            if (p2)
                x2 = __ldg(x + c.z);
            if (p3 && j + 3 >= start)
                x3 = __ldg(x + c.w);
            if (p0)
                sum = __dadd_rn(sum, __dmul_rn(v0.x, x0));
            if (p1)
                sum = __dadd_rn(sum, __dmul_rn(v0.y, x1));
            if (p2)
                sum = __dadd_rn(sum, __dmul_rn(v1.x, x2));
            if (p3 && j + 3 >= start)
                sum = __dadd_rn(sum, __dmul_rn(v1.y, x3));
        }
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1)
        sum = __dadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, o));
    double d = 0.0;
    if (row < rows && lane == 0)
        d = store_row<M>(y, row, sum, alpha, beta, w, &fan);
    if constexpr (M == YStore::Dot)
    {
        d = cta_tree_sum<256>(d);
        if (threadIdx.x == 0)
            part[blockIdx.x] = d;
    }
}

// =====================================================================================  TINY LOOP
// Matrices of a few thousand nonzeros (the reference's sample-data: ibm32 126, curtis54 291, pdp08-pg4 16): one pass
// is far shorter than a kernel launch, so the `-n` loop itself moves onto the device.  ONE CTA repeats the whole
// multiply `passes` times -- warp per row, lanes stride the row, __shfl_xor_sync fold, exactly the vector kernel's
// arithmetic -- with a block barrier between passes.  The arrays are read with plain loads after each barrier (no
// read-only promise), so every pass really re-reads row_ptr / col_ind / val / x (from L1) and re-writes y: work is
// repeated, not hoisted.  Only reachable from the batched `-n` loop of smvp_csr_mult.
constexpr int TINY_THREADS = 512;
constexpr int64_t TINY_MAX_NNZ = 16384;
constexpr int32_t TINY_MAX_ROWS = 4096;
template <int LPR> // lanes per row: 4 / 8 / 16 / 32 from the mean row length, so that few rounds cover all rows
__global__ void __launch_bounds__(TINY_THREADS) csr_tiny_loop_kernel(const int32_t *row_ptr, const int32_t *col_ind, const double *val,
                                                                     const double *x, double *y, int32_t rows, int passes)
{
    const int lane = threadIdx.x % LPR, group = threadIdx.x / LPR;
    for (int p = 0; p < passes; p++)
    {
        for (int32_t row0 = 0; row0 < rows; row0 += TINY_THREADS / LPR) // every thread takes part in the shuffles
        {
            const int32_t row = row0 + group;
            double sum = 0.0;
            if (row < rows)
            {
                const int32_t start = row_ptr[row], end = row_ptr[row + 1];
                for (int32_t j = start + lane; j < end; j += LPR)
                    sum = __dadd_rn(sum, __dmul_rn(val[j], x[col_ind[j]]));
            }
#pragma unroll
            for (int o = LPR / 2; o > 0; o >>= 1)
                sum = __dadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, o));
            if (row < rows && lane == 0)
                y[row] = sum;
        }
        __syncthreads(); // pass boundary: also a compiler barrier, the next pass reloads everything
    }
}

// the column indices the multiply kernels read: the relabelled copy when that plan is in use (relabel.cu)
static inline const int32_t *mult_cols(const smvp_csr *A) { return A->relabel_state == 1 ? A->col_rel.get() : A->col_ind.get(); }

// lanes per row of the vector kernel, from the mean row length
static int vector_lpr(const smvp_csr *A)
{
    const double mean = A->rows > 0 ? (double)A->nnz / A->rows : 0.0;
    return mean <= 8.0 ? 2 : mean <= 16.0 ? 4 : mean <= 32.0 ? 8 : mean <= 64.0 ? 16 : 32;
}

template <int LPR>
static int launch_vector(const smvp_csr *A, const double *d_x, double *d_y, const YFan *fan, const Axpby &ab, const DotOut *dot,
                         cudaStream_t s)
{
    const int64_t threads = (int64_t)A->rows * LPR;
    const int64_t blocks = ceil_div64(threads, 256);
    if (blocks > 0x7fffffffLL)
        return SMVP_E_TOOBIG;
    if (blocks == 0)
        return SMVP_OK;
    return with_store<YStore::Plain, YStore::Fanout, YStore::Axpby, YStore::Dot>(store_mode(dot, fan, ab), [&](auto S) {
        SMVP_LAUNCH((csr_vector_kernel<LPR, decltype(S)::value>), (unsigned)blocks, 256, 0, s, A->row_ptr.get(), mult_cols(A),
                    A->val.get(), d_x, d_y, A->rows, fan ? *fan : YFan(), ab.alpha, ab.beta, dot ? dot->w : nullptr,
                    dot ? dot->part : nullptr);
        return (int)SMVP_OK;
    });
}

static int csr_mult_vector(const smvp_csr *A, const double *d_x, double *d_y, const YFan *fan, const Axpby &ab, const DotOut *dot,
                           cudaStream_t s)
{
    switch (vector_lpr(A))
    {
    case 2:
        return launch_vector<2>(A, d_x, d_y, fan, ab, dot, s);
    case 4:
        return launch_vector<4>(A, d_x, d_y, fan, ab, dot, s);
    case 8:
        return launch_vector<8>(A, d_x, d_y, fan, ab, dot, s);
    case 16:
        return launch_vector<16>(A, d_x, d_y, fan, ab, dot, s);
    default:
        return launch_vector<32>(A, d_x, d_y, fan, ab, dot, s);
    }
}

// =====================================================================================  MERGE
// merge-path coordinate on diagonal d: number of row-end items among the first d merge items.
// row_end[r] = row_ptr[r+1]; row r's end item sits after all of its nonzeros.
__device__ __forceinline__ int32_t merge_rows_before(const int32_t *__restrict__ row_ptr, int32_t rows, int64_t nnz, int64_t d)
{
    int64_t lo = d > nnz ? d - nnz : 0, hi = d < rows ? d : rows;
    while (lo < hi)
    {
        const int64_t mid = (lo + hi) >> 1;
        if ((int64_t)row_ptr[mid + 1] <= d - mid - 1)
            lo = mid + 1;
        else
            hi = mid;
    }
    return (int32_t)lo;
}

__global__ void __launch_bounds__(256) merge_plan_kernel(const int32_t *__restrict__ row_ptr, int32_t rows, int64_t nnz,
                                                         int32_t tile_items, int32_t num_tiles, int32_t *__restrict__ tile_row)
{
    const int32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > num_tiles)
        return;
    const int64_t total = (int64_t)rows + nnz;
    int64_t d = (int64_t)t * tile_items;
    if (d > total)
        d = total;
    tile_row[t] = merge_rows_before(row_ptr, rows, nnz, d);
}

template <int THREADS, int IPT>
struct MergeShape
{
    static constexpr int TILE = THREADS * IPT;
    static constexpr int SMEM_BYTES = ((12 * TILE + 128) + 127) & ~127; // one stage per warp
};

struct TileView
{
    int32_t r0, rows_t;     // first row of the tile, complete-row slots in the tile
    int64_t n0;             // first nonzero of the tile
    int32_t nnz_t, items_t; // nonzeros / merge items in the tile
    int32_t va, ca, ra;     // aligned first element staged of val / col_ind / row_ptr
    uint32_t vb, cb, rb;    // bytes staged of each
};

// (r0, r1) = rows consumed before the tile / before the next tile (tile_row[t], tile_row[t+1])
__device__ __forceinline__ TileView make_tile(int32_t r0, int32_t r1, int32_t t, int32_t tile_items, int64_t total)
{
    TileView v;
    const int64_t d0 = (int64_t)t * tile_items;
    int64_t d1 = d0 + tile_items;
    if (d1 > total)
        d1 = total;
    v.r0 = r0;
    v.rows_t = r1 - v.r0;
    v.n0 = d0 - v.r0;
    const int64_t n1 = d1 - r1;
    v.nnz_t = (int32_t)(n1 - v.n0);
    v.items_t = (int32_t)(d1 - d0);
    const int32_t n0 = (int32_t)v.n0, n1i = (int32_t)n1;
    v.va = n0 & ~1;
    v.vb = v.nnz_t > 0 ? (uint32_t)(((n1i + 1) & ~1) - v.va) * 8u : 0u;
    v.ca = n0 & ~3;
    v.cb = v.nnz_t > 0 ? (uint32_t)(((n1i + 3) & ~3) - v.ca) * 4u : 0u;
    v.ra = (v.r0 + 1) & ~3;
    v.rb = v.rows_t > 0 ? (uint32_t)(((r1 + 1 + 3) & ~3) - v.ra) * 4u : 0u;
    return v;
}

// First row of a tile that ends a row there: y[row] = (carries of the tiles the row crossed, in tile order) + (partial
// of the tile where it ends).  tile_row[u+1] is the row tile u's carry belongs to.
// Dot: the row's dot term is added to tile t's partial, which the merge kernel left (its unit: the tile plus this row).
template <YStore M>
__device__ __forceinline__ void merge_fixup_tile(int32_t t, const int32_t *__restrict__ tile_row, const double *__restrict__ head_val,
                                                 const double *__restrict__ carry_val, double *__restrict__ y, const YFan &fan,
                                                 double alpha, double beta, const double *__restrict__ w, double *__restrict__ part)
{
    // everything the common case needs is loaded up front (independent loads: one memory round trip)
    const int32_t r = tile_row[t];
    const int32_t r_next = tile_row[t + 1];
    const int32_t r_prev = t > 0 ? tile_row[t - 1] : -1;
    const double c_prev = t > 0 ? __ldcg(carry_val + t - 1) : 0.0; // L2 loads: another SM wrote these in this launch
    const double h = __ldcg(head_val + t);
    if (r_next == r)
        return; // no row ends in this tile
    double acc;
    if (t == 0)
        acc = h;
    else if (r_prev != r)
        acc = __dadd_rn(c_prev, h); // the row was cut once: tile t-1 carries into it
    else
    {
        int32_t u = t - 1; // the row spans several tiles: carries of tiles [u, t-1], in tile order
        while (u > 0 && tile_row[u] == r)
            u--;
        if (tile_row[u + 1] != r)
            u++;
        acc = __ldcg(carry_val + u);
        for (int32_t k = u + 1; k < t; k++)
            acc = __dadd_rn(acc, __ldcg(carry_val + k));
        acc = __dadd_rn(acc, h);
    }
    const double d = store_row<M>(y, r, acc, alpha, beta, w, &fan);
    if constexpr (M == YStore::Dot)
        part[t] = __dadd_rn(__ldcg(part + t), d);
}

// ---------------------------------------------------------------------------------------------
// Warp-autonomous merge-path: the unit of work is a WARP tile of 32*IPT merge items.  Every warp owns
// its shared-memory stage and its mbarrier, fetches its tiles with its own TMA bulk copies and
// never meets a block-wide barrier: warps of a CTA drift apart freely, so while one waits for HBM
// or for its x gathers the others walk.  Rows cut by lane boundaries are stitched with a segmented
// warp scan (__shfl_up_sync), rows cut by tile boundaries by the fix-up kernel -- fixed order, no atomics.
// Dot (DESIGN.md §5.7): whole passes only.  The work unit is the warp tile -- each lane adds the dot terms of the rows it
// stores in the order it stores them, the lanes are added in a pairwise tree into part[t], and the fix-up kernel adds the
// term of the tile's first row (merge_fixup_tile).
template <int WARPS, int IPT, int MINB, bool RANKED, bool UNI, YStore M>
__global__ void __launch_bounds__(WARPS * 32, MINB)
    csr_merge_warp_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col_ind, const double *__restrict__ val,
                          const double *__restrict__ x, double *__restrict__ y, const int32_t *__restrict__ tile_row, int32_t rows,
                          int64_t nnz, int32_t tile_begin, int32_t num_tiles, double *__restrict__ head_val,
                          double *__restrict__ carry_val, const __grid_constant__ YFan fan, int32_t hot_l1, int32_t hot_l2,
                          int32_t early_dependents, double alpha, double beta, const double *__restrict__ dot_w,
                          double *__restrict__ part)
{
    // Small grids (early_dependents != 0): let the fix-up kernel, launched with programmatic stream serialization, be
    // scheduled NOW; it parks at griddepcontrol.wait until this grid has completed and flushed.  In the batched `-n` loop
    // of a matrix like memplus that hides the second launch's latency (a pass lasts as long as a launch).
    if (early_dependents)
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // processes tiles [tile_begin, num_tiles): a sub-range lets the host overlap the copy-out of finished rows.
    // One stage per warp: deeper rings lost to more resident warps in every sweep.
    using Shape = MergeShape<32, IPT>;
    extern __shared__ __align__(128) unsigned char stage_mem[];
    __shared__ __align__(8) uint64_t full_bar[WARPS];

    // UNI: the warp index and the tile coordinates below are broadcast from lane 0.  The values are the same in every lane
    // anyway, but the broadcast lets the compiler PROVE it and keep the whole tile bookkeeping (and the operands of the
    // bulk copies) in uniform registers instead of electing a lane and converting per copy.  Measured on B200
    // (profiles/r01_logs/diet_bisect.log): stencil configuration 2.78 -> 2.69 ms, but the R-MAT configuration 5.67 ->
    // 6.39 ms, so it is a per-configuration choice (MergeStencil::UNI, MergeSkewed::UNI).
#define SMVP_BCAST(v) (UNI ? __shfl_sync(0xffffffffu, (v), 0) : (v))
    const int lane = threadIdx.x & 31, w = SMVP_BCAST((int)(threadIdx.x >> 5));
    const int64_t total = (int64_t)rows + nnz;
    unsigned char *base = stage_mem + (size_t)w * Shape::SMEM_BYTES;
    uint64_t *my_bar = &full_bar[w];
    uint64_t policy = 0;
    if (lane == 0)
    {
        mbar_init(my_bar, 1);
        fence_mbar_init();
        policy = l2_evict_first_policy();
    }
    __syncwarp();

    const uint64_t pol_last = RANKED ? l2_evict_last_policy() : 0, pol_first = RANKED ? l2_evict_first_policy() : 0;
    const int32_t warp_stride = (int32_t)gridDim.x * WARPS;
    auto issue = [&](const TileView &v) { // lane 0 only
        mbar_expect_tx(my_bar, v.vb + v.cb + v.rb);
        if (v.vb)
            bulk_g2s(base, val + v.va, v.vb, my_bar, policy);
        if (v.cb)
            bulk_g2s(base + v.vb, col_ind + v.ca, v.cb, my_bar, policy);
        if (v.rb)
            bulk_g2s(base + v.vb + v.cb, row_ptr + v.ra, v.rb, my_bar, policy);
    };

    int32_t t = (M == YStore::Dot ? 0 : tile_begin) + (int32_t)blockIdx.x * WARPS + w; // a dot pass is a whole pass
    int32_t cur_r0 = 0, cur_r1 = 0; // merge coordinates of the tile in flight: the only tile state kept across the loop
    if (t < num_tiles)
    {
        cur_r0 = SMVP_BCAST(__ldg(tile_row + t));
        cur_r1 = SMVP_BCAST(__ldg(tile_row + t + 1));
        if (lane == 0)
            issue(make_tile(cur_r0, cur_r1, t, Shape::TILE, total));
    }
    uint32_t parity = 0;

    while (t < num_tiles)
    {
        // per-tile scalars: only what the walk needs stays live (the rest of the TileView dies here)
        int32_t n0, tile_r0, rows_t, nnz_t, items_t;
        uint32_t sval, scol, srow; // shared-window byte addresses of TILE-LOCAL nonzero 0 / row 0
        {
            const TileView v = make_tile(cur_r0, cur_r1, t, Shape::TILE, total);
            n0 = (int32_t)v.n0;
            tile_r0 = v.r0;
            rows_t = v.rows_t;
            nnz_t = v.nnz_t;
            items_t = v.items_t;
            const uint32_t b = smem_u32(base);
            sval = b + 8u * (uint32_t)(n0 - v.va);
            scol = b + v.vb + 4u * (uint32_t)(n0 - v.ca);
            srow = b + v.vb + v.cb + 4u * (uint32_t)(v.r0 + 1 - v.ra);
        }
        auto row_end = [&](int32_t i) -> int32_t { return lds_s32(srow + 4u * (uint32_t)i) - n0; };

        mbar_wait(my_bar, parity);
        parity ^= 1u;

        // ---- my first merge item: interpolate, gallop, bisect (2 probes on regular matrices)
        int32_t d = lane * IPT;
        if (d > items_t)
            d = items_t;
        int32_t lo = d > nnz_t ? d - nnz_t : 0, hi = d < rows_t ? d : rows_t;
        if (lo < hi)
        {
            // first guess by interpolation.  The divisor is the FULL tile size (a compile-time constant: multiply-shift
            // instead of a 25-instruction integer division); only the matrix's last tile is shorter, and there the guess
            // is merely a little low before the gallop corrects it.
            int32_t g = (int32_t)(((uint32_t)d * (uint32_t)rows_t) / (uint32_t)Shape::TILE); // < 2^20: 32-bit is exact
            g = g < lo ? lo : (g > hi - 1 ? hi - 1 : g);
            int32_t step = 1;
            if (row_end(g) <= d - g - 1)
            {
                lo = g + 1;
                while (lo < hi)
                {
                    const int32_t m = (lo + step - 1 < hi - 1) ? lo + step - 1 : hi - 1;
                    if (row_end(m) <= d - m - 1)
                    {
                        lo = m + 1;
                        step <<= 1;
                    }
                    else
                    {
                        hi = m;
                        break;
                    }
                }
            }
            else
            {
                hi = g;
                while (lo < hi)
                {
                    const int32_t m = (hi - step > lo) ? hi - step : lo;
                    if (!(row_end(m) <= d - m - 1))
                    {
                        hi = m;
                        step <<= 1;
                    }
                    else
                    {
                        lo = m + 1;
                        break;
                    }
                }
            }
            while (lo < hi)
            {
                const int32_t mid = (lo + hi) >> 1;
                if (row_end(mid) <= d - mid - 1)
                    lo = mid + 1;
                else
                    hi = mid;
            }
        }
        const int32_t i0 = lo, j0 = d - lo;
        int32_t d_next = (lane + 1) * IPT;
        if (d_next > items_t)
            d_next = items_t;
        int32_t j_next = __shfl_down_sync(0xffffffffu, j0, 1);
        if (lane == 31)
            j_next = nnz_t;
        const int32_t i_next = d_next - j_next;
        const int32_t cnt = j_next - j0;

        // ---- all my gathers first, in three phases pinned by volatile asm: the column indices, then every x gather of
        // the lane (IPT independent loads in flight together -- left alone, the compiler reuses one register pair and
        // waits for each load before issuing the next), then the products.  (Pinning the lane's two shared-window bases
        // in registers with an opaque move saves an address instruction per load but makes the 14-item configurations
        // spill; the nested "live slot / row end" walk this one replaced is in profiles/r01_logs/diet_bisect.log.)
        // Axpby / Dot: y of my first row end (tile row i0; row 0 of the tile is the fix-up kernel's), loaded before the gathers so
        // that its latency hides behind them; further row ends of the lane (short rows) load y at their store
        double y_first = 0.0;
        if (reads_y(M) && beta != 0.0 && i0 < i_next && i0 != 0)
            y_first = ld_y_early(y + (int64_t)tile_r0 + i0);
        double w_first = 0.0; // Dot: w of that row, loaded beside it
        if (M == YStore::Dot && dot_w && i0 < i_next && i0 != 0)
            w_first = __ldg(dot_w + (int64_t)tile_r0 + i0);
        double prod[IPT];
        {
            int32_t cq[IPT];
            uint32_t cbase = scol + 4u * (uint32_t)j0, vbase = sval + 8u * (uint32_t)j0;
            // (every slot gets a defined value: leaving the dead ones undefined makes the compiler carry the previous
            // tile's registers through the loop and spill them)
#pragma unroll
            for (int q = 0; q < IPT; q++)
                cq[q] = q < cnt ? lds_s32(cbase + 4u * q) : 0;
#pragma unroll
            for (int q = 0; q < IPT; q++)
            {
                prod[q] = 0.0;
                if (q < cnt)
                    prod[q] = RANKED ? ldg_x_ranked(x, cq[q], hot_l1, hot_l2, pol_last, pol_first) : ldg_x_pinned(x, cq[q]);
            }
#pragma unroll
            for (int q = 0; q < IPT; q++)
                if (q < cnt)
                    prod[q] = __dmul_rn(lds_f64(vbase + 8u * q), prod[q]);
        }

        double sum = 0.0, first_sum = 0.0;
        double dl = 0.0; // Dot: this lane's dot terms, in the order it stores its rows
        // a row end of mine that is not my first (Dot: the add exists only there -- a dead add of +0.0 moves the schedule of
        // the Fanout store loop)
        auto store_end = [&](int32_t row, double s) {
            const double d = store_row<M>(y, (int64_t)tile_r0 + row, s, alpha, beta, dot_w, &fan);
            if constexpr (M == YStore::Dot)
                dl = __dadd_rn(dl, d);
        };
        bool has_first = false;
        {
            // Walk.  `until` = nonzeros of mine before my next row end (relative to j0, so each test is against a constant;
            // "no further row end of mine" = never).  Dead slots (q >= cnt) hold +0.0, and a partial sum that starts at
            // +0.0 can never become -0.0, so adding them is exact: the loop needs no "is this slot live" test, and the row
            // ends that follow my last nonzero are flushed by the same test at the first dead slot.
            int32_t row = i0;
            int32_t until = (row < i_next ? row_end(row) : 0x7fffffff) - j0;
#pragma unroll
            for (int q = 0; q < IPT; q++)
            {
                if (until <= q) // rare: a row end (or a run of empty rows) sits before item q
                {
                    do
                    {
                        if (!has_first)
                        {
                            has_first = true;
                            first_sum = sum;
                        }
                        else
                            store_end(row, sum);
                        sum = 0.0;
                        row++;
                        until = (row < i_next ? row_end(row) : 0x7fffffff) - j0;
                    } while (until <= q);
                }
                sum = __dadd_rn(sum, prod[q]);
            }
            // every row end of mine has at most IPT - 1 of my nonzeros before it, so the loop above has seen them all;
            // this is only a safety net
            while (row < i_next)
            {
                if (!has_first)
                {
                    has_first = true;
                    first_sum = sum;
                }
                else
                    store_end(row, sum);
                sum = 0.0;
                row++;
            }
        }

        // ---- the stage is consumed: refill it for my next tile while the warp stitches
        __syncwarp();
        const int32_t tn = t + warp_stride;
        if (tn < num_tiles && tn > t)
        {
            cur_r0 = SMVP_BCAST(__ldg(tile_row + tn));
            cur_r1 = SMVP_BCAST(__ldg(tile_row + tn + 1));
            if (lane == 0)
                issue(make_tile(cur_r0, cur_r1, tn, Shape::TILE, total));
        }

        // ---- stitch rows cut by lane boundaries: segmented inclusive scan of (carry row, carry sum)
        const int32_t key = i_next; // the row my trailing partial belongs to
        double scan = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const int32_t pk = __shfl_up_sync(0xffffffffu, key, o);
            const bool take = lane >= o && pk == key;
            const double pv = __shfl_up_sync(0xffffffffu, scan, o);
            if (take)
                scan = __dadd_rn(pv, scan);
        }
        const double prev_scan = __shfl_up_sync(0xffffffffu, scan, 1);
        const int32_t prev_key = __shfl_up_sync(0xffffffffu, key, 1);
        if (has_first)
        {
            if (lane > 0 && prev_key == i0)
                first_sum = __dadd_rn(prev_scan, first_sum);
            // the tile's first row may have started in earlier tiles: its partial goes to the fix-up
            // kernel, which adds the carries and writes y -- and, under the epilogue, is the only one to read that
            // row of y.  Without the epilogue y is only ever WRITTEN here (never read), so it may be a write-only
            // mapping such as an NVSwitch multicast address.
            if (i0 == 0)
                head_val[t] = first_sum;
            else if constexpr (reads_y(M))
            {
                const double v = axpby(alpha, first_sum, beta, y_first);
                y[(int64_t)tile_r0 + i0] = v;
                if constexpr (M == YStore::Dot)
                    dl = __dadd_rn(dl, __dmul_rn(dot_w ? w_first : v, v));
            }
            else
                store_row<M>(y, (int64_t)tile_r0 + i0, first_sum, alpha, beta, dot_w, &fan);
        }
        if (lane == 31)
            carry_val[t] = scan; // partial of the row that continues into the next tile
        if constexpr (M == YStore::Dot)
        {
            dl = warp_tree_sum(dl); // the lanes in a pairwise tree: the tile's partial (the fix-up adds its first row)
            if (lane == 0)
                part[t] = dl;
        }
        if (tn <= t)
            break; // 32-bit overflow guard
        t = tn;
    }
#undef SMVP_BCAST
}

// The fix-up.  Under Dot: griddepcontrol.wait returns only once the merge kernel has completed and its writes are
// visible, and every thread of this grid executes it before it exits: so when this grid has completed -- which the
// reduction launched after it in stream order waits for -- the merge kernel's partials are final, also when this grid
// was launched early.  The reduction itself is an ordinary launch.
template <YStore M>
__global__ void __launch_bounds__(256) merge_fixup_kernel(const int32_t *__restrict__ tile_row, const double *__restrict__ head_val,
                                                          const double *__restrict__ carry_val, int32_t tile_begin,
                                                          int32_t num_tiles, double *__restrict__ y,
                                                          const __grid_constant__ YFan fan, double alpha, double beta,
                                                          const double *__restrict__ w, double *__restrict__ part)
{
    // no-op unless launched with programmatic stream serialization: then it waits here for the merge kernel's results
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int32_t t = (M == YStore::Dot ? 0 : tile_begin) + blockIdx.x * blockDim.x + threadIdx.x;
    if (t < num_tiles)
        merge_fixup_tile<M>(t, tile_row, head_val, carry_val, y, fan, alpha, beta, w, part);
}

// ---- the two instantiations AUTO chooses from (merge_skewed).  Measured on B200 (logs under profiles/, the swept
// configurations in DESIGN.md §5.2): shared memory holds 12 B per staged nonzero, so the items per thread bound how many
// warps an SM can keep busy; single-stage warps at <= 64 registers (32 warps/SM) beat deeper rings, and any register
// spill halves the throughput.
struct MergeStencil // 14 items per thread (two lanes per 27-point-stencil row), 4 warps per CTA
{
    static constexpr int WARPS = 4, IPT = 14, MINB = 8;
    static constexpr bool UNI = true;
};
struct MergeSkewed // 10 items per thread, 28 warps/SM (R-MAT scale 26: 8.0 ms vs 8.8 ms at 32 warps/SM and 62 registers)
{
    static constexpr int WARPS = 2, IPT = 10, MINB = 14;
    static constexpr bool UNI = false;
};

// skewed or short rows take MergeSkewed, the others MergeStencil
static bool merge_skewed(const smvp_csr *A)
{
    const double mean = A->rows > 0 ? (double)A->nnz / A->rows : 0.0;
    return A->max_row_nnz > 64.0 * (mean + 1.0) || mean < 20.0;
}

constexpr int32_t MERGE_PDL_TILES = 8192; // grids of at most this many warp tiles launch their fix-up early

static int merge_plan(smvp_csr *A, cudaStream_t s)
{
    const int32_t tile_items = 32 * (merge_skewed(A) ? MergeSkewed::IPT : MergeStencil::IPT);
    if (A->merge_cfg == tile_items)
        return SMVP_OK;
    const int64_t total = (int64_t)A->rows + A->nnz;
    const int64_t tiles = ceil_div64(total, tile_items);
    if (tiles > 0x7ffffff0LL)
        return SMVP_E_TOOBIG;
    DevPtr<int32_t> tile_row;
    DevPtr<double> head_val, carry_val;
    SMVP_CUDA(dev_alloc(tile_row, tiles + 1));
    SMVP_CUDA(dev_alloc(head_val, tiles));
    SMVP_CUDA(dev_alloc(carry_val, tiles));
    SMVP_LAUNCH(merge_plan_kernel, (unsigned)ceil_div64(tiles + 1, 256), 256, 0, s, A->row_ptr.get(), A->rows, A->nnz, tile_items,
                (int32_t)tiles, tile_row.get());
    SMVP_CUDA(cudaGetLastError());
    A->tile_row = std::move(tile_row);
    A->head_val = std::move(head_val);
    A->carry_val = std::move(carry_val);
    A->merge_tiles = (int32_t)tiles;
    A->merge_cfg = tile_items; // the plan depends on the tile size only
    return SMVP_OK;
}

// Persistent grid with a static stride over the tiles: the CTAs that fit on the device at once, at most `need`.
// smvp_csr_set_corunner_headroom / SMVP_MERGE_HEADROOM=k: leave room for k more CTAs per SM.  Every CTA must be resident
// from the start: a CTA that has to wait for a co-running kernel's CTA to retire (the exchange kernel of the multi-GPU
// path) begins its full share of tiles late and the pass ends that much later (measured: SpMV 1.34 ms + copy kernel
// 0.42 ms side by side = 1.78 ms).
struct Residency // CTAs per SM of one kernel, looked up per device and dynamic shared-memory size
{
    int dev = -1, smem = -1, ctas = 1;
};
template <typename K>
static int persistent_grid(K kern, int threads, int smem, int handle_headroom, int64_t need, Residency &res, int64_t *grid)
{
    int dev = 0;
    SMVP_CUDA(cudaGetDevice(&dev));
    if (res.dev != dev || res.smem != smem)
    {
        SMVP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        SMVP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&res.ctas, kern, threads, smem));
        if (res.ctas < 1)
            res.ctas = 1;
        res.dev = dev;
        res.smem = smem;
    }
    static thread_local const int env_headroom = env_int("SMVP_MERGE_HEADROOM", -1, -1, 8);
    const int headroom = env_headroom >= 0 ? env_headroom : handle_headroom;
    const int used = res.ctas - headroom >= 1 ? res.ctas - headroom : 1;
    const int64_t g = (int64_t)device_props().sms * used;
    *grid = g > need ? need : g;
    return SMVP_OK;
}

// The fix-up after the merge kernel: launched early with programmatic stream serialization (it parks at
// griddepcontrol.wait) when `early`, an ordinary launch otherwise
template <typename K, typename... Args>
static int launch_fixup(bool early, int32_t ntiles, cudaStream_t s, K kern, Args... args)
{
    if (early)
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)ceil_div64(ntiles, 256));
        cfg.blockDim = dim3(256);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        SMVP_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
        ::smvp::g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    else
        SMVP_LAUNCH(kern, (unsigned)ceil_div64(ntiles, 256), 256, 0, s, args...);
    return SMVP_OK;
}

// (a fix-up fused into the kernel -- the last warp of the grid to finish walks the tiles -- was tried for the batched `-n`
// loop of small matrices: one warp serialises the few hundred tiles of a matrix like memplus, 12.1 us per pass against
// 5.7 us with the second launch.  Two launches it stays.)
static bool merge_fixup_early(int32_t ntiles)
{
    static thread_local const bool pdl_ok = !env_set("SMVP_NO_PDL"); // SMVP_NO_PDL: no early launch of the fix-up
    return pdl_ok && ntiles <= MERGE_PDL_TILES;
}

// tiles [tile_begin, tile_end) of the plan; a dot pass (whole passes only) leaves the partials of its tiles in
// dot->part[0, merge_tiles)
template <class C, bool RANKED, YStore M>
static int launch_wmerge(const smvp_csr *A, const double *d_x, double *d_y, const YFan *fanp, const Axpby &ab, const DotOut *dot,
                         cudaStream_t s, int32_t tile_begin, int32_t tile_end)
{
    constexpr int SMEM = C::WARPS * MergeShape<32, C::IPT>::SMEM_BYTES;
    auto kern = csr_merge_warp_kernel<C::WARPS, C::IPT, C::MINB, RANKED, C::UNI, M>;
    const int32_t hot_l1 = RANKED ? HOT_L1_ENTRIES : 0, hot_l2 = RANKED ? HOT_L2_ENTRIES : 0;
    const YFan fan = fanp ? *fanp : YFan();
    const double *w = dot ? dot->w : nullptr;
    double *part = dot ? dot->part : nullptr;
    static thread_local Residency res;
    const int32_t ntiles = tile_end - tile_begin;
    int64_t grid = 0;
    SMVP_TRY(persistent_grid(kern, C::WARPS * 32, SMEM, A->merge_headroom, ceil_div64(ntiles, C::WARPS), res, &grid));
    if (grid > 0)
    {
        const bool early = merge_fixup_early(ntiles);
        SMVP_LAUNCH(kern, (unsigned)grid, C::WARPS * 32, SMEM, s, A->row_ptr.get(), mult_cols(A), A->val.get(), d_x, d_y,
                    A->tile_row.get(), A->rows, A->nnz, tile_begin, tile_end, A->head_val.get(), A->carry_val.get(), fan, hot_l1,
                    hot_l2, early ? 1 : 0, ab.alpha, ab.beta, w, part);
        SMVP_TRY(launch_fixup(early, ntiles, s, merge_fixup_kernel<M>, (const int32_t *)A->tile_row.get(),
                              (const double *)A->head_val.get(), (const double *)A->carry_val.get(), tile_begin, tile_end, d_y, fan,
                              ab.alpha, ab.beta, w, part));
    }
    return SMVP_OK;
}

// =====================================================================================  PATTERN
// Handles with the row-pattern plan (pattern.cu): the kernel streams val and one pattern id per row, never col_ind.
// Row per lane: a warp tile is 32*R consecutive rows, lane l owns rows r0 + l, r0 + 32 + l, ...  The warp stages the
// tile's val slice and pat_id slice into its own shared-memory ring with TMA bulk copies (evict-first) and never meets a
// block-wide barrier after the pattern table is loaded.  Row starts inside the tile come from a warp scan of the pattern
// lengths (one row_ptr entry per tile, not per row).  Step k of a round gathers x[r + off_k]: on the 91 % of rounds whose
// 32 rows share a pattern that is 32 consecutive doubles, and the offset load is a shared-memory broadcast.  Each row is
// summed left to right from +0.0, product rounded then added -- the reference loop's order (main-cli.c:410-416), so y
// is bit-identical to it.  One launch per pass: no row is cut, nothing to stitch.
template <int R>
struct PatternShape
{
    static constexpr int ROWS = 32 * R;
    // value slice of vsize-byte values (16-byte aligned start and length: up to 16 / vsize - 1 extra values at each end)
    // + pat_id slice (16-byte aligned)
    static int stage_bytes(int maxlen, int vsize)
    {
        return (((ROWS * maxlen + 2 * (16 / vsize - 1)) * vsize + 15) / 16 * 16 + ROWS + 32 + 127) & ~127;
    }
};

// a value of the stage at shared address a, widened to fp64 (V: double, float or fp16 as uint16_t)
template <typename V>
__device__ __forceinline__ double lds_value(uint32_t a)
{
    if constexpr (std::is_same<V, double>::value)
        return lds_f64(a);
    else if constexpr (std::is_same<V, float>::value)
    {
        float v;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
        return widen_value(v);
    }
    else
    {
        uint16_t v;
        asm volatile("ld.shared.b16 %0, [%1];" : "=h"(v) : "r"(a));
        return widen_value(v);
    }
}

// Dot: whole passes only.  The work unit is the tile of 32 rows; the lanes' dot terms are added in a pairwise tree into
// part[t].  w[r] is loaded beside the early load of y[r].
// V: the width the values are streamed at (A->pat_vbytes): val itself (double), or the plan's copy A->pat_val (float or
// fp16 as uint16_t).  Narrow values are widened exactly (pattern.cu checked every one), so the products and sums are
// those of the fp64 kernel.
template <typename V, int WARPS, int R, int STAGES, int CH, int MINB, YStore M>
__global__ void __launch_bounds__(WARPS * 32, MINB)
    csr_pattern_kernel(const int32_t *__restrict__ row_ptr, const V *__restrict__ val, const uint8_t *__restrict__ pat_id,
                       const int32_t *__restrict__ pat_off, const int32_t *__restrict__ pat_len, int32_t npat, int32_t maxlen,
                       const double *__restrict__ x, double *__restrict__ y, int32_t row_first, int32_t row_end, uint32_t stage_bytes,
                       const __grid_constant__ YFan fan, double alpha, double beta, const double *__restrict__ dot_w,
                       double *__restrict__ part)
{
    static_assert(!reads_y(M) || R == 1, "the epilogue keeps one y value per lane: one round per tile");
    const int32_t row_begin = M == YStore::Dot ? 0 : row_first;
    constexpr int ROWS = PatternShape<R>::ROWS;
    constexpr int VA = 16 / (int)sizeof(V); // values per 16 bytes: the alignment of a bulk copy
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[WARPS * STAGES];
    __shared__ int32_t stage_n0[WARPS * STAGES]; // first nonzero of the tile in each stage
    // pattern table: offsets with row stride maxlen, then the lengths; the stages follow, 128-byte aligned
    const uint32_t table_bytes = ((uint32_t)npat * (uint32_t)(maxlen + 1) * 4u + 127u) & ~127u;
    int32_t *s_off = reinterpret_cast<int32_t *>(smem), *s_len = s_off + npat * maxlen;
    for (int i = threadIdx.x; i < npat * maxlen; i += WARPS * 32)
        s_off[i] = pat_off[(i / maxlen) * PAT_LMAX + i % maxlen];
    for (int i = threadIdx.x; i < npat; i += WARPS * 32)
        s_len[i] = pat_len[i];

    const int lane = threadIdx.x & 31, w = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    uint64_t *bars = &full_bar[w * STAGES];
    const uint32_t base = smem_u32(smem) + table_bytes + (uint32_t)(w * STAGES) * stage_bytes;
    const uint32_t val_bytes = (stage_bytes - ROWS - 32) & ~15u; // where the pat_id slice starts inside a stage
    uint64_t policy = 0;
    if (lane == 0)
    {
        for (int s = 0; s < STAGES; s++)
            mbar_init(&bars[s], 1);
        fence_mbar_init();
        policy = l2_evict_first_policy();
    }
    __syncthreads(); // the table is complete; from here on the warps are on their own

    const int32_t ntiles = (int32_t)(((int64_t)row_end - row_begin + ROWS - 1) / ROWS);
    const int32_t warp_stride = (int32_t)gridDim.x * WARPS;
    // rows [r0, r1) of tile t; lane 0 stages it (n0 = row_ptr[r0], n1 = row_ptr[r1] loaded by the caller)
    auto issue = [&](int32_t t, int s, int32_t n0, int32_t n1) {
        const int32_t r0 = row_begin + t * ROWS, r1 = min(r0 + ROWS, row_end);
        const int32_t va = n0 & ~(VA - 1), pa = r0 & ~15;
        const uint32_t vb = n1 > n0 ? (uint32_t)(((n1 + VA - 1) & ~(VA - 1)) - va) * (uint32_t)sizeof(V) : 0u;
        const uint32_t pb = (uint32_t)(((r1 + 15) & ~15) - pa);
        unsigned char *dst = smem + (base - smem_u32(smem)) + (uint32_t)s * stage_bytes;
        stage_n0[w * STAGES + s] = n0;
        mbar_expect_tx(&bars[s], vb + pb);
        if (vb)
            bulk_g2s(dst, val + va, vb, &bars[s], policy);
        bulk_g2s(dst + val_bytes, pat_id + pa, pb, &bars[s], policy);
    };
    auto bounds = [&](int32_t t, int32_t *n0, int32_t *n1) {
        const int32_t r0 = row_begin + t * ROWS;
        *n0 = __ldg(row_ptr + r0);
        *n1 = __ldg(row_ptr + min(r0 + ROWS, row_end));
    };

    int32_t t = (int32_t)blockIdx.x * WARPS + w;
#pragma unroll
    for (int s = 0; s < STAGES; s++)
    {
        const int32_t ts = t + s * warp_stride;
        if (ts < ntiles)
        {
            int32_t n0, n1;
            bounds(ts, &n0, &n1);
            if (lane == 0)
                issue(ts, s, n0, n1);
        }
    }
    __syncwarp();
    uint32_t phase = 0;
    int s = 0;
    while (t < ntiles)
    {
        // bounds of the tile this stage takes next: loaded now, used after the walk
        const int32_t tn = t + STAGES * warp_stride;
        int32_t nn0 = 0, nn1 = 0;
        if (tn < ntiles && tn > t)
            bounds(tn, &nn0, &nn1);
        // the epilogue's y[r]: issued before the wait for the stage, its latency hides behind the staging and the gathers
        double y0 = 0.0, w0 = 0.0;
        if (reads_y(M) && beta != 0.0 && row_begin + t * ROWS + lane < row_end)
            y0 = ld_y_early(y + row_begin + t * ROWS + lane);
        if (M == YStore::Dot && dot_w && row_begin + t * ROWS + lane < row_end)
            w0 = ld_w_early(dot_w + row_begin + t * ROWS + lane);
        double d = 0.0; // Dot: the lane's dot term

        mbar_wait(&bars[s], (phase >> s) & 1u);
        phase ^= 1u << s;
        const int32_t r0 = row_begin + t * ROWS, r1 = min(r0 + ROWS, row_end);
        const int32_t n0 = stage_n0[w * STAGES + s];
        const uint32_t sb = base + (uint32_t)s * stage_bytes;
        const uint32_t sval = sb + (uint32_t)sizeof(V) * (uint32_t)(n0 - (n0 & ~(VA - 1))); // nonzero n0
        const uint32_t spid = sb + val_bytes + (uint32_t)(r0 - (r0 & ~15)); // row r0
        int32_t done = 0; // nonzeros of the tile before the current round
#pragma unroll 1
        for (int i = 0; i < R; i++)
        {
            const int32_t rr = 32 * i;
            if (r0 + rr >= r1)
                break;
            const int32_t r = r0 + rr + lane;
            const bool live = r < r1;
            int32_t p = 0, len = 0;
            if (live)
            {
                asm volatile("ld.shared.u8 %0, [%1];" : "=r"(p) : "r"(spid + (uint32_t)(rr + lane)));
                len = s_len[p];
            }
            int32_t incl = len; // inclusive scan of the row lengths of the round
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const int32_t v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o)
                    incl += v;
            }
            const uint32_t vrow = sval + (uint32_t)sizeof(V) * (uint32_t)(done + incl - len);
            const uint32_t orow = smem_u32(s_off) + 4u * (uint32_t)(p * maxlen);
            done += __shfl_sync(0xffffffffu, incl, 31);
            const int32_t kmax = __reduce_max_sync(0xffffffffu, len);
            double sum = 0.0;
#pragma unroll 1
            for (int32_t k0 = 0; k0 < kmax; k0 += CH)
            {
                // three phases pinned by volatile asm: the offsets, every gather of the chunk (CH loads in flight), the sums
                int32_t off[CH];
                double xv[CH];
#pragma unroll
                for (int q = 0; q < CH; q++)
                    off[q] = k0 + q < len ? lds_s32(orow + 4u * (uint32_t)(k0 + q)) : 0;
#pragma unroll
                for (int q = 0; q < CH; q++)
                {
                    xv[q] = 0.0;
                    if (k0 + q < len)
                        xv[q] = ldg_x_pinned(x, r + off[q]);
                }
#pragma unroll
                for (int q = 0; q < CH; q++)
                    if (k0 + q < len)
                        sum = __dadd_rn(sum, __dmul_rn(lds_value<V>(vrow + (uint32_t)sizeof(V) * (uint32_t)(k0 + q)), xv[q]));
            }
            if (live)
            {
                if constexpr (reads_y(M))
                {
                    const double v = axpby(alpha, sum, beta, y0);
                    y[r] = v;
                    if constexpr (M == YStore::Dot)
                        d = __dmul_rn(dot_w ? w0 : v, v);
                }
                else
                    store_row<M>(y, r, sum, alpha, beta, dot_w, &fan);
            }
        }
        if constexpr (M == YStore::Dot)
        {
            d = warp_tree_sum(d);
            if (lane == 0)
                part[t] = d;
        }
        // the stage is consumed: refill it with tile tn
        __syncwarp();
        if (tn < ntiles && tn > t && lane == 0)
            issue(tn, s, nn0, nn1);
        __syncwarp();
        if (t + warp_stride <= t)
            break; // 32-bit overflow guard
        t += warp_stride;
        s = s + 1 == STAGES ? 0 : s + 1;
    }
}
// ---- the pattern kernel's configuration.  Measured on B200 (profiles/r03_logs/sweep_pattern.log, stencil 369^3, the
// swept configurations in DESIGN.md §5.2): one stage per warp and 28 warps per SM (1.75 ms) against 2.1-3.2 ms for every
// configuration with two stages or two rounds per tile -- a 7 KB stage per warp, so resident warps, not staging depth,
// keep enough gathers in flight.
struct PatternCfg
{
    static constexpr int WARPS = 4; // warps per CTA
    static constexpr int R = 1;     // rounds of 32 rows per tile
    static constexpr int STAGES = 1; // stages per warp
    static constexpr int CH = 14;   // gathers in flight per lane
    static constexpr int MINB = 7;  // min CTAs per SM
};
// narrow values: a smaller stage per warp, so more CTAs fit.  Swept per width on the same stencil over {CH, CTAs/SM} =
// {14, 7}, {14, 8}, {14, 9}, {10, 10}, {8, 12}, {6, 16 (fp32: 13)} (profiles/r05_logs/sweep_width.log, DESIGN.md §5.2):
// fp16 keeps fp64's configuration, fp32 takes 8 CTAs/SM.  WARPS and R stay those of fp64 at every width: the dot's work
// units are tiles of 32 rows.
template <typename V>
struct PatternCfgOf : PatternCfg
{
};
template <>
struct PatternCfgOf<float> : PatternCfg
{
    static constexpr int MINB = 8;
};

// rows [row_begin, row_end); a dot pass (whole passes only) leaves the partial of tile t in dot->part[t]
template <typename V>
static int launch_pattern(const smvp_csr *A, const V *val, const double *d_x, double *d_y, const YFan *fan, const Axpby &ab,
                          cudaStream_t s, int32_t row_begin, int32_t row_end, const DotOut *dot)
{
    using C = PatternCfgOf<V>;
    const int maxlen = A->pattern_maxlen > 0 ? A->pattern_maxlen : 1;
    const int stage = PatternShape<C::R>::stage_bytes(maxlen, (int)sizeof(V));
    const int table = (A->pattern_count * (maxlen + 1) * 4 + 127) & ~127;
    const int smem = table + C::WARPS * C::STAGES * stage;
    const int64_t need = ceil_div64(ceil_div64((int64_t)row_end - row_begin, PatternShape<C::R>::ROWS), C::WARPS);
    return with_store<YStore::Plain, YStore::Fanout, YStore::Axpby, YStore::Dot>(store_mode(dot, fan, ab), [&](auto S) {
        auto kern = csr_pattern_kernel<V, C::WARPS, C::R, C::STAGES, C::CH, C::MINB, decltype(S)::value>;
        // the shared memory depends on the matrix (longest pattern, pattern count): occupancy is looked up per size
        static thread_local Residency res;
        int64_t grid = 0;
        SMVP_TRY(persistent_grid(kern, C::WARPS * 32, smem, A->merge_headroom, need, res, &grid));
        if (grid > 0)
            SMVP_LAUNCH(kern, (unsigned)grid, C::WARPS * 32, smem, s, A->row_ptr.get(), val, A->pat_id.get(), A->pat_off.get(),
                        A->pat_len.get(), A->pattern_count, maxlen, d_x, d_y, row_begin, row_end, (uint32_t)stage, fan ? *fan : YFan(),
                        ab.alpha, ab.beta, dot ? dot->w : nullptr, dot ? dot->part : nullptr);
        return (int)SMVP_OK;
    });
}

// rows [row_begin, row_end) of a handle with the row-pattern plan, its values streamed at the plan's width
static int csr_mult_pattern(const smvp_csr *A, const double *d_x, double *d_y, const YFan *fan, const Axpby &ab, cudaStream_t s,
                            int32_t row_begin, int32_t row_end, const DotOut *dot = nullptr)
{
    if (A->pat_vbytes == 2)
        return launch_pattern(A, (const uint16_t *)A->pat_val.get(), d_x, d_y, fan, ab, s, row_begin, row_end, dot);
    if (A->pat_vbytes == 4)
        return launch_pattern(A, (const float *)A->pat_val.get(), d_x, d_y, fan, ab, s, row_begin, row_end, dot);
    return launch_pattern(A, (const double *)A->val.get(), d_x, d_y, fan, ab, s, row_begin, row_end, dot);
}

constexpr Axpby AXPBY_PLAIN = {1.0, 0.0};

// tiles [tile_begin, tile_end) of the plan; (0, -1) = all
// dot != NULL: a whole pass with the epilogue whose dot partials go to dot->part (csr_dot_units counts them)
static int csr_mult_merge(smvp_csr *A, const double *d_x, double *d_y, const YFan *fan, const Axpby &ab, cudaStream_t s,
                          int32_t tile_begin = 0, int32_t tile_end = -1, const DotOut *dot = nullptr)
{
    // the row-pattern plan serves whole passes (the pipelined host call cuts its ranges on rows: csr_mult_pattern)
    if (A->pattern_state == 1 && tile_begin == 0 && tile_end < 0)
        return csr_mult_pattern(A, d_x, d_y, fan, ab, s, 0, A->rows, dot);
    SMVP_TRY(merge_plan(A, s));
    if (tile_end < 0)
        tile_end = A->merge_tiles;
    // a relabelled handle indexes x by popularity rank: the gathers carry cache-retention hints (without them: 7.62 against
    // 6.69 ms on R-MAT scale 26, DESIGN.md §5.4)
    const bool ranked = A->relabel_state == 1;
    const bool skewed = merge_skewed(A);
    return with_flag(ranked, [&](auto R) {
        return with_store<YStore::Plain, YStore::Fanout, YStore::Axpby, YStore::Dot>(store_mode(dot, fan, ab), [&](auto S) {
            constexpr bool RANKED = decltype(R)::value;
            constexpr YStore M = decltype(S)::value;
            return skewed ? launch_wmerge<MergeSkewed, RANKED, M>(A, d_x, d_y, fan, ab, dot, s, tile_begin, tile_end)
                          : launch_wmerge<MergeStencil, RANKED, M>(A, d_x, d_y, fan, ab, dot, s, tile_begin, tile_end);
        });
    });
}

// work units of a dot pass with resolved variant v (DESIGN.md §5.7); builds the plan they depend on
static int csr_dot_units(smvp_csr *A, int v, cudaStream_t s, int64_t *units)
{
    if (v == SMVP_CSR_VECTOR)
        *units = ceil_div64((int64_t)A->rows * vector_lpr(A), 256); // the vector kernel's CTAs
    else if (A->pattern_state == 1)
        *units = ceil_div64(A->rows, PatternShape<PatternCfg::R>::ROWS);
    else
    {
        SMVP_TRY(merge_plan(A, s));
        *units = A->merge_tiles;
    }
    return SMVP_OK;
}

// the most work units any plan of the handle can give a dot pass: the scratch is sized for it at the first dot call, so
// that a later call with another variant or plan never allocates (nor synchronises)
static int64_t csr_dot_units_max(const smvp_csr *A)
{
    constexpr int32_t min_tile = 32 * (MergeSkewed::IPT < MergeStencil::IPT ? MergeSkewed::IPT : MergeStencil::IPT);
    const int64_t vec = ceil_div64((int64_t)A->rows * vector_lpr(A), 256);
    const int64_t pat = ceil_div64(A->rows, PatternShape<PatternCfg::R>::ROWS);
    const int64_t merge = ceil_div64((int64_t)A->rows + A->nnz, min_tile);
    const int64_t m = vec > pat ? vec : pat;
    return m > merge ? m : merge;
}

int csr_resolve_variant(const smvp_csr *A, int variant)
{
    if (variant == SMVP_CSR_AUTO)
    {
        const char *env = env_str("SMVP_CSR_VARIANT");
        if (env && (env[0] == '1' || env[0] == '2'))
            return env[0] - '0';
        return A->auto_variant;
    }
    return variant;
}

} // namespace smvp

using namespace smvp;

// x is already in the space the kernels index (x itself, or x_rel when the relabelling plan is in use)
static int csr_mult_launch(smvp_csr *A, const double *x, double *d_y, const YFan *fan, const Axpby &ab, int variant, cudaStream_t s,
                           const DotOut *dot = nullptr)
{
    if (A->rows == 0)
        return SMVP_OK;
    const int v = csr_resolve_variant(A, variant);
    int rc = (v == SMVP_CSR_VECTOR) ? csr_mult_vector(A, x, d_y, fan, ab, dot, s) : csr_mult_merge(A, x, d_y, fan, ab, s, 0, -1, dot);
    if (rc != SMVP_OK)
        return rc;
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

// d_dot != NULL: a dot pass (smvp_csr_mult_device_axpby_dot), *d_dot = sum of w[r] * y_new[r] (w = d_w, or y_new)
static int csr_mult_any(smvp_csr *A, const double *d_x, double *d_y, const YFan *fan, const Axpby &ab, int variant, void *stream,
                        const double *d_w = nullptr, double *d_dot = nullptr)
{
    if (variant != SMVP_CSR_AUTO && variant != SMVP_CSR_VECTOR && variant != SMVP_CSR_MERGE)
        return SMVP_E_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    if (A->rows == 0)
    {
        if (!d_dot)
            return SMVP_OK;
        SMVP_TRY(dot_scratch(&A->dot_buf, &A->dot_cap, &A->device_bytes, csr_dot_units_max(A), s));
        return dot_reduce(A->dot_buf.get(), A->dot_cap, 0, d_dot, s); // no rows: +0.0
    }
    SMVP_TRY(csr_pattern_plan(A, s)); // decides the relabelling first
    const double *x = d_x; // NULL: the x last given to smvp_csr_set_x_device
    if (A->relabel_state == 1)
    {
        if (d_x)
            SMVP_TRY(csr_relabel_x(A, d_x, s));
        else if (!A->x_set)
            return SMVP_E_ARG;
        x = A->x_rel.get();
    }
    else if (!d_x)
    {
        x = A->x_set;
        if (!x && A->cols > 0)
            return SMVP_E_ARG;
    }
    if (!d_dot)
        return csr_mult_launch(A, x, d_y, fan, ab, variant, s);
    int64_t units = 0;
    SMVP_TRY(csr_dot_units(A, csr_resolve_variant(A, variant), s, &units));
    SMVP_TRY(dot_scratch(&A->dot_buf, &A->dot_cap, &A->device_bytes, csr_dot_units_max(A), s));
    const DotOut dot = {d_w, A->dot_buf.get()};
    SMVP_TRY(csr_mult_launch(A, x, d_y, nullptr, ab, variant, s, &dot));
    return dot_reduce(A->dot_buf.get(), A->dot_cap, units, d_dot, s);
}

extern "C" int smvp_csr_set_x_device(smvp_csr *A, const double *d_x, void *stream)
{
    if (!A || (A->cols > 0 && !d_x))
        return SMVP_E_ARG;
    SMVP_TRY(csr_pattern_plan(A, (cudaStream_t)stream)); // decides the relabelling first
    if (A->relabel_state == 1)
        SMVP_TRY(csr_relabel_x(A, d_x, (cudaStream_t)stream));
    A->x_set = d_x;
    return SMVP_OK;
}

extern "C" int smvp_csr_set_corunner_headroom(smvp_csr *A, int ctas_per_sm)
{
    if (!A || ctas_per_sm < 0 || ctas_per_sm > 8)
        return SMVP_E_ARG;
    A->merge_headroom = ctas_per_sm;
    return SMVP_OK;
}

extern "C" int smvp_csr_mult_device(smvp_csr *A, const double *d_x, double *d_y, int variant, void *stream)
{
    if (!A || (A->rows > 0 && !d_y))
        return SMVP_E_ARG;
    return csr_mult_any(A, d_x, d_y, nullptr, AXPBY_PLAIN, variant, stream);
}

extern "C" int smvp_csr_mult_device_axpby(smvp_csr *A, double alpha, const double *d_x, double beta, double *d_y, int variant,
                                          void *stream)
{
    if (!A || (A->rows > 0 && !d_y))
        return SMVP_E_ARG;
    if (d_y && d_y == (d_x ? d_x : A->x_set))
        return SMVP_E_ARG; // y would be read and written while the kernels gather it as x
    return csr_mult_any(A, d_x, d_y, nullptr, Axpby{alpha, beta}, variant, stream);
}

extern "C" int smvp_csr_mult_device_axpby_dot(smvp_csr *A, double alpha, const double *d_x, double beta, double *d_y,
                                              const double *d_w, double *d_dot, int variant, void *stream)
{
    if (!A || (A->rows > 0 && !d_y) || !d_dot)
        return SMVP_E_ARG;
    const double *x = d_x ? d_x : A->x_set;
    if (d_y && d_y == x)
        return SMVP_E_ARG; // y would be read and written while the kernels gather it as x
    if ((d_w && d_w == d_y) || d_dot == x || d_dot == d_y || d_dot == d_w)
        return SMVP_E_ARG;
    return csr_mult_any(A, d_x, d_y, nullptr, Axpby{alpha, beta}, variant, stream, d_w, d_dot);
}

extern "C" int smvp_csr_mult_device_fanout(smvp_csr *A, const double *d_x, double *const *d_y_list, int n_out, int variant,
                                           void *stream)
{
    if (!A || !d_y_list || n_out < 1 || n_out > SMVP_MAX_FANOUT)
        return SMVP_E_ARG;
    YFan fan;
    fan.n = n_out;
    for (int k = 0; k < SMVP_MAX_FANOUT; k++)
        fan.p[k] = k < n_out ? d_y_list[k] : nullptr;
    for (int k = 0; k < n_out; k++)
        if (A->rows > 0 && !fan.p[k])
            return SMVP_E_ARG;
    return csr_mult_any(A, d_x, fan.p[0], &fan, AXPBY_PLAIN, variant, stream);
}

// ------------------------------------------------------------------ host-vector entry point
// For large matrices the pass that touches the host is cut into consecutive ranges (32 by default) of merge-path
// tiles and pipelined against both PCIe directions:
//   * first pass: x goes up in pieces (64 by default) on an upload stream; range c starts as soon as the leading
//     part of x it reads (x[0 .. xneed_c), xneed_c = 1 + the largest column index among its nonzeros, a property
//     of the matrix found once per handle) has arrived.  A banded matrix (stencils, meshes) therefore multiplies
//     while x is still uploading; a matrix whose first rows reach the last column simply waits for all of x.
//   * last pass: the rows a range completes are copied to the host on a download stream while the next range
//     multiplies.
// With iters == 1 both happen in the same pass and the call costs about ONE vector transfer (PCIe is full
// duplex) instead of upload + multiply + download back to back.  ms_each still reports the multiply alone: the
// sum of the ranges' own event brackets, each opened after the range's wait for x.
// Piece sizes from the sweep on B200 (DESIGN.md §6, profiles/).  Piece SIZE, not piece count, is fixed, so the fixed cost
// of a call shrinks with the block a rank owns (round 1: e2e did not scale with N).  6 MB in both directions: on the
// 402 MB vectors of the 369^3 stencil that is 64 ranges x 64 upload pieces, the best of every sweep (round 2: 9.8 ms per
// call against 12.2 ms for 32 x 64 and 11.2 ms for 16 x 16 in the same run; the PCIe floor with both directions busy is
// 8.05 ms).  SMVP_PIPE_TRACE=1 shows why the numbers scatter: with both directions busy the UPLOAD of the 402 MB ends
// anywhere between 8.3 and 11.5 ms depending on how the pieces of the two directions interleave, equal-sized pieces
// interleave best.  Price: a pass cut into 64 ranges spends 5.7 ms of GPU time instead of 2.7 (short launches), which is
// what ms_each reports for it.
// Shorter vectors (the row block of one GPU out of N) download in 12 MB pieces: 17 ranges x 33 upload pieces measured
// 6.8 ms per call on the 201 MB blocks of 2 GPUs, 32 x 33 measured 7.95 ms.
constexpr int64_t PIPE_DOWN_PIECE_BYTES = 12 << 20;
constexpr int64_t PIPE_DOWN_PIECE_BYTES_LONG = 6 << 20; // vectors of 300 MB and more
constexpr int64_t PIPE_UP_PIECE_BYTES = 6 << 20;
static int pipe_ranges(int64_t y_bytes)
{
    const int64_t want = ceil_div64(y_bytes, y_bytes >= (300ll << 20) ? PIPE_DOWN_PIECE_BYTES_LONG : PIPE_DOWN_PIECE_BYTES);
    return (int)(want < 2 ? 2 : (want > PIPE_MAX_RANGES ? PIPE_MAX_RANGES : want));
}
static int pipe_xchunks(int64_t x_bytes)
{
    const int64_t want = ceil_div64(x_bytes, PIPE_UP_PIECE_BYTES);
    return (int)(want < 2 ? 2 : (want > PIPE_MAX_XCHUNKS ? PIPE_MAX_XCHUNKS : want));
}

// n equal pieces: boundaries f[0] = 0 ... f[n] = 1 as fractions of the whole.  (Ramped pieces -- 2, 4, 8, 16 MB at both
// ends, 24 MB in the middle -- lost: 10.9 ms per call against 9.8 ms; with both directions busy, many small equal pieces
// interleave better than a few large ones.)
static void pipe_profile(int n, double *f)
{
    for (int i = 0; i <= n; i++)
        f[i] = (double)i / n;
}

// largest and smallest column index among nonzeros [n0, n1): out[0] = max (start -1), out[1] = min (start INT32_MAX)
__global__ void __launch_bounds__(256) col_range_kernel(const int32_t *__restrict__ col_ind, int64_t n0, int64_t n1,
                                                        int32_t *__restrict__ out)
{
    int32_t hi = -1, lo = 0x7fffffff;
    for (int64_t j = n0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n1; j += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t c = __ldg(col_ind + j);
        hi = max(hi, c);
        lo = min(lo, c);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    }
    if ((threadIdx.x & 31) == 0 && hi >= 0)
    {
        atomicMax(out, hi);
        atomicMin(out + 1, lo);
    }
}

// Ranges of a handle with the row-pattern plan are cut on rows (the pattern kernel takes a row range, pipe_tile = pipe_row);
// pipe_cfg is then PIPE_CFG_PATTERN instead of a merge tile size.
constexpr int32_t PIPE_CFG_PATTERN = -2;
static int pipe_plan(smvp_csr *A)
{
    const bool pat = A->pattern_state == 1;
    if (!pat)
        SMVP_TRY(merge_plan(A, 0));
    const int NR = pipe_ranges(8 * (int64_t)A->rows);
    const int32_t key = pat ? PIPE_CFG_PATTERN : A->merge_cfg;
    if (A->pipe_cfg == key && A->pipe_ranges == NR)
        return SMVP_OK;
    double rf[PIPE_MAX_RANGES + 1];
    pipe_profile(NR, rf);
    const int32_t T = pat ? 0 : A->merge_tiles;
    const int64_t tile_items = pat ? 0 : A->merge_cfg;
    DevPtr<int32_t> d_max; // per range: {largest, smallest} column index
    int32_t h_max[2 * PIPE_MAX_RANGES];
    for (int c = 0; c < PIPE_MAX_RANGES; c++)
    {
        h_max[2 * c] = -1; // the range reads no x at all
        h_max[2 * c + 1] = 0x7fffffff;
    }
    SMVP_CUDA(dev_alloc(d_max, 2 * PIPE_MAX_RANGES));
    SMVP_CUDA(cudaMemcpy(d_max.get(), h_max, sizeof(h_max), cudaMemcpyHostToDevice));
    int32_t pat_nz[PIPE_MAX_RANGES + 1]; // pattern plan: first nonzero of each range (row_ptr at its first row)
    for (int c = 0; c <= NR; c++)
    {
        if (pat)
        {
            A->pipe_tile[c] = A->pipe_row[c] = c == NR ? A->rows : (int32_t)((double)A->rows * rf[c]);
            SMVP_CUDA(cudaMemcpy(&pat_nz[c], A->row_ptr.get() + A->pipe_row[c], sizeof(int32_t), cudaMemcpyDeviceToHost));
            continue;
        }
        A->pipe_tile[c] = c == NR ? T : (int32_t)((double)T * rf[c]);
        // rows consumed before each boundary tile (tile_row[T] = rows)
        SMVP_CUDA(cudaMemcpy(&A->pipe_row[c], A->tile_row.get() + A->pipe_tile[c], sizeof(int32_t), cudaMemcpyDeviceToHost));
    }
    for (int c = 0; c < NR; c++)
    {
        // nonzeros of the range: merge items before the boundary minus the row ends among them
        int64_t n0 = pat ? pat_nz[c] : (int64_t)A->pipe_tile[c] * tile_items - A->pipe_row[c];
        int64_t n1 = pat ? pat_nz[c + 1] : (int64_t)A->pipe_tile[c + 1] * tile_items - A->pipe_row[c + 1];
        n0 = n0 < A->nnz ? n0 : A->nnz;
        n1 = (c + 1 == NR || n1 > A->nnz) ? A->nnz : n1;
        if (n1 > n0)
        {
            int64_t grid = ceil_div64(n1 - n0, 256 * 16);
            const int64_t cap = (int64_t)device_props().sms * 8;
            SMVP_LAUNCH(col_range_kernel, (unsigned)(grid < cap ? grid : cap), 256, 0, 0, (const int32_t *)A->col_ind.get(), n0, n1,
                        d_max.get() + 2 * c);
        }
    }
    SMVP_CUDA(cudaMemcpy(h_max, d_max.get(), sizeof(h_max), cudaMemcpyDeviceToHost));
    int32_t need = 0, lowest = 0x7fffffff; // x arrives front to back: a range needs everything up to the largest column so far
    for (int c = 0; c < NR; c++)
    {
        need = h_max[2 * c] + 1 > need ? h_max[2 * c] + 1 : need;
        lowest = h_max[2 * c + 1] < lowest ? h_max[2 * c + 1] : lowest;
        A->pipe_xneed[c] = need;
    }
    // nothing below the smallest column index is ever read: the upload starts there (a row block of a banded matrix,
    // the shard of one GPU, reads a window of x, not a prefix).  Rounded down to 512 bytes.
    A->pipe_xlo = need > 0 ? (lowest / 64) * 64 : 0;
    A->pipe_cfg = key;
    A->pipe_ranges = NR;
    return SMVP_OK;
}

// one pass in ranges; x_host != NULL: upload x under the pass; y_host != NULL: download y under the pass
static int csr_mult_pipelined(smvp_csr *A, const double *x_host, double *y_host, float *ms)
{
    SMVP_TRY(pipe_plan(A));
    if (!A->pipe_res) // streams and events live with the handle: creating ~160 events per call costs more than a range
    {
        std::unique_ptr<PipeResources> fresh(new (std::nothrow) PipeResources());
        if (!fresh)
            return SMVP_E_ALLOC;
        // the pass runs on its own non-blocking stream: the legacy stream would serialise it against every other
        // blocking stream of the process
        SMVP_CUDA(cudaStreamCreateWithFlags(out(fresh->compute), cudaStreamNonBlocking));
        SMVP_CUDA(cudaEventCreate(out(fresh->begin)));
        SMVP_CUDA(cudaStreamCreateWithFlags(out(fresh->up), cudaStreamNonBlocking));
        SMVP_CUDA(cudaStreamCreateWithFlags(out(fresh->down), cudaStreamNonBlocking));
        for (Event &ev : fresh->x_ready)
            SMVP_CUDA(cudaEventCreate(out(ev)));
        for (int c = 0; c < PIPE_MAX_RANGES; c++)
        {
            SMVP_CUDA(cudaEventCreate(out(fresh->done[c])));
            SMVP_CUDA(cudaEventCreate(out(fresh->down_done[c])));
            SMVP_CUDA(cudaEventCreate(out(fresh->t0[c])));
            SMVP_CUDA(cudaEventCreate(out(fresh->t1[c])));
        }
        A->pipe_res = std::move(fresh);
    }
    const PipeResources &R = *A->pipe_res;
    cudaError_t e = cudaSuccess;
    // the part of x this matrix reads: [xlo, xhi).  Entries outside it are never gathered, so they are not uploaded
    const int NR = A->pipe_ranges;
    const int64_t xlo = A->pipe_xlo, xhi = NR > 0 ? A->pipe_xneed[NR - 1] : 0;
    const int64_t xlen = xhi > xlo ? xhi - xlo : 0;
    const int NX = pipe_xchunks(8 * xlen);
    double xf[PIPE_MAX_XCHUNKS + 1];
    pipe_profile(NX, xf);
    int64_t xb[PIPE_MAX_XCHUNKS + 1]; // piece k uploads x[xb[k], xb[k+1]) (boundaries on 512-byte multiples)
    for (int k = 0; k <= NX; k++)
    {
        int64_t at = xlo + (((int64_t)((double)xlen * xf[k]) + 63) / 64) * 64;
        xb[k] = (k == NX || at > xhi) ? xhi : at;
    }
    cudaStream_t cs = R.compute.get();
    // first failing runtime call of the pass; later calls are skipped, the streams are still drained below
#define PIPE_CK(expr)            \
    do                           \
    {                            \
        if (e == cudaSuccess)    \
            e = (expr);          \
    } while (0)
    // everything queued on the legacy stream before the call (the zero-fill of y, an earlier pass) comes first
    PIPE_CK(cudaEventRecord(R.begin.get(), 0));
    PIPE_CK(cudaStreamWaitEvent(cs, R.begin.get(), 0));
    PIPE_CK(cudaStreamWaitEvent(R.up.get(), R.begin.get(), 0));
    PIPE_CK(cudaStreamWaitEvent(R.down.get(), R.begin.get(), 0));
    if (x_host)
    {
        for (int k = 0; k < NX; k++)
        {
            const int64_t a = xb[k], b = xb[k + 1];
            if (b > a)
                PIPE_CK(cudaMemcpyAsync(A->d_x.get() + a, x_host + a, sizeof(double) * (size_t)(b - a), cudaMemcpyHostToDevice,
                                        R.up.get()));
            PIPE_CK(cudaEventRecord(R.x_ready[k].get(), R.up.get()));
        }
    }
    int rc = SMVP_OK;
    const double *xm = A->relabel_state == 1 ? A->x_rel.get() : A->d_x.get(); // callers upload under the pass only without relabelling
    int waited = -1; // last upload piece the compute stream already waits for
    for (int c = 0; c < NR && rc == SMVP_OK && e == cudaSuccess; c++)
    {
        if (x_host && A->pipe_xneed[c] > xlo)
        {
            int k = waited < 0 ? 0 : waited; // first piece whose end covers what the range reads
            while (k < NX - 1 && xb[k + 1] < (int64_t)A->pipe_xneed[c])
                k++;
            if (k > waited) // the pieces complete in order on one stream: piece k's event covers every earlier one
            {
                PIPE_CK(cudaStreamWaitEvent(cs, R.x_ready[k].get(), 0));
                waited = k;
            }
        }
        PIPE_CK(cudaEventRecord(R.t0[c].get(), cs));
        if (A->pipe_tile[c + 1] > A->pipe_tile[c] && e == cudaSuccess)
            rc = A->pattern_state == 1
                     ? csr_mult_pattern(A, xm, A->d_y.get(), nullptr, AXPBY_PLAIN, cs, A->pipe_row[c], A->pipe_row[c + 1])
                     : csr_mult_merge(A, xm, A->d_y.get(), nullptr, AXPBY_PLAIN, cs, A->pipe_tile[c], A->pipe_tile[c + 1]);
        PIPE_CK(cudaEventRecord(R.t1[c].get(), cs));
        if (y_host)
        {
            PIPE_CK(cudaEventRecord(R.done[c].get(), cs));
            PIPE_CK(cudaStreamWaitEvent(R.down.get(), R.done[c].get(), 0));
            const int32_t r0 = A->pipe_row[c], r1 = A->pipe_row[c + 1];
            if (r1 > r0)
                PIPE_CK(cudaMemcpyAsync(y_host + r0, A->d_y.get() + r0, sizeof(double) * (size_t)(r1 - r0), cudaMemcpyDeviceToHost,
                                        R.down.get()));
            PIPE_CK(cudaEventRecord(R.down_done[c].get(), R.down.get()));
        }
    }
    // drain every stream of the pass, also after a failure (nothing may still touch the caller's buffers on return)
    cudaError_t es = cudaStreamSynchronize(cs);
    // the upload stream too: a matrix may read less than all of x
    const cudaError_t eu = cudaStreamSynchronize(R.up.get()), ed = cudaStreamSynchronize(R.down.get());
    if (es == cudaSuccess)
        es = eu != cudaSuccess ? eu : ed;
#undef PIPE_CK
    if (rc != SMVP_OK)
        return rc;
    if (e == cudaSuccess)
        e = es;
    if (e != cudaSuccess)
        return cuda_fail(e, "pipelined pass", __FILE__, __LINE__);
    float total = 0.f;
    for (int c = 0; c < NR; c++)
    {
        float t = 0.f;
        cudaEventElapsedTime(&t, R.t0[c].get(), R.t1[c].get());
        total += t;
    }
    *ms = total;
    if (env_set("SMVP_PIPE_TRACE")) // where the pass spends its time (ms after the start of the pass)
    {
        auto at = [&](cudaEvent_t ev) {
            float t = 0.f;
            cudaEventElapsedTime(&t, R.begin.get(), ev);
            return t;
        };
        fprintf(stderr, "[pipe] %d ranges, %d x pieces (first %lld, largest %lld entries): ", NR, NX, (long long)(xb[1] - xb[0]),
                (long long)(NX > 4 ? xb[NX / 2 + 1] - xb[NX / 2] : xb[1] - xb[0]));
        if (x_host)
            fprintf(stderr, "x piece 0 at %.3f, last x piece at %.3f | ", at(R.x_ready[0].get()), at(R.x_ready[NX - 1].get()));
        fprintf(stderr, "range 0 computed at %.3f, last range at %.3f", at(R.t1[0].get()), at(R.t1[NR - 1].get()));
        if (y_host)
            fprintf(stderr, " | first rows down at %.3f, last rows down at %.3f", at(R.down_done[0].get()),
                    at(R.down_done[NR - 1].get()));
        fprintf(stderr, " ms\n");
    }
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

extern "C" int smvp_csr_mult(smvp_csr *A, const double *x_host, double *y_host, int iters, double *ms_each, int variant)
{
    if (!A || iters < 1 || (A->cols > 0 && !x_host) || (A->rows > 0 && !y_host))
        return SMVP_E_ARG;
    if (variant != SMVP_CSR_AUTO && variant != SMVP_CSR_VECTOR && variant != SMVP_CSR_MERGE)
        return SMVP_E_ARG;
    if (!A->d_x)
        SMVP_CUDA(dev_alloc(A->d_x, A->cols));
    if (!A->d_y)
        SMVP_CUDA(dev_alloc(A->d_y, A->rows));
    const bool merge = csr_resolve_variant(A, variant) == SMVP_CSR_MERGE && A->rows > 0;
    // big vectors: pipeline their PCIe transfers with the first / last pass (SMVP_NO_OVERLAP=1: plain copies).
    // Only from page-locked buffers (smvp_host_alloc, cudaHostAlloc, torch pin_memory): an asynchronous copy from or to
    // PAGEABLE memory blocks the host until it is done, so every range would be enqueued only after the previous
    // range's download and the GPU would idle in between -- plain copies are faster then.  SMVP_FORCE_OVERLAP=1
    // pipelines regardless (tests).
    auto page_locked = [](const void *p) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess)
        {
            cudaGetLastError();
            return false;
        }
        return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
    };
    const bool pipelined = merge && ((int64_t)A->rows + A->cols) >= (1 << 21) && !env_set("SMVP_NO_OVERLAP") &&
                           (env_set("SMVP_FORCE_OVERLAP") || (page_locked(x_host) && page_locked(y_host)));
    int rc = SMVP_OK;
    // plans outside the timed bracket (the reference builds its format before the loop too)
    if (A->rows > 0)
        rc = csr_pattern_plan(A, 0); // decides the relabelling first
    if (rc == SMVP_OK && pipelined)
        rc = pipe_plan(A);
    else if (rc == SMVP_OK && merge && A->pattern_state != 1)
        rc = merge_plan(A, 0);
    if (rc != SMVP_OK)
        return rc;
    const bool relabeled = A->relabel_state == 1;
    const bool upload_under_pass = pipelined && !relabeled; // a relabelled x has to be complete before it is permuted
    if (A->cols > 0 && !upload_under_pass)
        SMVP_CUDA(cudaMemcpy(A->d_x.get(), x_host, sizeof(double) * (size_t)A->cols, cudaMemcpyHostToDevice));
    if (relabeled) // once, before the loop, as the reference permutes x for TJDS (main-cli.c:907-923)
        SMVP_TRY(csr_relabel_x(A, A->d_x.get(), 0));
    const double *xm = relabeled ? A->x_rel.get() : A->d_x.get();
    bool y_copied = false;
    // y is zero-filled outside the timed passes (main-cli.c:405); both kernels write every row, the fill only keeps
    // the reference's structure observable
    if (A->rows > 0)
        SMVP_CUDA(cudaMemsetAsync(A->d_y.get(), 0, sizeof(double) * (size_t)A->rows, 0));
    if (!pipelined)
    {
        // small matrices: a pass is shorter than a launch + synchronisation, so the loop runs batched in CUDA graphs
        const bool small = (int64_t)A->rows + A->cols + A->nnz < SMVP_SMALL_LOOP_ITEMS;
        // (an explicitly requested variant is honoured pass by pass; AUTO may pick the looping kernel)
        const bool tiny = variant == SMVP_CSR_AUTO && A->nnz <= TINY_MAX_NNZ && A->rows <= TINY_MAX_ROWS &&
                          !env_set("SMVP_NO_TINY_LOOP");
        std::function<int(cudaStream_t, int)> multi;
        if (tiny)
            multi = [&](cudaStream_t s, int n) {
                const double mean = A->rows > 0 ? (double)A->nnz / A->rows : 0.0;
#define SMVP_TINY(L)                                                                                                              \
    SMVP_LAUNCH(csr_tiny_loop_kernel<L>, 1, TINY_THREADS, 0, s, (const int32_t *)A->row_ptr.get(), mult_cols(A),                   \
                (const double *)A->val.get(), xm, A->d_y.get(), A->rows, n)
                if (mean <= 4.5)
                    SMVP_TINY(4);
                else if (mean <= 9.0)
                    SMVP_TINY(8);
                else if (mean <= 18.0)
                    SMVP_TINY(16);
                else
                    SMVP_TINY(32);
#undef SMVP_TINY
                SMVP_CUDA(cudaGetLastError());
                return (int)SMVP_OK;
            };
        if (A->rows > 0)
            rc = timed_loop(
                iters, ms_each, small,
                [&](cudaStream_t s) { return csr_mult_launch(A, xm, A->d_y.get(), nullptr, AXPBY_PLAIN, variant, s); }, multi);
        else if (ms_each)
            for (int it = 0; it < iters; it++)
                ms_each[it] = 0.0;
    }
    else
    {
        Event e0, e1;
        SMVP_CUDA(cudaEventCreate(out(e0)));
        SMVP_CUDA(cudaEventCreate(out(e1)));
        for (int it = 0; it < iters; it++)
        {
            float ms = 0.f;
            const bool first = it == 0, last = it == iters - 1;
            if ((first && upload_under_pass) || last)
            {
                SMVP_TRY(csr_mult_pipelined(A, (first && upload_under_pass) ? x_host : nullptr, last ? y_host : nullptr, &ms));
                y_copied = last;
            }
            else
            {
                cudaEventRecord(e0.get(), 0);
                SMVP_TRY(csr_mult_launch(A, xm, A->d_y.get(), nullptr, AXPBY_PLAIN, variant, 0));
                cudaEventRecord(e1.get(), 0);
                SMVP_CUDA(cudaEventSynchronize(e1.get()));
                cudaEventElapsedTime(&ms, e0.get(), e1.get());
            }
            if (ms_each)
                ms_each[it] = (double)ms;
        }
    }
    if (rc != SMVP_OK)
        return rc;
    if (A->rows > 0 && !y_copied)
        SMVP_CUDA(cudaMemcpy(y_host, A->d_y.get(), sizeof(double) * (size_t)A->rows, cudaMemcpyDeviceToHost));
    return SMVP_OK;
}

extern "C" int smvp_csr_info(const smvp_csr *A, smvp_csr_info_t *out)
{
    if (!A || !out)
        return SMVP_E_ARG;
    out->rows = A->rows;
    out->cols = A->cols;
    out->nnz = A->nnz;
    out->max_row_nnz = A->max_row_nnz;
    out->auto_variant = csr_resolve_variant(A, SMVP_CSR_AUTO);
    out->input_order = A->input_order;
    out->bytes_per_mult = 12 * A->nnz + 4 * ((int64_t)A->rows + 1) + 8 * (int64_t)A->cols + 8 * (int64_t)A->rows;
    out->device_bytes = A->device_bytes;
    out->launches_per_mult[SMVP_CSR_VECTOR] = 1;
    out->launches_per_mult[SMVP_CSR_MERGE] = A->pattern_state == 1 ? 1 : 2;
    out->launches_per_mult[SMVP_CSR_AUTO] = out->launches_per_mult[out->auto_variant];
    out->x_relabel = A->relabel_state;
    out->row_patterns = A->pattern_state == 1 ? A->pattern_count : A->pattern_state;
    out->value_bytes = A->pat_vbytes;
    return SMVP_OK;
}
