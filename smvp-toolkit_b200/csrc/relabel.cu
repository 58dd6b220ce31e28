// relabel.cu -- popularity relabelling of an index space: the COLUMNS of a CSR handle (the gather side) and the ROWS
// of a TJDS handle (the scatter side).  A multiply-side plan: the arrays the reference defines (CSRData / TJDSData,
// main-cli.c:61-75) stay untouched and bit-exact.
//
// Why: the CSR loop (main-cli.c:410-416) gathers x[col_ind[j]].  On a power-law matrix whose x does not fit
// the 126 MB L2 (R-MAT scale 26: 537 MB) half of those 8-byte gathers miss L2 and each miss moves a 32-byte
// DRAM sector: ncu counted 30.6 GB of DRAM traffic for 14.1 GB of algorithmic bytes
// (profiles/r01_csr_merge_warp_rmat26.txt).  The gathers are far from uniform, though: a few million columns
// receive most of them -- but they are scattered over the whole index range, so they share their sectors and
// cache lines with cold columns.  The TJDS loop (main-cli.c:1013-1020) has the mirror problem on y[row_ind[j]].
//
// What: number the columns by descending entry count (ties keep column order) -- exactly the permutation
// the TJDS format defines (main-cli.c:868, txtable_comparator_len :209-223) -- and keep
//     col_rel[j] = rank[col_ind[j]]        one extra int32 per nonzero, read INSTEAD of col_ind by the kernels
//     x_order[p] = column with rank p      x_rel[p] = x[x_order[p]] is formed once per x
// The hot columns become one dense prefix of x_rel that stays resident in L2 (and partly in L1).  Entries keep
// their order inside each row, so every row is summed in exactly the order it was before: y is bit-identical
// with and without the plan.  For TJDS: row_rel[j] = rank[row_ind[j]], sums land in rank order, one pass per
// multiply puts them back (y[r] = y_rel[row_rank[r]]).
//
// When (AUTO): at least RELABEL_MIN_COLS indices of the space actually occur in the handle, and the RELABEL_HOT_COLS most
// popular ones hold at least half of the nonzeros and at least twice their fair share AMONG THE OCCURRING ONES (round 2:
// "four times" could never hold for the row block of one GPU out of 4 or 8 of an R-MAT matrix -- it touches 12 - 20 Mi
// columns, so the fair share of 4 Mi of them is already 0.2 - 0.35 -- and those blocks lost their relabelling).  Banded and uniform matrices fail
// the test and keep their natural (already local, or hopeless) order.  SMVP_CSR_RELABEL / SMVP_TJDS_RELABEL = 1 / 0
// force it on / off.
#include "common.cuh"

namespace smvp
{

// x of 64 MB and more: beyond what L2 keeps next to the matrix streams; 32 MB of x: the part expected to stay L2-resident.
// SMVP_RELABEL_MIN_COLS / SMVP_RELABEL_HOT_COLS (entries) scale the AUTO test down so that it can be exercised on small
// matrices (tests); they do not touch the cache hints of the multiply.
static int64_t relabel_min_cols()
{
    const int v = env_int("SMVP_RELABEL_MIN_COLS", 0, 0, INT32_MAX);
    return v > 0 ? v : 8 << 20;
}
static int64_t relabel_hot_cols()
{
    const int v = env_int("SMVP_RELABEL_HOT_COLS", 0, 0, INT32_MAX);
    return v > 0 ? v : 4 << 20;
}

__global__ void __launch_bounds__(256) relabel_key_kernel(const uint32_t *__restrict__ count, int32_t cols, uint32_t maxc,
                                                          uint32_t *__restrict__ key, uint32_t *__restrict__ idx)
{
    const int32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < cols)
    {
        key[c] = maxc - count[c]; // ascending key == descending count; the stable sort keeps col ascending on ties
        idx[c] = (uint32_t)c;
    }
}

// nonzeros held by the first k columns of the sorted order
__global__ void __launch_bounds__(256) relabel_cover_kernel(const uint32_t *__restrict__ sorted_key, int32_t k, uint32_t maxc,
                                                            unsigned long long *__restrict__ sum)
{
    unsigned long long t = 0;
    for (int32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < k; p += gridDim.x * blockDim.x)
        t += maxc - sorted_key[p];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        t += __shfl_xor_sync(0xffffffffu, t, o);
    if ((threadIdx.x & 31) == 0 && t)
        atomicAdd(sum, t);
}

// number of indices that occur at all: sorted_key ascends, an index that never occurs has key == maxc
__global__ void relabel_touched_kernel(const uint32_t *__restrict__ sorted_key, int32_t n, uint32_t maxc, int32_t *__restrict__ touched)
{
    int32_t lo = 0, hi = n;
    while (lo < hi)
    {
        const int32_t mid = lo + ((hi - lo) >> 1);
        if (sorted_key[mid] < maxc)
            lo = mid + 1;
        else
            hi = mid;
    }
    *touched = lo;
}

__global__ void __launch_bounds__(256) relabel_rank_kernel(const uint32_t *__restrict__ sorted_col, int32_t cols,
                                                           int32_t *__restrict__ x_order, int32_t *__restrict__ rank)
{
    const int32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < cols)
    {
        const int32_t c = (int32_t)sorted_col[p];
        x_order[p] = c;
        rank[c] = p;
    }
}

__global__ void __launch_bounds__(256) relabel_cols_kernel(const int32_t *__restrict__ col_ind, int64_t nnz,
                                                           const int32_t *__restrict__ rank, int32_t *__restrict__ col_rel)
{
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nnz; j += (int64_t)gridDim.x * blockDim.x)
        col_rel[j] = __ldg(rank + __ldg(col_ind + j));
}

__global__ void __launch_bounds__(256) relabel_permute_x_kernel(const double *__restrict__ x, const int32_t *__restrict__ x_order,
                                                                int32_t cols, double *__restrict__ x_rel)
{
    for (int32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < cols; p += gridDim.x * blockDim.x)
        x_rel[p] = __ldg(x + __ldg(x_order + p));
}

// Popularity order of an index space: d_idx[nnz] holds indices in [0, n).  forced > 0 builds the order whatever the
// distribution; forced == 0 builds it only when the index space is large and skewed enough (see the header).
// On success with *use = 1: (*d_order)[p] = index with rank p, (*d_rank)[i] = rank of index i (caller frees both).
// Synchronous.
int popularity_plan(const int32_t *d_idx, int64_t nnz, int32_t n, int forced, double min_ratio, int32_t **d_order, int32_t **d_rank,
                    int *use, cudaStream_t s)
{
    *use = 0;
    *d_order = *d_rank = nullptr;
    if (forced < 0 || nnz == 0 || n == 0 || (forced == 0 && n < relabel_min_cols()))
        return SMVP_OK;
    uint32_t *count = nullptr, *d_max = nullptr, *key_a = nullptr, *key_b = nullptr, *idx_a = nullptr, *idx_b = nullptr;
    unsigned long long *d_cover = nullptr;
    int32_t *order = nullptr, *rank = nullptr;
    auto cleanup = [&]() {
        cudaFree(count);
        cudaFree(d_max);
        cudaFree(key_a);
        cudaFree(key_b);
        cudaFree(idx_a);
        cudaFree(idx_b);
        cudaFree(d_cover);
    };
    auto body = [&]() -> int {
        const unsigned cblocks = (unsigned)ceil_div64(n, 256);
        SMVP_CUDA(dev_alloc(&count, (int64_t)n + 1));
        SMVP_CUDA(dev_alloc(&d_max, 1));
        SMVP_CUDA(dev_alloc(&d_cover, 1));
        SMVP_CUDA(dev_alloc(&key_a, n));
        SMVP_CUDA(dev_alloc(&key_b, n));
        SMVP_CUDA(dev_alloc(&idx_a, n));
        SMVP_CUDA(dev_alloc(&idx_b, n));
        SMVP_TRY(histogram_i32(d_idx, nnz, count, (int64_t)n + 1, s));
        SMVP_TRY(max_u32(count, n, d_max, s));
        uint32_t maxc = 0;
        SMVP_CUDA(cudaMemcpyAsync(&maxc, d_max, sizeof(maxc), cudaMemcpyDeviceToHost, s));
        SMVP_CUDA(cudaStreamSynchronize(s));
        SMVP_LAUNCH(relabel_key_kernel, cblocks, 256, 0, s, (const uint32_t *)count, n, maxc, key_a, idx_a);
        uint32_t *rk = nullptr, *ri = nullptr;
        const int lo = 0, hi = bits_for(maxc + 1u);
        SMVP_TRY(radix_sort_pairs<uint32_t>(key_a, idx_a, key_b, idx_b, n, &lo, &hi, 1, &rk, &ri, s));
        if (forced == 0)
        {
            // The test runs over the indices the handle actually TOUCHES, not over the whole index space: a row block
            // of a banded matrix (the shard of one GPU out of 8) reads a 1/8 window of x, and measured against all n
            // columns that window looked like a hot set holding every nonzero (round-1 misfire at 8 GPUs).
            int32_t touched = 0;
            SMVP_LAUNCH(relabel_touched_kernel, 1, 1, 0, s, (const uint32_t *)rk, n, maxc, (int32_t *)d_max);
            SMVP_CUDA(cudaMemcpyAsync(&touched, d_max, sizeof(touched), cudaMemcpyDeviceToHost, s));
            SMVP_CUDA(cudaStreamSynchronize(s));
            if (touched < relabel_min_cols())
                return SMVP_OK; // what is gathered fits L2 next to the streams
            const int32_t k = (int32_t)(touched < relabel_hot_cols() ? touched : relabel_hot_cols());
            SMVP_CUDA(cudaMemsetAsync(d_cover, 0, sizeof(unsigned long long), s));
            SMVP_LAUNCH(relabel_cover_kernel, (unsigned)device_props().sms * 8, 256, 0, s, (const uint32_t *)rk, k, maxc, d_cover);
            unsigned long long cover = 0;
            SMVP_CUDA(cudaMemcpyAsync(&cover, d_cover, sizeof(cover), cudaMemcpyDeviceToHost, s));
            SMVP_CUDA(cudaStreamSynchronize(s));
            const double share = (double)cover / (double)nnz, fair = (double)k / (double)touched;
            // skewed enough: the hot set holds most of the gathers AND at least twice what a flat distribution over the
            // touched columns would give it (a banded block is exactly flat: share == fair)
            // (min_ratio: 2 for the CSR gathers; 4 for the TJDS scatter, where the plan gains 5 % on the whole R-MAT
            // matrix and LOSES 20 % on the column block of one GPU out of 8 -- profiles/r02_logs/r02_bench_n8_final.json
            // before / after -- so only a pronounced skew selects it)
            if (!(share >= 0.5 && share >= min_ratio * fair))
                return SMVP_OK;
        }
        SMVP_CUDA(dev_alloc(&order, n));
        SMVP_CUDA(dev_alloc(&rank, n));
        SMVP_LAUNCH(relabel_rank_kernel, cblocks, 256, 0, s, (const uint32_t *)ri, n, order, rank);
        SMVP_CUDA(cudaStreamSynchronize(s));
        SMVP_CUDA(cudaGetLastError());
        *use = 1;
        return SMVP_OK;
    };
    const int rc = body();
    cleanup();
    if (rc != SMVP_OK || !*use)
    {
        cudaFree(order);
        cudaFree(rank);
        *use = 0;
        return rc;
    }
    *d_order = order;
    *d_rank = rank;
    return SMVP_OK;
}

// out[j] = rank[idx[j]] (asynchronous on s)
int relabel_indices(const int32_t *d_idx, int64_t nnz, const int32_t *d_rank, int32_t *d_out, cudaStream_t s)
{
    if (nnz > 0)
    {
        int64_t blocks = ceil_div64(nnz, 256 * 4);
        const int64_t cap = (int64_t)device_props().sms * 16;
        SMVP_LAUNCH(relabel_cols_kernel, (unsigned)(blocks < cap ? blocks : cap), 256, 0, s, d_idx, nnz, d_rank, d_out);
        SMVP_CUDA(cudaGetLastError());
    }
    return SMVP_OK;
}

// decides (once per handle) and, if the plan is worth it, builds col_rel / x_order / x_rel.  Synchronous.
int csr_relabel_plan(smvp_csr *A, cudaStream_t s)
{
    if (A->relabel_state != 0)
        return SMVP_OK;
    int use = 0;
    int32_t *order = nullptr, *rank = nullptr;
    SMVP_TRY(popularity_plan(A->col_ind, A->nnz, A->cols, env_tristate("SMVP_CSR_RELABEL"), 2.0, &order, &rank, &use, s));
    if (!use)
    {
        A->relabel_state = -1;
        return SMVP_OK;
    }
    A->x_order = order;
    auto body = [&]() -> int {
        SMVP_CUDA(dev_alloc(&A->x_rel, A->cols));
        SMVP_CUDA(dev_alloc(&A->col_rel, A->nnz));
        SMVP_TRY(relabel_indices(A->col_ind, A->nnz, rank, A->col_rel, s));
        SMVP_CUDA(cudaStreamSynchronize(s));
        return SMVP_OK;
    };
    const int rc = body();
    cudaFree(rank);
    if (rc != SMVP_OK)
    {
        csr_relabel_release(A);
        return rc;
    }
    A->device_bytes += 4 * A->nnz + 12 * (int64_t)A->cols;
    A->relabel_state = 1;
    return SMVP_OK;
}

// the same for the ROWS of a TJDS handle: the multiply scatters into y[row_ind[j]], and on a power-law matrix whose
// y exceeds L2 those read-modify-writes miss the way the CSR gathers do.  row_rel replaces row_ind in the kernels,
// the sums land in rank order and one last pass puts them back: y[r] = y_rel[row_rank[r]].
int tjds_relabel_plan(smvp_tjds *A, cudaStream_t s)
{
    if (A->relabel_state != 0)
        return SMVP_OK;
    int use = 0;
    int32_t *order = nullptr, *rank = nullptr;
    SMVP_TRY(popularity_plan(A->row_ind, A->nnz, A->rows, env_tristate("SMVP_TJDS_RELABEL"), 4.0, &order, &rank, &use, s));
    if (!use)
    {
        A->relabel_state = -1;
        return SMVP_OK;
    }
    cudaFree(order);
    A->row_rank = rank;
    auto body = [&]() -> int {
        SMVP_CUDA(dev_alloc(&A->y_rel, A->rows));
        SMVP_CUDA(dev_alloc(&A->row_rel, A->nnz));
        SMVP_TRY(relabel_indices(A->row_ind, A->nnz, rank, A->row_rel, s));
        SMVP_CUDA(cudaStreamSynchronize(s));
        return SMVP_OK;
    };
    const int rc = body();
    if (rc != SMVP_OK)
    {
        tjds_relabel_release(A);
        return rc;
    }
    A->device_bytes += 4 * A->nnz + 12 * (int64_t)A->rows;
    A->relabel_state = 1;
    return SMVP_OK;
}

void tjds_relabel_release(smvp_tjds *A)
{
    cudaFree(A->row_rank);
    cudaFree(A->row_rel);
    cudaFree(A->y_rel);
    A->row_rank = A->row_rel = nullptr;
    A->y_rel = nullptr;
}

// x_rel = x in rank order (asynchronous on s)
int csr_relabel_x(smvp_csr *A, const double *d_x, cudaStream_t s)
{
    int64_t blocks = ceil_div64(A->cols, 256 * 4);
    const int64_t cap = (int64_t)device_props().sms * 8;
    SMVP_LAUNCH(relabel_permute_x_kernel, (unsigned)(blocks < cap ? blocks : cap), 256, 0, s, d_x, (const int32_t *)A->x_order, A->cols,
                A->x_rel);
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

void csr_relabel_release(smvp_csr *A)
{
    cudaFree(A->x_order);
    cudaFree(A->x_rel);
    cudaFree(A->col_rel);
    A->x_order = A->col_rel = nullptr;
    A->x_rel = nullptr;
}

} // namespace smvp
