// update.cu -- new values on the entries a CSR or TJDS handle already stores (smvp_csr_update_values*,
// smvp_tjds_update_values*): the way Newton steps, implicit time steps, continuation and shifted systems A - sigma I
// change a matrix whose sparsity stays put.  Every plan that depends only on where the entries are (merge tiles, row
// patterns, relabelling, TJDS walk and segment table, pipelined host plan, transposed and dot scratch) and the declared
// x stay; the two decisions that depend on the values are made again: the value width of the CSR row-pattern plan
// (csr_pattern_values) and the row bounds of the deterministic TJDS variants (tjds_update_det).
//
// One thread per list entry locates its entry in the handle:
//   CSR   binary search for col in col_ind[row_ptr[row], row_ptr[row+1]) -- columns ascend within a row in every handle
//         (the builder's sort, smvp_csr_transpose);
//   TJDS  slot q of the column (a temporary inverse of perm, cols int32), then a binary search for row along the column,
//         row_ind[start_pos[k] + q] for k < slot_len[q] -- rows ascend with the jagged diagonal k.
// Two passes of the same kernel: the first only raises range and pattern flags, which the host reads once; the second,
// run only when the whole list is valid, writes.  The positions are located twice rather than kept, so no temporary grows
// with the list's length.  Relabelled handles need nothing extra: col_rel and row_rel sit beside the
// entries they index.
#include "common.cuh"

namespace smvp
{

constexpr int32_t UPD_RANGE = 1, UPD_PATTERN = 2;

// WRITE = false: flags |= UPD_RANGE / UPD_PATTERN for a coordinate outside the matrix / a pair the handle does not store.
// WRITE = true: the list is valid; val[position of entry i] = u_val[i].
template <bool WRITE>
__global__ void __launch_bounds__(256) csr_update_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col_ind,
                                                         int32_t rows, int32_t cols, const int32_t *__restrict__ u_row,
                                                         const int32_t *__restrict__ u_col, const double *__restrict__ u_val, int64_t n,
                                                         double *__restrict__ val, int32_t *__restrict__ flags)
{
    int32_t f = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t r = __ldg(u_row + i), c = __ldg(u_col + i);
        if ((uint32_t)r >= (uint32_t)rows || (uint32_t)c >= (uint32_t)cols)
        {
            f |= UPD_RANGE;
            continue;
        }
        int32_t lo = __ldg(row_ptr + r), hi = __ldg(row_ptr + r + 1);
        const int32_t end = hi;
        while (lo < hi) // first position whose column is >= c
        {
            const int32_t mid = lo + ((hi - lo) >> 1);
            if (__ldg(col_ind + mid) < c)
                lo = mid + 1;
            else
                hi = mid;
        }
        if (lo == end || __ldg(col_ind + lo) != c)
            f |= UPD_PATTERN;
        else if (WRITE)
            val[lo] = __ldg(u_val + i);
    }
    if (!WRITE)
    {
        f = (int32_t)__reduce_or_sync(0xffffffffu, (unsigned)f);
        if ((threadIdx.x & 31) == 0 && f)
            atomicOr(flags, f);
    }
}

// slot_of[perm[q]] = q: the slot of every column
__global__ void __launch_bounds__(256) tjds_slot_of_kernel(const int32_t *__restrict__ perm, int32_t cols, int32_t *__restrict__ slot_of)
{
    const int32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < cols)
        slot_of[perm[q]] = q;
}

template <bool WRITE>
__global__ void __launch_bounds__(256) tjds_update_kernel(const int32_t *__restrict__ slot_of, const int32_t *__restrict__ slot_len,
                                                          const int32_t *__restrict__ start_pos, const int32_t *__restrict__ row_ind,
                                                          int32_t rows, int32_t cols, const int32_t *__restrict__ u_row,
                                                          const int32_t *__restrict__ u_col, const double *__restrict__ u_val, int64_t n,
                                                          double *__restrict__ val, int32_t *__restrict__ flags)
{
    int32_t f = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t r = __ldg(u_row + i), c = __ldg(u_col + i);
        if ((uint32_t)r >= (uint32_t)rows || (uint32_t)c >= (uint32_t)cols)
        {
            f |= UPD_RANGE;
            continue;
        }
        const int32_t q = __ldg(slot_of + c), len = __ldg(slot_len + q);
        int32_t lo = 0, hi = len;
        while (lo < hi) // first diagonal whose row is >= r
        {
            const int32_t mid = lo + ((hi - lo) >> 1);
            if (__ldg(row_ind + __ldg(start_pos + mid) + q) < r)
                lo = mid + 1;
            else
                hi = mid;
        }
        const int32_t j = lo < len ? __ldg(start_pos + lo) + q : -1;
        if (j < 0 || __ldg(row_ind + j) != r)
            f |= UPD_PATTERN;
        else if (WRITE)
            val[j] = __ldg(u_val + i);
    }
    if (!WRITE)
    {
        f = (int32_t)__reduce_or_sync(0xffffffffu, (unsigned)f);
        if ((threadIdx.x & 31) == 0 && f)
            atomicOr(flags, f);
    }
}

static unsigned update_grid(int64_t n)
{
    const int64_t blocks = ceil_div64(n, 256 * 4), cap = (int64_t)device_props().sms * 16;
    return (unsigned)(blocks < cap ? blocks : cap);
}

// The check pass (launched by `check`, into the zeroed device word flags) read back: SMVP_OK, SMVP_E_RANGE or
// SMVP_E_PATTERN.  Synchronous.
template <typename F>
static int update_check(int32_t *flags, cudaStream_t s, F &&check)
{
    SMVP_CUDA(cudaMemsetAsync(flags, 0, sizeof(int32_t), s));
    check();
    SMVP_CUDA(cudaGetLastError());
    int32_t h = 0;
    SMVP_CUDA(cudaMemcpyAsync(&h, flags, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaStreamSynchronize(s));
    return (h & UPD_RANGE) ? SMVP_E_RANGE : (h & UPD_PATTERN) ? SMVP_E_PATTERN : SMVP_OK;
}

static int csr_update(smvp_csr *A, const int32_t *d_row, const int32_t *d_col, const double *d_val, int64_t n, cudaStream_t s)
{
    const unsigned grid = update_grid(n);
    DevPtr<int32_t> flags;
    SMVP_CUDA(dev_alloc(flags, 1));
    SMVP_TRY(update_check(flags.get(), s, [&] {
        SMVP_LAUNCH(csr_update_kernel<false>, grid, 256, 0, s, (const int32_t *)A->row_ptr.get(), (const int32_t *)A->col_ind.get(),
                    A->rows, A->cols, d_row, d_col, d_val, n, A->val.get(), flags.get());
    }));
    SMVP_LAUNCH(csr_update_kernel<true>, grid, 256, 0, s, (const int32_t *)A->row_ptr.get(), (const int32_t *)A->col_ind.get(), A->rows,
                A->cols, d_row, d_col, d_val, n, A->val.get(), flags.get());
    SMVP_CUDA(cudaGetLastError()); // a launch that failed wrote nothing
    if (A->pattern_state == 1)
        return csr_pattern_values(A, s); // synchronises; a failure leaves the width undecided
    SMVP_CUDA(cudaStreamSynchronize(s));
    return SMVP_OK;
}

static int tjds_update(smvp_tjds *A, const int32_t *d_row, const int32_t *d_col, const double *d_val, int64_t n, cudaStream_t s)
{
    const unsigned grid = update_grid(n);
    DevPtr<int32_t> flags, slot_of;
    SMVP_CUDA(dev_alloc(flags, 1));
    SMVP_CUDA(dev_alloc(slot_of, A->cols));
    if (A->cols > 0)
        SMVP_LAUNCH(tjds_slot_of_kernel, (unsigned)ceil_div64(A->cols, 256), 256, 0, s, (const int32_t *)A->perm.get(), A->cols,
                    slot_of.get());
    SMVP_TRY(update_check(flags.get(), s, [&] {
        SMVP_LAUNCH(tjds_update_kernel<false>, grid, 256, 0, s, (const int32_t *)slot_of.get(), (const int32_t *)A->slot_len.get(),
                    (const int32_t *)A->start_pos.get(), (const int32_t *)A->row_ind.get(), A->rows, A->cols, d_row, d_col, d_val, n,
                    A->val.get(), flags.get());
    }));
    SMVP_LAUNCH(tjds_update_kernel<true>, grid, 256, 0, s, (const int32_t *)slot_of.get(), (const int32_t *)A->slot_len.get(),
                (const int32_t *)A->start_pos.get(), (const int32_t *)A->row_ind.get(), A->rows, A->cols, d_row, d_col, d_val, n,
                A->val.get(), flags.get());
    SMVP_CUDA(cudaGetLastError());
    SMVP_TRY(tjds_update_det(A, s)); // synchronises when the deterministic state exists; a failure drops that state
    SMVP_CUDA(cudaStreamSynchronize(s));
    return SMVP_OK;
}

// The host variants stage the list on the device as the builders do: one copy of the 16-byte entries, then unzipped.
template <typename H, typename F>
static int update_from_host(H *A, const smvp_coo *coo, int64_t n, F &&update_device)
{
    if (!A || n < 0 || (n > 0 && !coo))
        return SMVP_E_ARG;
    if (n == 0)
        return SMVP_OK;
    DevPtr<smvp_coo> d_aos;
    DevPtr<int32_t> d_row, d_col;
    DevPtr<double> d_val;
    SMVP_CUDA(dev_alloc(d_aos, n));
    SMVP_CUDA(dev_alloc(d_row, n));
    SMVP_CUDA(dev_alloc(d_col, n));
    SMVP_CUDA(dev_alloc(d_val, n));
    SMVP_CUDA(cudaMemcpy(d_aos.get(), coo, sizeof(smvp_coo) * (size_t)n, cudaMemcpyHostToDevice));
    SMVP_TRY(coo_unzip(d_aos.get(), n, d_row.get(), d_col.get(), d_val.get(), 0));
    d_aos.reset();
    return update_device(A, d_row.get(), d_col.get(), d_val.get(), n, nullptr);
}

} // namespace smvp

using namespace smvp;

extern "C" int smvp_csr_update_values_device(smvp_csr *A, const int32_t *d_row, const int32_t *d_col, const double *d_val, int64_t n,
                                             void *stream)
{
    if (!A || n < 0 || (n > 0 && (!d_row || !d_col || !d_val)))
        return SMVP_E_ARG;
    if (n == 0)
        return SMVP_OK;
    return csr_update(A, d_row, d_col, d_val, n, (cudaStream_t)stream);
}

extern "C" int smvp_tjds_update_values_device(smvp_tjds *A, const int32_t *d_row, const int32_t *d_col, const double *d_val, int64_t n,
                                              void *stream)
{
    if (!A || n < 0 || (n > 0 && (!d_row || !d_col || !d_val)))
        return SMVP_E_ARG;
    if (n == 0)
        return SMVP_OK;
    return tjds_update(A, d_row, d_col, d_val, n, (cudaStream_t)stream);
}

extern "C" int smvp_csr_update_values(smvp_csr *A, const smvp_coo *coo, int64_t n)
{
    return update_from_host(A, coo, n, smvp_csr_update_values_device);
}

extern "C" int smvp_tjds_update_values(smvp_tjds *A, const smvp_coo *coo, int64_t n)
{
    return update_from_host(A, coo, n, smvp_tjds_update_values_device);
}
