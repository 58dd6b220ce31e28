// csr_build.cu -- COO -> CSR on the device.  Replaces main-cli.c:336-365.
//
//   reference                                   here
//   qsort by (row, col)            :340         arrival-order check, else stable radix sort (coo_common.cu)
//   val[i], col_ind[i] = sorted[i] :350-351     gather through the sorting permutation
//   row_ptr from row changes       :353-364     row histogram + exclusive scan (== the slots the reference
//                                               writes; its unwritten slots, U3, get the intended value)
// Integer outputs are bit-exact against the reference's arrays; val is a copy (no arithmetic).
#include "common.cuh"

namespace smvp
{

__global__ void __launch_bounds__(256) gather_csr_kernel(const uint32_t *__restrict__ idx, const int32_t *__restrict__ col,
                                                         const double *__restrict__ val, int64_t nnz,
                                                         int32_t *__restrict__ col_out, double *__restrict__ val_out)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x)
    {
        const uint32_t s = idx[i];
        col_out[i] = col[s];
        val_out[i] = val[s];
    }
}

__global__ void set_last_kernel(int32_t *row_ptr, int32_t rows, int32_t nnz) { row_ptr[rows] = nnz; }

__global__ void __launch_bounds__(256) expand_rows_kernel(const int32_t *__restrict__ row_ptr, int32_t rows, int64_t nnz,
                                                          int32_t *__restrict__ row_of)
{
    // 8 consecutive nonzeros per thread: one binary search for the first, then a walk along row_ptr
    for (int64_t j0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8; j0 < nnz; j0 += (int64_t)gridDim.x * blockDim.x * 8)
    {
        int32_t lo = 0, hi = rows; // last row with row_ptr[row] <= j0
        while (hi - lo > 1)
        {
            const int32_t mid = lo + ((hi - lo) >> 1);
            if ((int64_t)__ldg(row_ptr + mid) <= j0)
                lo = mid;
            else
                hi = mid;
        }
        int32_t r = lo;
        const int64_t j1 = j0 + 8 < nnz ? j0 + 8 : nnz;
        for (int64_t j = j0; j < j1; j++)
        {
            while ((int64_t)__ldg(row_ptr + r + 1) <= j)
                r++;
            row_of[j] = r;
        }
    }
}

int csr_expand_rows(const int32_t *row_ptr, int32_t rows, int64_t nnz, int32_t *row_of, cudaStream_t s)
{
    if (nnz == 0)
        return SMVP_OK;
    const int64_t blocks = ceil_div64(nnz, 256 * 8), cap = (int64_t)device_props().sms * 16;
    SMVP_LAUNCH(expand_rows_kernel, (unsigned)(blocks < cap ? blocks : cap), 256, 0, s, row_ptr, rows, nnz, row_of);
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

void csr_release(smvp_csr *A)
{
    if (!A)
        return;
    csr_release(A->hot);
    csr_release(A->cold);
    cudaFree(A->row_ptr);
    cudaFree(A->col_ind);
    cudaFree(A->val);
    cudaFree(A->tile_row);
    cudaFree(A->head_val);
    cudaFree(A->carry_val);
    cudaFree(A->d_x);
    cudaFree(A->d_y);
    csr_pipe_release(A);
    csr_relabel_release(A);
    csr_pattern_release(A);
    delete A;
}

int csr_build_impl(const int32_t *d_row, const int32_t *d_col, const double *d_val, int32_t rows, int32_t cols,
                          int64_t nnz, smvp_csr *A, cudaStream_t s)
{
    int order = ORDER_ROW_COL;
    SMVP_TRY(coo_inspect(d_row, d_col, nnz, rows, cols, &order, s));
    A->input_order = order;

    SMVP_CUDA(dev_alloc(&A->row_ptr, (int64_t)rows + 1));
    SMVP_CUDA(dev_alloc(&A->col_ind, nnz));
    SMVP_CUDA(dev_alloc(&A->val, nnz));
    A->device_bytes = 4 * ((int64_t)rows + 1) + 12 * nnz;

    // row counts -> row_ptr by exclusive scan; row_ptr[rows] = nnz
    SMVP_TRY(histogram_i32(d_row, nnz, (uint32_t *)A->row_ptr, (int64_t)rows + 1, s));
    {
        DevTmp g_max;
        SMVP_CUDA(g_max.alloc<uint32_t>(1));
        uint32_t *d_max = g_max.as<uint32_t>();
        SMVP_TRY(max_u32((const uint32_t *)A->row_ptr, rows, d_max, s));
        uint32_t h = 0;
        SMVP_CUDA(cudaMemcpyAsync(&h, d_max, sizeof(h), cudaMemcpyDeviceToHost, s));
        SMVP_CUDA(cudaStreamSynchronize(s));
        A->max_row_nnz = (int32_t)h;
    }
    SMVP_TRY(exclusive_scan_u32((const uint32_t *)A->row_ptr, (uint32_t *)A->row_ptr, rows, nullptr, s));
    SMVP_LAUNCH(set_last_kernel, 1, 1, 0, s, A->row_ptr, rows, (int32_t)nnz);

    uint32_t *d_idx = nullptr;
    SMVP_TRY(coo_sort_index(d_row, d_col, nnz, rows, cols, order == ORDER_ROW_COL, order == ORDER_COL_ROW, &d_idx, s));
    DevTmp g_idx;
    g_idx.p = d_idx; // released on every return path below
    if (d_idx == nullptr)
    {
        if (nnz > 0)
        {
            SMVP_CUDA(cudaMemcpyAsync(A->col_ind, d_col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));
            SMVP_CUDA(cudaMemcpyAsync(A->val, d_val, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));
        }
    }
    else
    {
        int64_t blocks = ceil_div64(nnz, 256 * 4);
        const int64_t cap = (int64_t)device_props().sms * 16;
        if (blocks > cap)
            blocks = cap;
        SMVP_LAUNCH(gather_csr_kernel, (unsigned)blocks, 256, 0, s, (const uint32_t *)d_idx, d_col, d_val, nnz, A->col_ind,
                    A->val);
        SMVP_CUDA(cudaStreamSynchronize(s));
    }
    SMVP_CUDA(cudaStreamSynchronize(s));
    SMVP_CUDA(cudaGetLastError());

    // AUTO policy (see csr_mult.cu): regular, long rows stream best one sub-warp per row; everything
    // else (short rows, skew, empty rows) goes through the merge-path kernel.
    const double mean = rows > 0 ? (double)nnz / rows : 0.0;
    const bool tiny = nnz < (1 << 20);
    const bool skewed = A->max_row_nnz > 8.0 * (mean + 1.0); // memplus: vector 37 us, merge 13 us per SpMV
    // long regular rows: measured on dense-band matrices of ~1 B nnz (tools/sweep_vector.py, profiles/r02_logs/
    // r02_vector_sweep.log): 128 per row -- merge 1.97 ms, vector 2.33 ms; 512 per row -- vector 1.74 ms (7.09 TB/s, 88.6 % of
    // 8 TB/s), merge 2.59 ms (rows that span several warp tiles chain through the fix-up).  The crossover is put at 256.
    const bool regular_long = mean >= 256.0 && A->max_row_nnz <= 4.0 * mean + 32.0;
    A->auto_variant = ((tiny && !skewed) || regular_long) ? SMVP_CSR_VECTOR : SMVP_CSR_MERGE;
    return SMVP_OK;
}

} // namespace smvp

using namespace smvp;

extern "C" int smvp_csr_build_device(const int32_t *d_row, const int32_t *d_col, const double *d_val, int32_t rows,
                                     int32_t cols, int64_t nnz, smvp_csr **out)
{
    if (!out)
        return SMVP_E_ARG;
    *out = nullptr;
    if (rows < 0 || cols < 0 || nnz < 0 || (nnz > 0 && (!d_row || !d_col || !d_val)))
        return SMVP_E_ARG;
    if (nnz > 0x7fffffffLL - 8)
        return SMVP_E_TOOBIG;
    smvp_csr *A = new (std::nothrow) smvp_csr();
    if (!A)
        return SMVP_E_ALLOC;
    A->rows = rows;
    A->cols = cols;
    A->nnz = nnz;
    A->merge_cfg = -1;
    int rc = csr_build_impl(d_row, d_col, d_val, rows, cols, nnz, A, 0);
    if (rc != SMVP_OK)
    {
        csr_release(A);
        return rc;
    }
    *out = A;
    return SMVP_OK;
}

extern "C" int smvp_csr_build(const smvp_coo *coo, int32_t rows, int32_t cols, int64_t nnz, smvp_csr **out)
{
    if (!out)
        return SMVP_E_ARG;
    *out = nullptr;
    if (rows < 0 || cols < 0 || nnz < 0 || (nnz > 0 && !coo))
        return SMVP_E_ARG;
    if (nnz > 0x7fffffffLL - 8)
        return SMVP_E_TOOBIG;
    smvp_coo *d_aos = nullptr;
    int32_t *d_row = nullptr, *d_col = nullptr;
    double *d_val = nullptr;
    int rc = SMVP_OK;
    auto body = [&]() -> int {
        SMVP_CUDA(dev_alloc(&d_aos, nnz));
        SMVP_CUDA(dev_alloc(&d_row, nnz));
        SMVP_CUDA(dev_alloc(&d_col, nnz));
        SMVP_CUDA(dev_alloc(&d_val, nnz));
        if (nnz > 0)
            SMVP_CUDA(cudaMemcpy(d_aos, coo, sizeof(smvp_coo) * (size_t)nnz, cudaMemcpyHostToDevice));
        SMVP_TRY(coo_unzip(d_aos, nnz, d_row, d_col, d_val, 0));
        SMVP_CUDA(cudaFree(d_aos));
        d_aos = nullptr;
        return smvp_csr_build_device(d_row, d_col, d_val, rows, cols, nnz, out);
    };
    rc = body();
    cudaFree(d_aos);
    cudaFree(d_row);
    cudaFree(d_col);
    cudaFree(d_val);
    return rc;
}

// A^T from A's arrays: the entries of A, read in its (row, col) order, are the entries of A^T in (col, row) order, so
// coo_inspect reports ORDER_COL_ROW and the build's stable sort on the row key alone keeps each row of A^T in ascending
// column order.  A's natural col_ind is read whatever plan A uses (relabelled and split handles keep it).
extern "C" int smvp_csr_transpose(const smvp_csr *A, smvp_csr **out)
{
    if (!out)
        return SMVP_E_ARG;
    *out = nullptr;
    if (!A)
        return SMVP_E_ARG;
    smvp_csr *T = new (std::nothrow) smvp_csr();
    if (!T)
        return SMVP_E_ALLOC;
    T->rows = A->cols;
    T->cols = A->rows;
    T->nnz = A->nnz;
    T->merge_cfg = -1;
    auto body = [&]() -> int {
        DevTmp row_of;
        SMVP_CUDA(row_of.alloc<int32_t>(A->nnz));
        SMVP_TRY(csr_expand_rows(A->row_ptr, A->rows, A->nnz, row_of.as<int32_t>(), 0));
        return csr_build_impl(A->col_ind, row_of.as<int32_t>(), A->val, T->rows, T->cols, T->nnz, T, 0);
    };
    const int rc = body();
    if (rc != SMVP_OK)
    {
        csr_release(T);
        return rc;
    }
    *out = T;
    return SMVP_OK;
}

extern "C" void smvp_csr_free(smvp_csr *A) { smvp::csr_release(A); }

extern "C" int smvp_csr_export(const smvp_csr *A, int32_t *row_ptr, int32_t *col_ind, double *val)
{
    if (!A)
        return SMVP_E_ARG;
    if (row_ptr)
        SMVP_CUDA(cudaMemcpy(row_ptr, A->row_ptr, sizeof(int32_t) * ((size_t)A->rows + 1), cudaMemcpyDeviceToHost));
    if (col_ind && A->nnz > 0)
        SMVP_CUDA(cudaMemcpy(col_ind, A->col_ind, sizeof(int32_t) * (size_t)A->nnz, cudaMemcpyDeviceToHost));
    if (val && A->nnz > 0)
        SMVP_CUDA(cudaMemcpy(val, A->val, sizeof(double) * (size_t)A->nnz, cudaMemcpyDeviceToHost));
    return SMVP_OK;
}

extern "C" int smvp_csr_arrays_device(const smvp_csr *A, const int32_t **d_row_ptr, const int32_t **d_col_ind,
                                      const double **d_val)
{
    if (!A)
        return SMVP_E_ARG;
    if (d_row_ptr)
        *d_row_ptr = A->row_ptr;
    if (d_col_ind)
        *d_col_ind = A->col_ind;
    if (d_val)
        *d_val = A->val;
    return SMVP_OK;
}
