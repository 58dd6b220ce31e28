// tjds_build.cu -- COO -> TJDS (transposed jagged diagonal storage) on the device.
// Replaces main-cli.c:755-967.  Closed form of what the reference computes with three qsorts
// and two O(nnz*N) / O(M*N) linear searches (SURVEY.md 8a, a8):
//
//   reference                                             here
//   sort by (col,row), rank inside column   :766-826      arrival-order check / stable radix sort; rank = position - col_start[col]
//   txList[c] = {c, count_c - 1}            :845-862      column histogram
//   sort txList by (len desc, col asc)      :868          stable radix sort of the columns on key (maxcount - count)
//   col := slot of col (linear search)      :894-904      inverse permutation array
//   sort by (rank, slot)                    :926          position is known in closed form: start_pos[rank] + slot
//   start_pos[d] = first index of rank d    :944-967      L[d] = #{columns with count > d};  start_pos = exclusive scan(L)
//
// perm, start_pos, row_ind are bit-exact against the reference's arrays; val is a copy.
#include "common.cuh"

#include <new>

namespace smvp
{

__global__ void __launch_bounds__(256) tjds_colkey_kernel(const uint32_t *__restrict__ count, int32_t cols, uint32_t maxc,
                                                          uint32_t *__restrict__ key, uint32_t *__restrict__ idx)
{
    const int32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < cols)
    {
        key[c] = maxc - count[c]; // ascending key == descending count; the stable sort keeps col ascending on ties
        idx[c] = (uint32_t)c;
    }
}

__global__ void __launch_bounds__(256) tjds_perm_kernel(const uint32_t *__restrict__ sorted_key, const uint32_t *__restrict__ sorted_col,
                                                        int32_t cols, uint32_t maxc, int32_t *__restrict__ perm,
                                                        int32_t *__restrict__ slot_len, int32_t *__restrict__ slot_of)
{
    const int32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < cols)
    {
        const int32_t c = (int32_t)sorted_col[p];
        perm[p] = c;
        slot_len[p] = (int32_t)(maxc - sorted_key[p]);
        slot_of[c] = p;
    }
}

// L[d] = number of slots whose column holds more than d entries (slot_len is descending)
__global__ void __launch_bounds__(256) tjds_diag_len_kernel(const int32_t *__restrict__ slot_len, int32_t cols, int32_t ndiag,
                                                            uint32_t *__restrict__ L)
{
    const int32_t d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= ndiag)
        return;
    int32_t lo = 0, hi = cols; // first slot with slot_len <= d
    while (lo < hi)
    {
        const int32_t mid = (lo + hi) >> 1;
        if (slot_len[mid] > d)
            lo = mid + 1;
        else
            hi = mid;
    }
    L[d] = (uint32_t)lo;
}

__global__ void tjds_set_last_kernel(int32_t *start_pos, int32_t ndiag, int32_t nnz) { start_pos[ndiag] = nnz; }

// entry at sorted position i (column-major order) -> jagged diagonal `rank`, slot of its column
__global__ void __launch_bounds__(256) tjds_scatter_kernel(const uint32_t *__restrict__ idx, const int32_t *__restrict__ row,
                                                           const int32_t *__restrict__ col, const double *__restrict__ val,
                                                           int64_t nnz, const uint32_t *__restrict__ col_start,
                                                           const int32_t *__restrict__ slot_of, const int32_t *__restrict__ start_pos,
                                                           int32_t *__restrict__ row_ind, double *__restrict__ val_out)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x)
    {
        const int64_t src = idx ? (int64_t)idx[i] : i;
        const int32_t c = col[src];
        const int32_t rank = (int32_t)(i - (int64_t)col_start[c]);
        const int32_t dest = start_pos[rank] + slot_of[c];
        row_ind[dest] = row[src];
        val_out[dest] = val[src];
    }
}

// a new handle of rows x cols with nnz entries, built from COO arrays on the device; handed to *out on success
static int tjds_build_impl(const int32_t *d_row, const int32_t *d_col, const double *d_val, int32_t rows, int32_t cols,
                           int64_t nnz, smvp_tjds **out, cudaStream_t s)
{
    std::unique_ptr<smvp_tjds> A(new (std::nothrow) smvp_tjds());
    if (!A)
        return SMVP_E_ALLOC;
    A->rows = rows;
    A->cols = cols;
    A->nnz = nnz;
    int order = ORDER_ROW_COL;
    SMVP_TRY(coo_inspect(d_row, d_col, nnz, rows, cols, &order, s));
    A->input_order = order;

    const unsigned cblocks = (unsigned)ceil_div64(cols > 0 ? cols : 1, 256);
    // ---- column histogram, largest column = number of jagged diagonals
    DevPtr<uint32_t> count, col_start, d_max;
    SMVP_CUDA(dev_alloc(count, (int64_t)cols + 1));
    SMVP_CUDA(dev_alloc(col_start, (int64_t)cols + 1));
    SMVP_CUDA(dev_alloc(d_max, 1));
    SMVP_TRY(histogram_i32(d_col, nnz, count.get(), (int64_t)cols + 1, s));
    SMVP_TRY(max_u32(count.get(), cols, d_max.get(), s));
    uint32_t maxc = 0, count0 = 0;
    SMVP_CUDA(cudaMemcpyAsync(&maxc, d_max.get(), sizeof(maxc), cudaMemcpyDeviceToHost, s));
    if (cols > 0)
        SMVP_CUDA(cudaMemcpyAsync(&count0, count.get(), sizeof(count0), cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaStreamSynchronize(s));
    A->ndiag = (int32_t)maxc;
    A->ref_diag_limit = (int32_t)count0 + 1; // main-cli.c:865 (before the sort) + the `+ 1` of :1013

    // ---- perm: columns by count descending, column ascending on ties
    DevPtr<int32_t> slot_of;
    DevPtr<uint32_t> key_a, key_b, idx_a, idx_b;
    SMVP_CUDA(dev_alloc(A->perm, cols));
    SMVP_CUDA(dev_alloc(A->slot_len, cols));
    SMVP_CUDA(dev_alloc(A->x_perm, cols));
    SMVP_CUDA(dev_alloc(slot_of, cols));
    SMVP_CUDA(dev_alloc(key_a, cols));
    SMVP_CUDA(dev_alloc(key_b, cols));
    SMVP_CUDA(dev_alloc(idx_a, cols));
    SMVP_CUDA(dev_alloc(idx_b, cols));
    if (cols > 0)
    {
        SMVP_LAUNCH(tjds_colkey_kernel, cblocks, 256, 0, s, (const uint32_t *)count.get(), cols, maxc, key_a.get(), idx_a.get());
        uint32_t *rk = nullptr, *ri = nullptr;
        const int lo = 0, hi = bits_for(maxc + 1u);
        SMVP_TRY(radix_sort_pairs<uint32_t>(key_a.get(), idx_a.get(), key_b.get(), idx_b.get(), cols, &lo, &hi, 1, &rk, &ri, s));
        SMVP_LAUNCH(tjds_perm_kernel, cblocks, 256, 0, s, (const uint32_t *)rk, (const uint32_t *)ri, cols, maxc, A->perm.get(),
                    A->slot_len.get(), slot_of.get());
    }

    // ---- start_pos
    SMVP_CUDA(dev_alloc(A->start_pos, (int64_t)A->ndiag + 1));
    if (A->ndiag > 0)
    {
        uint32_t *start_pos = (uint32_t *)A->start_pos.get();
        SMVP_LAUNCH(tjds_diag_len_kernel, (unsigned)ceil_div64(A->ndiag, 256), 256, 0, s, (const int32_t *)A->slot_len.get(), cols,
                    A->ndiag, start_pos);
        SMVP_CUDA(cudaMemcpyAsync(&A->nslots, start_pos, sizeof(int32_t), cudaMemcpyDeviceToHost, s)); // L[0]
        SMVP_CUDA(cudaStreamSynchronize(s));
        SMVP_TRY(exclusive_scan_u32(start_pos, start_pos, A->ndiag, nullptr, s));
        int32_t last_start = 0;
        SMVP_CUDA(cudaMemcpyAsync(&last_start, start_pos + (A->ndiag - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        SMVP_CUDA(cudaStreamSynchronize(s));
        A->last_diag_len = (int32_t)(nnz - last_start);
    }
    else
    {
        A->nslots = 0;
        A->last_diag_len = 0;
    }
    SMVP_LAUNCH(tjds_set_last_kernel, 1, 1, 0, s, A->start_pos.get(), A->ndiag, (int32_t)nnz);

    // ---- rank inside the column needs column-major order
    DevPtr<uint32_t> d_idx;
    SMVP_TRY(exclusive_scan_u32(count.get(), col_start.get(), cols, nullptr, s));
    SMVP_TRY(coo_sort_index(d_col, d_row, nnz, cols, rows, order == ORDER_COL_ROW, order == ORDER_ROW_COL, &d_idx, s));
    SMVP_CUDA(dev_alloc(A->row_ind, nnz));
    SMVP_CUDA(dev_alloc(A->val, nnz));
    if (nnz > 0)
    {
        int64_t blocks = ceil_div64(nnz, 256 * 4);
        const int64_t cap = (int64_t)device_props().sms * 16;
        if (blocks > cap)
            blocks = cap;
        SMVP_LAUNCH(tjds_scatter_kernel, (unsigned)blocks, 256, 0, s, (const uint32_t *)d_idx.get(), d_row, d_col, d_val, nnz,
                    (const uint32_t *)col_start.get(), (const int32_t *)slot_of.get(), (const int32_t *)A->start_pos.get(),
                    A->row_ind.get(), A->val.get());
    }
    SMVP_CUDA(cudaStreamSynchronize(s));
    SMVP_CUDA(cudaGetLastError());
    A->device_bytes = 12 * nnz + 4 * ((int64_t)A->ndiag + 1) + 16 * (int64_t)cols;
    *out = A.release();
    return SMVP_OK;
}

} // namespace smvp

using namespace smvp;

extern "C" int smvp_tjds_build_device(const int32_t *d_row, const int32_t *d_col, const double *d_val, int32_t rows,
                                      int32_t cols, int64_t nnz, smvp_tjds **out)
{
    if (!out)
        return SMVP_E_ARG;
    *out = nullptr;
    if (rows < 0 || cols < 0 || nnz < 0 || (nnz > 0 && (!d_row || !d_col || !d_val)))
        return SMVP_E_ARG;
    if (nnz > 0x7fffffffLL - 1024)
        return SMVP_E_TOOBIG;
    return tjds_build_impl(d_row, d_col, d_val, rows, cols, nnz, out, 0);
}

extern "C" int smvp_tjds_build(const smvp_coo *coo, int32_t rows, int32_t cols, int64_t nnz, smvp_tjds **out)
{
    if (!out)
        return SMVP_E_ARG;
    *out = nullptr;
    if (rows < 0 || cols < 0 || nnz < 0 || (nnz > 0 && !coo))
        return SMVP_E_ARG;
    if (nnz > 0x7fffffffLL - 1024)
        return SMVP_E_TOOBIG;
    DevPtr<smvp_coo> d_aos;
    DevPtr<int32_t> d_row, d_col;
    DevPtr<double> d_val;
    SMVP_CUDA(dev_alloc(d_aos, nnz));
    SMVP_CUDA(dev_alloc(d_row, nnz));
    SMVP_CUDA(dev_alloc(d_col, nnz));
    SMVP_CUDA(dev_alloc(d_val, nnz));
    if (nnz > 0)
        SMVP_CUDA(cudaMemcpy(d_aos.get(), coo, sizeof(smvp_coo) * (size_t)nnz, cudaMemcpyHostToDevice));
    SMVP_TRY(coo_unzip(d_aos.get(), nnz, d_row.get(), d_col.get(), d_val.get(), 0));
    d_aos.reset(); // before the build: lowers the peak
    return smvp_tjds_build_device(d_row.get(), d_col.get(), d_val.get(), rows, cols, nnz, out);
}

extern "C" void smvp_tjds_free(smvp_tjds *A) { delete A; }

extern "C" int smvp_tjds_export(const smvp_tjds *A, int32_t *perm, int32_t *start_pos, int32_t *row_ind, double *val)
{
    if (!A)
        return SMVP_E_ARG;
    if (perm && A->cols > 0)
        SMVP_CUDA(cudaMemcpy(perm, A->perm.get(), sizeof(int32_t) * (size_t)A->cols, cudaMemcpyDeviceToHost));
    if (start_pos)
        SMVP_CUDA(cudaMemcpy(start_pos, A->start_pos.get(), sizeof(int32_t) * ((size_t)A->ndiag + 1), cudaMemcpyDeviceToHost));
    if (row_ind && A->nnz > 0)
        SMVP_CUDA(cudaMemcpy(row_ind, A->row_ind.get(), sizeof(int32_t) * (size_t)A->nnz, cudaMemcpyDeviceToHost));
    if (val && A->nnz > 0)
        SMVP_CUDA(cudaMemcpy(val, A->val.get(), sizeof(double) * (size_t)A->nnz, cudaMemcpyDeviceToHost));
    return SMVP_OK;
}
