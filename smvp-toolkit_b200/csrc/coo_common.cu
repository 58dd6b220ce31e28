// coo_common.cu -- what both builders do to the COO list before they diverge: range validation,
// arrival-order detection, AoS->SoA split and the sorting permutation.
//
// The reference always qsorts (main-cli.c:340 by (row,col); :766 by (col,row)).  Matrix Market files
// arrive (col,row)-sorted and the synthetic generators emit (row,col)-sorted lists, so most sorts here
// collapse to nothing or to a stable sort on the major key alone; the result is the same total order.
#include "common.cuh"

namespace smvp
{

// flags[0] = out-of-range seen, flags[1] = NOT strictly (row,col)-increasing, flags[2] = NOT strictly (col,row)-increasing
__global__ void __launch_bounds__(256) coo_inspect_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col,
                                                          int64_t nnz, int32_t rows, int32_t cols, int *__restrict__ flags)
{
    bool bad = false, not_rc = false, not_cr = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t r = row[i], c = col[i];
        if (r < 0 || r >= rows || c < 0 || c >= cols)
            bad = true;
        if (i > 0)
        {
            const int32_t pr = row[i - 1], pc = col[i - 1];
            if (!(pr < r || (pr == r && pc < c)))
                not_rc = true;
            if (!(pc < c || (pc == c && pr < r)))
                not_cr = true;
        }
    }
    if (bad)
        flags[0] = 1;
    if (not_rc)
        flags[1] = 1;
    if (not_cr)
        flags[2] = 1;
}

int coo_inspect(const int32_t *d_row, const int32_t *d_col, int64_t nnz, int32_t rows, int32_t cols, int *order,
                cudaStream_t s)
{
    *order = ORDER_ROW_COL;
    if (nnz == 0)
        return SMVP_OK;
    DevPtr<int> flags;
    SMVP_CUDA(dev_alloc(flags, 4));
    SMVP_CUDA(cudaMemsetAsync(flags.get(), 0, 4 * sizeof(int), s));
    int64_t blocks = ceil_div64(nnz, 256 * 4);
    const int64_t cap = (int64_t)device_props().sms * 16;
    if (blocks > cap)
        blocks = cap;
    SMVP_LAUNCH(coo_inspect_kernel, (unsigned)blocks, 256, 0, s, d_row, d_col, nnz, rows, cols, flags.get());
    int h[4] = {0, 0, 0, 0};
    SMVP_CUDA(cudaMemcpyAsync(h, flags.get(), sizeof(h), cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaStreamSynchronize(s));
    if (h[0])
        return SMVP_E_RANGE;
    *order = !h[1] ? ORDER_ROW_COL : (!h[2] ? ORDER_COL_ROW : ORDER_NONE);
    return SMVP_OK;
}

__global__ void __launch_bounds__(256) coo_unzip_kernel(const smvp_coo *__restrict__ aos, int64_t nnz, int32_t *__restrict__ row,
                                                        int32_t *__restrict__ col, double *__restrict__ val)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (int64_t)gridDim.x * blockDim.x)
    {
        // one 16-byte load per entry: {row, col, val}
        const int4 e = *reinterpret_cast<const int4 *>(aos + i);
        row[i] = e.x;
        col[i] = e.y;
        val[i] = __hiloint2double(e.w, e.z);
    }
}

int coo_unzip(const smvp_coo *d_aos, int64_t nnz, int32_t *d_row, int32_t *d_col, double *d_val, cudaStream_t s)
{
    if (nnz == 0)
        return SMVP_OK;
    int64_t blocks = ceil_div64(nnz, 256 * 4);
    const int64_t cap = (int64_t)device_props().sms * 16;
    if (blocks > cap)
        blocks = cap;
    SMVP_LAUNCH(coo_unzip_kernel, (unsigned)blocks, 256, 0, s, d_aos, nnz, d_row, d_col, d_val);
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

__global__ void __launch_bounds__(256) make_key32_kernel(const int32_t *__restrict__ major, int64_t n, uint32_t *__restrict__ key,
                                                         uint32_t *__restrict__ idx)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        key[i] = (uint32_t)major[i];
        idx[i] = (uint32_t)i;
    }
}

__global__ void __launch_bounds__(256) make_key64_kernel(const int32_t *__restrict__ major, const int32_t *__restrict__ minor,
                                                         int64_t n, int minor_bits, uint64_t *__restrict__ key,
                                                         uint32_t *__restrict__ idx)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        key[i] = ((uint64_t)(uint32_t)major[i] << minor_bits) | (uint64_t)(uint32_t)minor[i];
        idx[i] = (uint32_t)i;
    }
}

// Sorting permutation for the lexicographic order (major, minor).
//   already_sorted      : the list arrived in that order                  -> *d_idx = NULL, nothing to do
//   sorted_transposed   : the list arrived sorted by (minor, major)       -> stable sort on `major` alone
//   otherwise           : stable sort on the packed key major * 2^minor_bits + minor
int coo_sort_index(const int32_t *d_major, const int32_t *d_minor, int64_t nnz, int32_t n_major, int32_t n_minor,
                   bool already_sorted, bool sorted_transposed, DevPtr<uint32_t> *d_idx, cudaStream_t s)
{
    if (already_sorted || nnz <= 1)
        return SMVP_OK;
    int64_t blocks = ceil_div64(nnz, 256 * 4);
    const int64_t cap = (int64_t)device_props().sms * 16;
    if (blocks > cap)
        blocks = cap;
    const int major_bits = bits_for((uint32_t)n_major), minor_bits = bits_for((uint32_t)n_minor);
    DevPtr<uint32_t> idx_a, idx_b;
    uint32_t *res_idx = nullptr;
    SMVP_CUDA(dev_alloc(idx_a, nnz));
    SMVP_CUDA(dev_alloc(idx_b, nnz));
    if (sorted_transposed)
    {
        DevPtr<uint32_t> key_a, key_b;
        uint32_t *res_key = nullptr;
        SMVP_CUDA(dev_alloc(key_a, nnz));
        SMVP_CUDA(dev_alloc(key_b, nnz));
        SMVP_LAUNCH(make_key32_kernel, (unsigned)blocks, 256, 0, s, d_major, nnz, key_a.get(), idx_a.get());
        const int lo = 0, hi = major_bits;
        SMVP_TRY(radix_sort_pairs<uint32_t>(key_a.get(), idx_a.get(), key_b.get(), idx_b.get(), nnz, &lo, &hi, 1, &res_key, &res_idx,
                                            s));
    }
    else
    {
        DevPtr<uint64_t> key_a, key_b;
        uint64_t *res_key = nullptr;
        SMVP_CUDA(dev_alloc(key_a, nnz));
        SMVP_CUDA(dev_alloc(key_b, nnz));
        SMVP_LAUNCH(make_key64_kernel, (unsigned)blocks, 256, 0, s, d_major, d_minor, nnz, minor_bits, key_a.get(), idx_a.get());
        const int lo = 0, hi = major_bits + minor_bits;
        SMVP_TRY(radix_sort_pairs<uint64_t>(key_a.get(), idx_a.get(), key_b.get(), idx_b.get(), nnz, &lo, &hi, 1, &res_key, &res_idx,
                                            s));
    }
    *d_idx = std::move(res_idx == idx_a.get() ? idx_a : idx_b); // the sorted positions go to the caller
    return SMVP_OK;
}

} // namespace smvp
