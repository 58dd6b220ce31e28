// pattern.cu -- row-pattern plan of a CSR handle: the multiply reads a one-byte pattern id per row INSTEAD of col_ind.
// A multiply-side plan, like relabel.cu: the arrays the reference defines (CSRData, main-cli.c:61-66) stay untouched.
//
// Why: on a structured-grid operator col_ind carries almost no information.  Written relative to its row, `col - row`,
// every row of the 27-point stencil holds one of 27 offset lists (interior, face, edge or corner in x, y and z); 5-, 7-
// and 9-point stencils and banded matrices work the same way.  col_ind is 4 of the 12 bytes a nonzero streams, so a
// pass that reads pat_id[rows] (1 B per row) and a table of a few KB instead moves about 30 % fewer bytes.
//
// What: pat_off[p * PAT_LMAX + k] = k-th column offset of pattern p, pat_len[p] = its length, pat_id[r] = pattern of row
// r.  Row r's k-th nonzero sits in column r + pat_off[pat_id[r] * PAT_LMAX + k] -- exactly col_ind[row_ptr[r] + k].
//
// How (decided from row_ptr and col_ind only, once per handle, synchronous):
//   1. every row hashes its length and offsets; the hashes go into a small open-addressing table on the device, each
//      slot keeping the smallest row that produced it (its representative);
//   2. the host numbers the slots by representative row (deterministic ids) and the table of offsets is read from
//      those rows;
//   3. every row looks its hash up again and compares its offsets ENTRY BY ENTRY with its pattern: any mismatch (a hash
//      collision) rejects the plan.  A hash match alone never decides a column.
// The plan is given up when a row is longer than PAT_LMAX, when more than PAT_MAX patterns occur, or when the handle is
// relabelled (that plan decides first).  SMVP_CSR_PATTERN=0 keeps it off.
//
// Value width: with col_ind gone, val is 93 % of what the pattern kernel streams.  Once the plan is accepted, one pass
// over val checks which of fp16 and fp32 hold every value with the same 64 bits (pattern and integer matrices,
// constant-coefficient stencils such as the benchmark's {26, -1}); the kernel then streams a copy at the narrowest such
// width and widens each value exactly, so y is unchanged.  It depends on the precision the values need, not on how many
// distinct values there are.  val itself stays for every other path.
#include "common.cuh"

#include <algorithm>
#include <vector>

namespace smvp
{

constexpr int PAT_SLOTS = 4096; // hash table of the detection: 16x the largest pattern count keeps the probe chains short
constexpr int PAT_FLAG_LONG = 1, PAT_FLAG_MANY = 2, PAT_FLAG_MISMATCH = 4;

__device__ __forceinline__ uint64_t mix64(uint64_t h)
{
    h ^= h >> 33;
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    h *= 0xc4ceb9fe1a85ec53ull;
    h ^= h >> 33;
    return h;
}

// hash of (length, offsets in order); never 0, which marks an empty slot
__device__ __forceinline__ uint64_t row_hash(const int32_t *__restrict__ col_ind, int32_t a, int32_t len, int32_t r)
{
    uint64_t h = mix64(0x9e3779b97f4a7c15ull + (uint64_t)len);
    for (int32_t k = 0; k < len; k++)
        h = mix64(h ^ ((uint64_t)(uint32_t)(col_ind[a + k] - r) + ((uint64_t)k << 32)));
    return h | 1ull;
}

__global__ void __launch_bounds__(256) pattern_hash_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col_ind,
                                                           int32_t rows, unsigned long long *keys, int32_t *rep, int32_t *count,
                                                           int32_t *flags)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x)
    {
        if (*(volatile int32_t *)flags)
            return; // rejected already: the other rows need not be looked at
        const int32_t a = row_ptr[r], len = row_ptr[r + 1] - a;
        if (len > PAT_LMAX)
        {
            atomicOr(flags, PAT_FLAG_LONG);
            return;
        }
        const uint64_t h = row_hash(col_ind, a, len, (int32_t)r);
        uint32_t slot = (uint32_t)h & (PAT_SLOTS - 1);
        for (int probe = 0; probe < PAT_SLOTS; probe++, slot = (slot + 1) & (PAT_SLOTS - 1))
        {
            // plain reads first: almost every row finds its pattern already there with a smaller representative, and an
            // atomic per row on the same few addresses would serialise the whole pass
            unsigned long long k = __ldcg(keys + slot);
            if (k == 0)
            {
                k = atomicCAS(keys + slot, 0ull, (unsigned long long)h);
                if (k == 0 && atomicAdd(count, 1) >= PAT_MAX)
                {
                    atomicOr(flags, PAT_FLAG_MANY);
                    return;
                }
                if (k == 0)
                    k = h;
            }
            if (k == h)
            {
                if ((int32_t)r < __ldcg(rep + slot))
                    atomicMin(rep + slot, (int32_t)r);
                break;
            }
        }
    }
}

// pattern p = the offsets of its representative row
__global__ void pattern_table_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col_ind,
                                     const int32_t *__restrict__ reps, int32_t npat, int32_t *__restrict__ pat_off,
                                     int32_t *__restrict__ pat_len)
{
    const int32_t p = blockIdx.x, k = threadIdx.x;
    if (p >= npat)
        return;
    const int32_t r = reps[p], a = row_ptr[r], len = row_ptr[r + 1] - a;
    if (k == 0)
        pat_len[p] = len;
    pat_off[p * PAT_LMAX + k] = k < len ? col_ind[a + k] - r : 0;
}

__global__ void __launch_bounds__(256) pattern_assign_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col_ind,
                                                             int32_t rows, const unsigned long long *__restrict__ keys,
                                                             const int32_t *__restrict__ slot_id, const int32_t *__restrict__ pat_off,
                                                             const int32_t *__restrict__ pat_len, uint8_t *__restrict__ pat_id,
                                                             int32_t *flags)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t a = row_ptr[r], len = row_ptr[r + 1] - a;
        const uint64_t h = row_hash(col_ind, a, len, (int32_t)r);
        uint32_t slot = (uint32_t)h & (PAT_SLOTS - 1);
        int32_t id = -1;
        for (int probe = 0; probe < PAT_SLOTS; probe++, slot = (slot + 1) & (PAT_SLOTS - 1))
        {
            const unsigned long long k = keys[slot];
            if (k == h)
            {
                id = slot_id[slot];
                break;
            }
            if (k == 0)
                break;
        }
        bool same = id >= 0 && pat_len[id] == len;
        for (int32_t k = 0; same && k < len; k++)
            same = col_ind[a + k] - (int32_t)r == pat_off[id * PAT_LMAX + k];
        if (!same)
        {
            atomicOr(flags, PAT_FLAG_MISMATCH);
            return;
        }
        pat_id[r] = (uint8_t)id;
    }
}

// flags |= 1 when some value does not survive fp16 and back with its 64 bits, |= 2 when some value does not survive fp32.
// Bits, not ==: -0.0 keeps its sign, subnormals and out-of-range values fail, a NaN passes only with its payload intact.
__global__ void __launch_bounds__(256) pattern_width_kernel(const double *__restrict__ val, int64_t nnz, int32_t *flags)
{
    unsigned f = 0;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nnz; j += (int64_t)gridDim.x * blockDim.x)
    {
        const double v = val[j];
        const long long b = __double_as_longlong(v);
        if (__double_as_longlong(widen_value(narrow_value<uint16_t>(v))) != b)
            f |= 1u;
        if (__double_as_longlong(widen_value(narrow_value<float>(v))) != b)
            f |= 2u;
    }
    f = __reduce_or_sync(0xffffffffu, f);
    if ((threadIdx.x & 31) == 0 && f)
        atomicOr(flags, (int32_t)f);
}

template <typename V>
__global__ void __launch_bounds__(256) pattern_narrow_kernel(const double *__restrict__ val, int64_t nnz, V *__restrict__ out)
{
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nnz; j += (int64_t)gridDim.x * blockDim.x)
        out[j] = narrow_value<V>(val[j]);
}

// the narrowest width (2, 4 or 8 bytes) that holds every value exactly, and the copy of val at that width
static int pattern_values(smvp_csr *A, unsigned grid, cudaStream_t s)
{
    DevTmp g_flags;
    SMVP_CUDA(g_flags.alloc<int32_t>(1));
    int32_t *flags = g_flags.as<int32_t>(), h_flags = 0;
    SMVP_CUDA(cudaMemsetAsync(flags, 0, sizeof(int32_t), s));
    if (A->nnz > 0)
        SMVP_LAUNCH(pattern_width_kernel, grid, 256, 0, s, (const double *)A->val, A->nnz, flags);
    SMVP_CUDA(cudaGetLastError());
    SMVP_CUDA(cudaMemcpyAsync(&h_flags, flags, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaStreamSynchronize(s));
    const int32_t vbytes = !(h_flags & 1) ? 2 : !(h_flags & 2) ? 4 : 8;
    if (vbytes == 2)
    {
        SMVP_CUDA(dev_alloc((uint16_t **)&A->pat_val, A->nnz));
        if (A->nnz > 0)
            SMVP_LAUNCH(pattern_narrow_kernel<uint16_t>, grid, 256, 0, s, (const double *)A->val, A->nnz, (uint16_t *)A->pat_val);
    }
    else if (vbytes == 4)
    {
        SMVP_CUDA(dev_alloc((float **)&A->pat_val, A->nnz));
        if (A->nnz > 0)
            SMVP_LAUNCH(pattern_narrow_kernel<float>, grid, 256, 0, s, (const double *)A->val, A->nnz, (float *)A->pat_val);
    }
    SMVP_CUDA(cudaGetLastError());
    SMVP_CUDA(cudaStreamSynchronize(s));
    A->pat_vbytes = vbytes;
    return SMVP_OK;
}

void csr_pattern_release(smvp_csr *A)
{
    cudaFree(A->pat_id);
    cudaFree(A->pat_off);
    cudaFree(A->pat_len);
    cudaFree(A->pat_val);
    A->pat_id = nullptr;
    A->pat_off = A->pat_len = nullptr;
    A->pat_val = nullptr;
    A->pat_vbytes = 0;
}

// decides (once per handle) and, when every row matches one of at most PAT_MAX patterns, builds the plan.  Synchronous.
int csr_pattern_plan(smvp_csr *A, cudaStream_t s)
{
    SMVP_TRY(csr_relabel_plan(A, s)); // a relabelled handle reads col_rel: that plan decides first
    if (A->pattern_state != 0)
        return SMVP_OK;
    if (A->relabel_state == 1 || A->rows == 0 || env_tristate("SMVP_CSR_PATTERN") == -1)
    {
        A->pattern_state = -1;
        return SMVP_OK;
    }
    DevTmp g_keys, g_rep, g_flags, g_slot_id, g_reps;
    SMVP_CUDA(g_keys.alloc<unsigned long long>(PAT_SLOTS));
    SMVP_CUDA(g_rep.alloc<int32_t>(PAT_SLOTS));
    SMVP_CUDA(g_flags.alloc<int32_t>(2)); // [0] flags, [1] patterns inserted
    SMVP_CUDA(g_slot_id.alloc<int32_t>(PAT_SLOTS));
    SMVP_CUDA(g_reps.alloc<int32_t>(PAT_MAX));
    unsigned long long *keys = g_keys.as<unsigned long long>();
    int32_t *rep = g_rep.as<int32_t>(), *flags = g_flags.as<int32_t>();
    SMVP_CUDA(cudaMemsetAsync(keys, 0, sizeof(unsigned long long) * PAT_SLOTS, s));
    SMVP_CUDA(cudaMemsetAsync(rep, 0x7f, sizeof(int32_t) * PAT_SLOTS, s));
    SMVP_CUDA(cudaMemsetAsync(flags, 0, 2 * sizeof(int32_t), s));
    const int64_t blocks = ceil_div64(A->rows, 256), cap = (int64_t)device_props().sms * 8;
    const unsigned grid = (unsigned)(blocks < cap ? blocks : cap);
    SMVP_LAUNCH(pattern_hash_kernel, grid, 256, 0, s, A->row_ptr, A->col_ind, A->rows, keys, rep, flags + 1, flags);
    SMVP_CUDA(cudaGetLastError());
    std::vector<unsigned long long> h_keys(PAT_SLOTS);
    std::vector<int32_t> h_rep(PAT_SLOTS);
    int32_t h_flags[2] = {0, 0};
    SMVP_CUDA(cudaMemcpyAsync(h_flags, flags, sizeof(h_flags), cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaMemcpyAsync(h_keys.data(), keys, sizeof(unsigned long long) * PAT_SLOTS, cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaMemcpyAsync(h_rep.data(), rep, sizeof(int32_t) * PAT_SLOTS, cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaStreamSynchronize(s));
    if (h_flags[0])
    {
        A->pattern_state = -1;
        return SMVP_OK;
    }
    // deterministic ids: patterns numbered by their representative rows, ascending
    std::vector<std::pair<int32_t, int32_t>> by_rep; // (representative row, slot)
    for (int k = 0; k < PAT_SLOTS; k++)
        if (h_keys[k])
            by_rep.push_back({h_rep[k], k});
    std::sort(by_rep.begin(), by_rep.end());
    const int32_t npat = (int32_t)by_rep.size();
    std::vector<int32_t> h_slot_id(PAT_SLOTS, -1), h_reps(npat);
    for (int32_t p = 0; p < npat; p++)
    {
        h_slot_id[by_rep[p].second] = p;
        h_reps[p] = by_rep[p].first;
    }
    auto body = [&]() -> int {
        SMVP_CUDA(dev_alloc(&A->pat_id, A->rows));
        SMVP_CUDA(dev_alloc(&A->pat_off, (int64_t)npat * PAT_LMAX));
        SMVP_CUDA(dev_alloc(&A->pat_len, npat));
        SMVP_CUDA(cudaMemcpyAsync(g_slot_id.p, h_slot_id.data(), sizeof(int32_t) * PAT_SLOTS, cudaMemcpyHostToDevice, s));
        SMVP_CUDA(cudaMemcpyAsync(g_reps.p, h_reps.data(), sizeof(int32_t) * npat, cudaMemcpyHostToDevice, s));
        SMVP_LAUNCH(pattern_table_kernel, (unsigned)npat, PAT_LMAX, 0, s, A->row_ptr, A->col_ind, g_reps.as<int32_t>(), npat,
                    A->pat_off, A->pat_len);
        SMVP_LAUNCH(pattern_assign_kernel, grid, 256, 0, s, A->row_ptr, A->col_ind, A->rows, keys, g_slot_id.as<int32_t>(),
                    A->pat_off, A->pat_len, A->pat_id, flags);
        SMVP_CUDA(cudaGetLastError());
        std::vector<int32_t> h_len(npat);
        SMVP_CUDA(cudaMemcpyAsync(h_flags, flags, sizeof(h_flags), cudaMemcpyDeviceToHost, s));
        SMVP_CUDA(cudaMemcpyAsync(h_len.data(), A->pat_len, sizeof(int32_t) * npat, cudaMemcpyDeviceToHost, s));
        SMVP_CUDA(cudaStreamSynchronize(s));
        A->pattern_maxlen = npat > 0 ? *std::max_element(h_len.begin(), h_len.end()) : 0;
        return SMVP_OK;
    };
    const int rc = body();
    if (rc != SMVP_OK || h_flags[0])
    {
        csr_pattern_release(A);
        A->pattern_state = rc == SMVP_OK ? -1 : 0;
        return rc;
    }
    const int rv = pattern_values(A, grid, s);
    if (rv != SMVP_OK)
    {
        csr_pattern_release(A);
        return rv; // undecided: the next pass tries again
    }
    A->pattern_count = npat;
    A->device_bytes += (int64_t)A->rows + 4 * (int64_t)npat * (PAT_LMAX + 1) + (A->pat_vbytes < 8 ? A->pat_vbytes * A->nnz : 0);
    A->pattern_state = 1;
    return SMVP_OK;
}

} // namespace smvp
