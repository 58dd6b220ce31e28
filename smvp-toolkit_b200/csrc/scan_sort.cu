// scan_sort.cu -- integer primitives of the format builders: exclusive scan, histogram, stable LSD
// radix sort, max.  All hand-written; no CUB/Thrust.  Everything here is bit-exact integer work.
//
// They implement, on the device, the pieces the reference does with qsort() and running counters:
//   row-count scan      -> row_ptr            (main-cli.c:353-364)
//   column histogram    -> TXTable.colLength  (main-cli.c:845-862)
//   stable sorts        -> qsort by (row,col) :340, by (col,row) :766, by (len desc, col) :868,
//                          by (rank, slot) :926 -- all total orders when coordinates are unique,
//                          so a STABLE radix sort over the packed key reproduces them exactly.
#include "common.cuh"

namespace smvp
{

thread_local char g_last_cuda_error[256] = {0};
std::atomic<long long> g_launches{0};

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "%s: %s (%s:%d)", cudaGetErrorName(e), what, file, line);
    cudaGetLastError(); // clear the sticky-less error state
    if (e == cudaErrorMemoryAllocation)
        return SMVP_E_ALLOC;
    return SMVP_E_CUDA;
}

const DeviceProps &device_props()
{
    static thread_local DeviceProps p = {0, 0};
    static thread_local int cached_dev = -1;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess)
        dev = 0;
    if (cached_dev != dev)
    {
        cudaDeviceGetAttribute(&p.sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&p.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (p.sms <= 0)
            p.sms = 148;
        cached_dev = dev;
    }
    return p;
}

// =====================================================================================  scan
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) >= o)
            v += t;
    }
    return v;
}

// block-wide exclusive scan of one value per thread; returns exclusive prefix, *total = block sum
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *total)
{
    __shared__ uint32_t warp_sums[SCAN_THREADS / 32];
    __shared__ uint32_t block_total;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t incl = warp_incl_scan(v);
    if (lane == 31)
        warp_sums[w] = incl;
    __syncthreads();
    if (w == 0)
    {
        uint32_t s = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0;
        uint32_t si = warp_incl_scan(s);
        if (lane < SCAN_THREADS / 32)
            warp_sums[lane] = si - s;
        if (lane == SCAN_THREADS / 32 - 1)
            block_total = si;
    }
    __syncthreads();
    uint32_t r = incl - v + warp_sums[w];
    *total = block_total;
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_reduce_kernel(const uint32_t *__restrict__ in, int64_t n,
                                                                   uint32_t *__restrict__ block_sums)
{
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++)
    {
        int64_t i = base + (int64_t)k * SCAN_THREADS + threadIdx.x;
        if (i < n)
            s += in[i];
    }
    uint32_t total;
    block_excl_scan(s, &total);
    if (threadIdx.x == 0)
        block_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out,
                                                                  int64_t n, const uint32_t *__restrict__ block_offsets)
{
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++)
    {
        int64_t i = base + k;
        v[k] = i < n ? in[i] : 0;
        s += v[k];
    }
    uint32_t total;
    uint32_t prefix = block_excl_scan(s, &total) + (block_offsets ? block_offsets[blockIdx.x] : 0);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++)
    {
        int64_t i = base + k;
        if (i < n)
            out[i] = prefix;
        prefix += v[k];
    }
}

__global__ void scan_total_kernel(const uint32_t *in_last, const uint32_t *out_last, uint32_t *total)
{
    *total = *in_last + *out_last;
}

int exclusive_scan_u32(const uint32_t *d_in, uint32_t *d_out, int64_t n, uint32_t *d_total, cudaStream_t s)
{
    if (n <= 0)
    {
        if (d_total)
            SMVP_CUDA(cudaMemsetAsync(d_total, 0, sizeof(uint32_t), s));
        return SMVP_OK;
    }
    // the grand total needs in[n-1] before an in-place scan overwrites it
    DevPtr<uint32_t> last, sums;
    if (d_total)
    {
        SMVP_CUDA(dev_alloc(last, 1));
        SMVP_CUDA(cudaMemcpyAsync(last.get(), d_in + (n - 1), sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
    }
    const int64_t blocks = ceil_div64(n, SCAN_TILE);
    if (blocks == 1)
    {
        SMVP_LAUNCH(scan_apply_kernel, 1, SCAN_THREADS, 0, s, d_in, d_out, n, (const uint32_t *)nullptr);
    }
    else
    {
        SMVP_CUDA(dev_alloc(sums, blocks));
        uint32_t *d_sums = sums.get();
        SMVP_LAUNCH(scan_reduce_kernel, (unsigned)blocks, SCAN_THREADS, 0, s, d_in, n, d_sums);
        SMVP_TRY(exclusive_scan_u32(d_sums, d_sums, blocks, nullptr, s));
        SMVP_LAUNCH(scan_apply_kernel, (unsigned)blocks, SCAN_THREADS, 0, s, d_in, d_out, n, (const uint32_t *)d_sums);
    }
    if (d_total)
        SMVP_LAUNCH(scan_total_kernel, 1, 1, 0, s, (const uint32_t *)last.get(), (const uint32_t *)(d_out + (n - 1)), d_total);
    SMVP_CUDA(cudaStreamSynchronize(s));
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

// =====================================================================================  histogram
// warp-aggregated: lanes holding the same key elect a leader that adds the group's size once
__global__ void __launch_bounds__(256) histogram_kernel(const int32_t *__restrict__ keys, int64_t n,
                                                        uint32_t *__restrict__ counts)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x - lane; i0 < n; i0 += stride)
    {
        const int64_t i = i0 + lane;
        const bool ok = i < n;
        const int32_t k = ok ? keys[i] : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, k);
        if (ok && lane == __ffs(peers) - 1)
            atomicAdd(&counts[k], (uint32_t)__popc(peers));
    }
}

int histogram_i32(const int32_t *d_keys, int64_t n, uint32_t *d_counts, int64_t nbins, cudaStream_t s)
{
    SMVP_CUDA(cudaMemsetAsync(d_counts, 0, sizeof(uint32_t) * (size_t)nbins, s));
    if (n > 0)
    {
        int64_t blocks = ceil_div64(n, 256 * 8);
        const int64_t cap = (int64_t)device_props().sms * 32;
        if (blocks > cap)
            blocks = cap;
        SMVP_LAUNCH(histogram_kernel, (unsigned)blocks, 256, 0, s, d_keys, n, d_counts);
    }
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

// =====================================================================================  max
__global__ void __launch_bounds__(256) max_kernel(const uint32_t *__restrict__ in, int64_t n, uint32_t *__restrict__ out)
{
    uint32_t m = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        m = max(m, in[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0)
        atomicMax(out, m);
}

int max_u32(const uint32_t *d_in, int64_t n, uint32_t *d_out, cudaStream_t s)
{
    SMVP_CUDA(cudaMemsetAsync(d_out, 0, sizeof(uint32_t), s));
    if (n > 0)
    {
        int64_t blocks = ceil_div64(n, 256 * 8);
        const int64_t cap = (int64_t)device_props().sms * 16;
        if (blocks > cap)
            blocks = cap;
        SMVP_LAUNCH(max_kernel, (unsigned)blocks, 256, 0, s, d_in, n, d_out);
    }
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

// =====================================================================================  radix sort
// Stable LSD radix sort, 8-bit digits.  Per pass: (1) per-block digit histogram, (2) exclusive scan
// of the digit-major table, (3) stable scatter.  Stability inside a block comes from processing the
// tile in index order: warp w owns a contiguous 512-key chunk and walks it 32 keys at a time, ranking
// equal digits with __match_any_sync.
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_ITEMS = 16;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;
constexpr int RS_RADIX = 256;

template <typename KeyT>
__global__ void __launch_bounds__(RS_THREADS) rs_hist_kernel(const KeyT *__restrict__ keys, int64_t n, int shift,
                                                             uint32_t mask, uint32_t *__restrict__ block_hist,
                                                             uint32_t num_blocks)
{
    __shared__ uint32_t h[RS_RADIX];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * RS_TILE;
#pragma unroll
    for (int k = 0; k < RS_ITEMS; k++)
    {
        int64_t i = base + (int64_t)k * RS_THREADS + threadIdx.x;
        if (i < n)
            atomicAdd(&h[(uint32_t)(keys[i] >> shift) & mask], 1u);
    }
    __syncthreads();
    block_hist[(size_t)threadIdx.x * num_blocks + blockIdx.x] = h[threadIdx.x];
}

template <typename KeyT>
__global__ void __launch_bounds__(RS_THREADS) rs_scatter_kernel(const KeyT *__restrict__ keys_in,
                                                                const uint32_t *__restrict__ vals_in,
                                                                KeyT *__restrict__ keys_out, uint32_t *__restrict__ vals_out,
                                                                int64_t n, int shift, uint32_t mask,
                                                                const uint32_t *__restrict__ scanned, uint32_t num_blocks)
{
    __shared__ uint32_t cnt[RS_WARPS][RS_RADIX];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < RS_WARPS * RS_RADIX; i += RS_THREADS)
        (&cnt[0][0])[i] = 0;
    __syncthreads();

    const int64_t warp_base = (int64_t)blockIdx.x * RS_TILE + (int64_t)w * (RS_ITEMS * 32);
    KeyT key[RS_ITEMS];
    uint32_t val[RS_ITEMS];
    uint32_t rank[RS_ITEMS]; // low 16 bits: rank inside (warp, digit); high 16 bits: digit (0xffff = padding)
#pragma unroll
    for (int k = 0; k < RS_ITEMS; k++)
    {
        const int64_t i = warp_base + k * 32 + lane;
        const bool ok = i < n;
        key[k] = ok ? keys_in[i] : (KeyT)0;
        val[k] = ok ? vals_in[i] : 0u;
        const uint32_t d = ok ? ((uint32_t)(key[k] >> shift) & mask) : 0xffffu;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const uint32_t before = __popc(peers & ((1u << lane) - 1u));
        uint32_t c = 0;
        if (ok)
            c = cnt[w][d];
        __syncwarp();
        if (ok && before == 0)
            cnt[w][d] = c + __popc(peers);
        __syncwarp();
        rank[k] = (d << 16) | (c + before);
    }
    __syncthreads();
    {
        // thread t owns digit t: turn per-warp counts into per-warp bases inside the global run of digit t
        const uint32_t d = threadIdx.x;
        uint32_t base = scanned[(size_t)d * num_blocks + blockIdx.x];
#pragma unroll
        for (int ww = 0; ww < RS_WARPS; ww++)
        {
            const uint32_t t = cnt[ww][d];
            cnt[ww][d] = base;
            base += t;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < RS_ITEMS; k++)
    {
        const uint32_t d = rank[k] >> 16;
        if (d != 0xffffu)
        {
            const uint32_t pos = cnt[w][d] + (rank[k] & 0xffffu);
            keys_out[pos] = key[k];
            vals_out[pos] = val[k];
        }
    }
}

template <typename KeyT>
int radix_sort_pairs(KeyT *keys_a, uint32_t *vals_a, KeyT *keys_b, uint32_t *vals_b, int64_t n, const int *bit_lo,
                     const int *bit_hi, int nranges, KeyT **out_keys, uint32_t **out_vals, cudaStream_t s)
{
    *out_keys = keys_a;
    *out_vals = vals_a;
    if (n <= 1)
        return SMVP_OK;
    if (n >= ((int64_t)1 << 32))
        return SMVP_E_TOOBIG;
    const uint32_t blocks = (uint32_t)ceil_div64(n, RS_TILE);
    DevPtr<uint32_t> hist;
    SMVP_CUDA(dev_alloc(hist, (int64_t)blocks * RS_RADIX));
    uint32_t *d_hist = hist.get();
    KeyT *kin = keys_a, *kout = keys_b;
    uint32_t *vin = vals_a, *vout = vals_b;
    int rc = SMVP_OK;
    for (int r = 0; r < nranges && rc == SMVP_OK; r++)
    {
        for (int lo = bit_lo[r]; lo < bit_hi[r] && rc == SMVP_OK; lo += 8)
        {
            const int nb = (bit_hi[r] - lo) < 8 ? (bit_hi[r] - lo) : 8;
            const uint32_t mask = (1u << nb) - 1u;
            auto k_hist = rs_hist_kernel<KeyT>;
            auto k_scatter = rs_scatter_kernel<KeyT>;
            SMVP_LAUNCH(k_hist, blocks, RS_THREADS, 0, s, (const KeyT *)kin, n, lo, mask, d_hist, blocks);
            rc = exclusive_scan_u32(d_hist, d_hist, (int64_t)blocks * RS_RADIX, nullptr, s);
            if (rc != SMVP_OK)
                break;
            SMVP_LAUNCH(k_scatter, blocks, RS_THREADS, 0, s, (const KeyT *)kin, (const uint32_t *)vin, kout, vout, n, lo,
                        mask, (const uint32_t *)d_hist, blocks);
            KeyT *tk = kin;
            kin = kout;
            kout = tk;
            uint32_t *tv = vin;
            vin = vout;
            vout = tv;
        }
    }
    cudaError_t e = cudaStreamSynchronize(s);
    if (rc != SMVP_OK)
        return rc;
    SMVP_CUDA(e);
    SMVP_CUDA(cudaGetLastError());
    *out_keys = kin;
    *out_vals = vin;
    return SMVP_OK;
}

template int radix_sort_pairs<uint32_t>(uint32_t *, uint32_t *, uint32_t *, uint32_t *, int64_t, const int *, const int *, int,
                                        uint32_t **, uint32_t **, cudaStream_t);
template int radix_sort_pairs<uint64_t>(uint64_t *, uint32_t *, uint64_t *, uint32_t *, int64_t, const int *, const int *, int,
                                        uint64_t **, uint32_t **, cudaStream_t);

} // namespace smvp
