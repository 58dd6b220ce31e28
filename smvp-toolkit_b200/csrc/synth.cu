// synth.cu -- device-side synthetic inputs for the configurations BASELINE.json names
// (27-point stencil, R-MAT) and the COO shard helpers of the multi-GPU path.  See include/smvp_synth.h.
// The reference has no generator (its only input is the .mtx loader, main-cli.c:1405-1441).
#include "common.cuh"
#include "../../include/smvp_synth.h"

namespace smvp
{

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
__host__ __device__ __forceinline__ double hash_uniform(uint64_t h) // (-1, 1)
{
    return 2.0 * ((double)(h >> 11) * (1.0 / 9007199254740992.0)) - 1.0;
}
__host__ __device__ __forceinline__ double hash_value(uint64_t seed, uint32_t row, uint32_t col)
{
    return hash_uniform(splitmix64(seed ^ splitmix64(((uint64_t)row << 32) | (uint64_t)col)));
}

// ------------------------------------------------------------------ 27-point stencil
__host__ __device__ __forceinline__ int span1d(int32_t i, int32_t n) { return 1 + (i > 0 ? 1 : 0) + (i < n - 1 ? 1 : 0); }

__global__ void __launch_bounds__(256) stencil_count_kernel(int32_t nx, int32_t ny, int32_t nz, int64_t row_begin, int64_t nrows,
                                                            uint32_t *__restrict__ counts)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrows)
        return;
    const int64_t r = row_begin + i;
    const int32_t ix = (int32_t)(r % nx), iy = (int32_t)((r / nx) % ny), iz = (int32_t)(r / ((int64_t)nx * ny));
    counts[i] = (uint32_t)(span1d(ix, nx) * span1d(iy, ny) * span1d(iz, nz));
}

__global__ void __launch_bounds__(256) stencil_fill_kernel(int32_t nx, int32_t ny, int32_t nz, int64_t row_begin, int64_t nrows,
                                                           const uint32_t *__restrict__ offsets, int value_mode, uint64_t seed,
                                                           int32_t *__restrict__ row, int32_t *__restrict__ col, double *__restrict__ val)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrows)
        return;
    const int64_t r = row_begin + i;
    const int32_t ix = (int32_t)(r % nx), iy = (int32_t)((r / nx) % ny), iz = (int32_t)(r / ((int64_t)nx * ny));
    int64_t o = offsets[i];
    for (int dz = -1; dz <= 1; dz++)
    {
        const int32_t z = iz + dz;
        if (z < 0 || z >= nz)
            continue;
        for (int dy = -1; dy <= 1; dy++)
        {
            const int32_t y = iy + dy;
            if (y < 0 || y >= ny)
                continue;
            for (int dx = -1; dx <= 1; dx++)
            {
                const int32_t x = ix + dx;
                if (x < 0 || x >= nx)
                    continue;
                const int64_t c = (int64_t)x + (int64_t)nx * ((int64_t)y + (int64_t)ny * z);
                row[o] = (int32_t)i;
                col[o] = (int32_t)c;
                double v;
                if (value_mode == SMVP_VAL_STENCIL)
                    v = (c == r) ? 26.0 : -1.0;
                else if (value_mode == SMVP_VAL_HASH)
                    v = hash_value(seed, (uint32_t)r, (uint32_t)c);
                else
                    v = 1.0;
                val[o] = v;
                o++;
            }
        }
    }
}

// ------------------------------------------------------------------ R-MAT
__global__ void __launch_bounds__(256) rmat_edges_kernel(int scale, int64_t nedges, double a, double ab, double abc, uint64_t seed,
                                                         uint64_t *__restrict__ key, uint32_t *__restrict__ idx)
{
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nedges; e += (int64_t)gridDim.x * blockDim.x)
    {
        const uint64_t base = splitmix64(seed ^ (uint64_t)e);
        uint32_t r = 0, c = 0;
        for (int l = 0; l < scale; l++)
        {
            const double u = (double)(splitmix64(base + (uint64_t)l) >> 11) * (1.0 / 9007199254740992.0);
            const uint32_t rb = u >= ab ? 1u : 0u;                       // quadrants c, d -> lower half
            const uint32_t cb = (u >= a && u < ab) || (u >= abc) ? 1u : 0u; // quadrants b, d -> right half
            r = (r << 1) | rb;
            c = (c << 1) | cb;
        }
        key[e] = ((uint64_t)r << scale) | (uint64_t)c;
        idx[e] = (uint32_t)e;
    }
}

__global__ void __launch_bounds__(256) unique_flag_kernel(const uint64_t *__restrict__ key, int64_t n, uint32_t *__restrict__ flag)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        flag[i] = (i == 0 || key[i] != key[i - 1]) ? 1u : 0u;
}

__global__ void __launch_bounds__(256) rmat_compact_kernel(const uint64_t *__restrict__ key, const uint32_t *__restrict__ pos, int64_t n,
                                                           int scale, int value_mode, uint64_t seed, int32_t *__restrict__ row,
                                                           int32_t *__restrict__ col, double *__restrict__ val)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        if (i == 0 || key[i] != key[i - 1])
        {
            const uint32_t o = pos[i];
            const uint32_t r = (uint32_t)(key[i] >> scale), c = (uint32_t)(key[i] & ((1ULL << scale) - 1ULL));
            row[o] = (int32_t)r;
            col[o] = (int32_t)c;
            val[o] = value_mode == SMVP_VAL_HASH ? hash_value(seed, r, c) : 1.0;
        }
    }
}

__global__ void __launch_bounds__(256) vector_fill_kernel(double *__restrict__ x, int64_t n, uint64_t seed)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        x[i] = seed == 0 ? 1.0 : hash_uniform(splitmix64(seed ^ splitmix64((uint64_t)i)));
}

// ------------------------------------------------------------------ COO filter
__global__ void __launch_bounds__(256) filter_flag_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col, int64_t n,
                                                          int32_t rlo, int32_t rhi, int32_t clo, int32_t chi, uint32_t *__restrict__ flag)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t r = row[i], c = col[i];
        flag[i] = (r >= rlo && r < rhi && c >= clo && c < chi) ? 1u : 0u;
    }
}

__global__ void __launch_bounds__(256) filter_scatter_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col,
                                                             const double *__restrict__ val, int64_t n, int32_t rlo, int32_t rhi,
                                                             int32_t clo, int32_t chi, int32_t rshift, int32_t cshift,
                                                             const uint32_t *__restrict__ pos, int32_t *__restrict__ o_row,
                                                             int32_t *__restrict__ o_col, double *__restrict__ o_val)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t r = row[i], c = col[i];
        if (r >= rlo && r < rhi && c >= clo && c < chi)
        {
            const uint32_t o = pos[i];
            o_row[o] = r - rshift;
            o_col[o] = c - cshift;
            o_val[o] = val[i];
        }
    }
}

__global__ void __launch_bounds__(256) vector_add_kernel(double *__restrict__ y, const double *__restrict__ a, int64_t n)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        y[i] = __dadd_rn(y[i], a[i]);
}

__global__ void __launch_bounds__(512) push_kernel(double2 *__restrict__ dst, const double2 *__restrict__ src, int64_t n16,
                                                   double *__restrict__ dst_tail, const double *__restrict__ src_tail, int tail)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n16; i += 4 * stride) // four independent loads in flight per thread
    {
        const double2 a = src[i], b = src[i + stride], c = src[i + 2 * stride], d = src[i + 3 * stride];
        dst[i] = a;
        dst[i + stride] = b;
        dst[i + 2 * stride] = c;
        dst[i + 3 * stride] = d;
    }
    for (; i < n16; i += stride)
        dst[i] = src[i];
    if (blockIdx.x == 0 && (int)threadIdx.x < tail)
        dst_tail[threadIdx.x] = src_tail[threadIdx.x];
}

// the same with up to 8 destinations: src is read once, every 16-byte piece is stored to each destination (peer
// mappings of a symmetric-memory buffer: the unicast all-gather of one rank's block)
struct PushFan
{
    double2 *dst[8];
    double *dst_tail[8];
    int n;
};
__global__ void __launch_bounds__(512) push_fanout_kernel(const __grid_constant__ PushFan fan, const double2 *__restrict__ src, int64_t n16,
                                                          const double *__restrict__ src_tail, int tail)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n16; i += 4 * stride) // four independent loads in flight per thread
    {
        const double2 a = src[i], b = src[i + stride], c = src[i + 2 * stride], d = src[i + 3 * stride];
        for (int k = 0; k < fan.n; k++)
        {
            fan.dst[k][i] = a;
            fan.dst[k][i + stride] = b;
            fan.dst[k][i + 2 * stride] = c;
            fan.dst[k][i + 3 * stride] = d;
        }
    }
    for (; i < n16; i += stride)
    {
        const double2 a = src[i];
        for (int k = 0; k < fan.n; k++)
            fan.dst[k][i] = a;
    }
    if (blockIdx.x == 0 && (int)threadIdx.x < tail)
        for (int k = 0; k < fan.n; k++)
            fan.dst_tail[k][threadIdx.x] = src_tail[threadIdx.x];
}

// ---- the same fan-out done by the TMA engine: a CTA is ONE warp whose lane 0 streams 4 KB chunks of the source through a
// ring of shared-memory stages with cp.async.bulk (global -> shared, mbarrier completion) and sends each stage to every
// destination with cp.async.bulk (shared -> global, bulk groups).  No register staging, no per-thread stores: the SM
// only issues descriptors, the copies leave the chip as full-size write packets (what a copy engine emits) and the
// source is read once whatever the number of destinations.  `ctas` one-warp CTAs with 16 KB of shared memory each sit
// beside the SpMV's CTAs; 64 of them keep ~1 MB in flight.
// 4 x 4 KB = 16 KB per CTA, 6 registers: such a CTA fits into what a fully resident merge-path SpMV leaves free on an SM
// (9 CTAs x (21.5 + 1) KB of the 228 KB of shared memory, 63 K of the 64 K registers), so the SpMV's persistent grid stays
// completely resident beside it.  A co-runner that does NOT fit (the 512-thread store kernels above, or 64 KB stages here) makes
// part of the persistent grid start only when another CTA retires -- a tail as long as the kernel itself (measured at
// 2 GPUs: 1.34 -> 1.7 ms per SpMV under such a push, 1.44 ms under a copy-engine transfer).
constexpr int PUSH_TMA_STAGES = 4;
constexpr int PUSH_TMA_CHUNK = 4096;
struct PushTma
{
    char *dst[8];
    int n;
};
__device__ __forceinline__ uint32_t push_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__global__ void __launch_bounds__(32) push_tma_kernel(const __grid_constant__ PushTma fan, const char *__restrict__ src, int64_t bytes16)
{
    // bytes16: multiple of 16; chunk i = bytes [i * CHUNK, min((i+1) * CHUNK, bytes16))
    extern __shared__ __align__(128) unsigned char push_stage[];
    __shared__ __align__(8) uint64_t full_bar[PUSH_TMA_STAGES];
    if (threadIdx.x != 0)
        return;
    for (int s = 0; s < PUSH_TMA_STAGES; s++)
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(push_smem_u32(&full_bar[s])), "r"(1));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const int64_t nchunks = (bytes16 + PUSH_TMA_CHUNK - 1) / PUSH_TMA_CHUNK;
    const int64_t G = gridDim.x;
    auto chunk_bytes = [&](int64_t c) -> uint32_t {
        const int64_t left = bytes16 - c * PUSH_TMA_CHUNK;
        return (uint32_t)(left < PUSH_TMA_CHUNK ? left : PUSH_TMA_CHUNK);
    };
    auto load = [&](int64_t c, int s) {
        const uint32_t n = chunk_bytes(c), bar = push_smem_u32(&full_bar[s]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(n) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         push_smem_u32(push_stage + (size_t)s * PUSH_TMA_CHUNK)),
                     "l"(src + c * PUSH_TMA_CHUNK), "r"(n), "r"(bar)
                     : "memory");
    };
    // my chunks: blockIdx.x, blockIdx.x + G, ...; `it` counts them
    int64_t c_load = blockIdx.x;
    int it_load = 0;
    for (; it_load < PUSH_TMA_STAGES - 1 && c_load < nchunks; it_load++, c_load += G)
        load(c_load, it_load % PUSH_TMA_STAGES);
    int it = 0;
    for (int64_t c = blockIdx.x; c < nchunks; c += G, it++)
    {
        const int s = it % PUSH_TMA_STAGES;
        const uint32_t bar = push_smem_u32(&full_bar[s]), parity = (uint32_t)((it / PUSH_TMA_STAGES) & 1);
        asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\t"
                     "bra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(bar),
                     "r"(parity)
                     : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        const uint32_t n = chunk_bytes(c), sm = push_smem_u32(push_stage + (size_t)s * PUSH_TMA_CHUNK);
        for (int k = 0; k < fan.n; k++)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(fan.dst[k] + c * PUSH_TMA_CHUNK), "r"(sm), "r"(n)
                         : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        // refill the stage the PREVIOUS chunk used: its stores must have read shared memory (not reached the peers)
        if (c_load < nchunks)
        {
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            load(c_load, it_load % PUSH_TMA_STAGES);
            it_load++;
            c_load += G;
        }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); // every store performed before the kernel ends
}

// out[i] = (((p_0[i] + p_1[i]) + p_2[i]) + ...), p_k = parts + k * stride: the fixed-order combine of per-rank partial
// results (column-block TJDS): the same bits whatever order the parts arrived in
__global__ void __launch_bounds__(256) sum_ordered_kernel(double *__restrict__ out, const double *__restrict__ parts, int nparts,
                                                          int64_t stride, int64_t n)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        double acc = parts[i];
        for (int k = 1; k < nparts; k++)
            acc = __dadd_rn(acc, parts[(int64_t)k * stride + i]);
        out[i] = acc;
    }
}

// the same with the parts given as separate pointers (peer mappings of a symmetric-memory buffer): the owner of a row
// block PULLS that block of every rank's partial y over NVLink and adds them in rank order -- a reduce-scatter whose
// bits do not depend on any library's reduction order
struct PartPtrs
{
    const double *p[16];
    int n;
};
__global__ void __launch_bounds__(256) sum_ordered_ptrs_kernel(double *__restrict__ out, const __grid_constant__ PartPtrs parts, int64_t n)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n2 = n / 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride)
    {
        double2 v[16];
#pragma unroll
        for (int k = 0; k < 16; k++) // all loads first: one NVLink round trip per element pair, not one per part
            if (k < parts.n)
                v[k] = reinterpret_cast<const double2 *>(parts.p[k])[i];
        double2 acc = v[0];
#pragma unroll
        for (int k = 1; k < 16; k++)
            if (k < parts.n)
            {
                acc.x = __dadd_rn(acc.x, v[k].x);
                acc.y = __dadd_rn(acc.y, v[k].y);
            }
        reinterpret_cast<double2 *>(out)[i] = acc;
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0)
    {
        double acc = parts.p[0][n - 1];
        for (int k = 1; k < parts.n; k++)
            acc = __dadd_rn(acc, parts.p[k][n - 1]);
        out[n - 1] = acc;
    }
}

static inline unsigned grid_for(int64_t n, int per_thread = 4)
{
    int64_t blocks = ceil_div64(n > 0 ? n : 1, 256 * per_thread);
    const int64_t cap = (int64_t)device_props().sms * 16;
    if (blocks > cap)
        blocks = cap;
    return (unsigned)blocks;
}

} // namespace smvp

using namespace smvp;

static int64_t prefix1d(int32_t n, int64_t k) // sum of span1d(i, n) for i < k
{
    if (k <= 0)
        return 0;
    if (n == 1)
        return 1;
    return 3 * k - 1 - (k == n ? 1 : 0);
}

extern "C" int64_t smvp_synth_stencil27_prefix(int32_t nx, int32_t ny, int32_t nz, int64_t row)
{
    const int64_t total = (int64_t)nx * ny * nz;
    if (row <= 0)
        return 0;
    if (row > total)
        row = total;
    const int64_t sx = prefix1d(nx, nx), sy = prefix1d(ny, ny);
    const int32_t ix = (int32_t)(row % nx), iy = (int32_t)((row / nx) % ny);
    const int64_t iz = row / ((int64_t)nx * ny);
    if (iz >= nz)
        return prefix1d(nz, nz) * sy * sx;
    const int64_t cz = span1d((int32_t)iz, nz), cy = span1d(iy, ny);
    return prefix1d(nz, iz) * sy * sx + cz * prefix1d(ny, iy) * sx + cz * cy * prefix1d(nx, ix);
}

extern "C" int smvp_synth_stencil27(int32_t nx, int32_t ny, int32_t nz, int64_t row_begin, int64_t row_end, int value_mode,
                                    uint64_t seed, int32_t **d_row, int32_t **d_col, double **d_val, int64_t *nnz)
{
    if (!d_row || !d_col || !d_val || !nnz || nx < 1 || ny < 1 || nz < 1)
        return SMVP_E_ARG;
    const int64_t total = (int64_t)nx * ny * nz;
    if (total > 0x7fffffffLL || row_begin < 0 || row_end > total || row_begin > row_end)
        return SMVP_E_ARG;
    const int64_t nrows = row_end - row_begin;
    const int64_t n = smvp_synth_stencil27_prefix(nx, ny, nz, row_end) - smvp_synth_stencil27_prefix(nx, ny, nz, row_begin);
    if (n > 0x7fffffffLL - 1024)
        return SMVP_E_TOOBIG;
    *nnz = n;
    *d_row = *d_col = nullptr;
    *d_val = nullptr;
    DevPtr<uint32_t> offs;
    DevPtr<int32_t> row, col;
    DevPtr<double> val;
    SMVP_CUDA(dev_alloc(offs, nrows));
    SMVP_CUDA(dev_alloc(row, n));
    SMVP_CUDA(dev_alloc(col, n));
    SMVP_CUDA(dev_alloc(val, n));
    if (nrows > 0)
    {
        const unsigned blocks = (unsigned)ceil_div64(nrows, 256);
        SMVP_LAUNCH(stencil_count_kernel, blocks, 256, 0, 0, nx, ny, nz, row_begin, nrows, offs.get());
        SMVP_TRY(exclusive_scan_u32(offs.get(), offs.get(), nrows, nullptr, 0));
        SMVP_LAUNCH(stencil_fill_kernel, blocks, 256, 0, 0, nx, ny, nz, row_begin, nrows, (const uint32_t *)offs.get(), value_mode,
                    seed, row.get(), col.get(), val.get());
    }
    SMVP_CUDA(cudaDeviceSynchronize());
    SMVP_CUDA(cudaGetLastError());
    *d_row = row.release();
    *d_col = col.release();
    *d_val = val.release();
    return SMVP_OK;
}

extern "C" int smvp_synth_rmat(int scale, int64_t nedges, double a, double b, double c, int value_mode, uint64_t seed,
                               int32_t **d_row, int32_t **d_col, double **d_val, int64_t *nnz)
{
    if (!d_row || !d_col || !d_val || !nnz || scale < 1 || scale > 30 || nedges < 0 || nedges > 0x7fffffffLL - 1024)
        return SMVP_E_ARG;
    *d_row = *d_col = nullptr;
    *d_val = nullptr;
    *nnz = 0;
    DevPtr<uint64_t> key_a, key_b;
    DevPtr<uint32_t> idx_a, idx_b, d_total;
    SMVP_CUDA(dev_alloc(key_a, nedges));
    SMVP_CUDA(dev_alloc(key_b, nedges));
    SMVP_CUDA(dev_alloc(idx_a, nedges));
    SMVP_CUDA(dev_alloc(idx_b, nedges));
    SMVP_CUDA(dev_alloc(d_total, 1));
    if (nedges == 0)
        return SMVP_OK;
    SMVP_LAUNCH(rmat_edges_kernel, grid_for(nedges), 256, 0, 0, scale, nedges, a, a + b, a + b + c, seed, key_a.get(), idx_a.get());
    uint64_t *rk = nullptr;
    uint32_t *ri = nullptr;
    const int lo = 0, hi = 2 * scale;
    SMVP_TRY(radix_sort_pairs<uint64_t>(key_a.get(), idx_a.get(), key_b.get(), idx_b.get(), nedges, &lo, &hi, 1, &rk, &ri, 0));
    // the payload is not needed: reuse its spare buffer for the flags
    uint32_t *flag = (ri == idx_a.get()) ? idx_b.get() : idx_a.get();
    SMVP_LAUNCH(unique_flag_kernel, grid_for(nedges), 256, 0, 0, (const uint64_t *)rk, nedges, flag);
    SMVP_TRY(exclusive_scan_u32(flag, flag, nedges, d_total.get(), 0));
    uint32_t total = 0;
    SMVP_CUDA(cudaMemcpy(&total, d_total.get(), sizeof(total), cudaMemcpyDeviceToHost));
    *nnz = (int64_t)total;
    DevPtr<int32_t> row, col;
    DevPtr<double> val;
    SMVP_CUDA(dev_alloc(row, total));
    SMVP_CUDA(dev_alloc(col, total));
    SMVP_CUDA(dev_alloc(val, total));
    SMVP_LAUNCH(rmat_compact_kernel, grid_for(nedges), 256, 0, 0, (const uint64_t *)rk, (const uint32_t *)flag, nedges, scale,
                value_mode, seed, row.get(), col.get(), val.get());
    SMVP_CUDA(cudaDeviceSynchronize());
    *d_row = row.release();
    *d_col = col.release();
    *d_val = val.release();
    return SMVP_OK;
}

extern "C" int smvp_synth_vector(double *d_x, int64_t n, uint64_t seed, void *stream)
{
    if (n < 0 || (n > 0 && !d_x))
        return SMVP_E_ARG;
    if (n > 0)
        SMVP_LAUNCH(vector_fill_kernel, grid_for(n), 256, 0, (cudaStream_t)stream, d_x, n, seed);
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

extern "C" int smvp_coo_filter_device(const int32_t *d_row, const int32_t *d_col, const double *d_val, int64_t nnz, int32_t row_lo,
                                      int32_t row_hi, int32_t col_lo, int32_t col_hi, int32_t row_shift, int32_t col_shift,
                                      int32_t **o_row, int32_t **o_col, double **o_val, int64_t *o_nnz)
{
    if (!o_row || !o_col || !o_val || !o_nnz || nnz < 0 || (nnz > 0 && (!d_row || !d_col || !d_val)))
        return SMVP_E_ARG;
    *o_row = *o_col = nullptr;
    *o_val = nullptr;
    *o_nnz = 0;
    DevPtr<uint32_t> pos, d_total;
    SMVP_CUDA(dev_alloc(pos, nnz));
    SMVP_CUDA(dev_alloc(d_total, 1));
    uint32_t total = 0;
    if (nnz > 0)
    {
        SMVP_LAUNCH(filter_flag_kernel, grid_for(nnz), 256, 0, 0, d_row, d_col, nnz, row_lo, row_hi, col_lo, col_hi, pos.get());
        SMVP_TRY(exclusive_scan_u32(pos.get(), pos.get(), nnz, d_total.get(), 0));
        SMVP_CUDA(cudaMemcpy(&total, d_total.get(), sizeof(total), cudaMemcpyDeviceToHost));
    }
    *o_nnz = (int64_t)total;
    DevPtr<int32_t> row, col;
    DevPtr<double> val;
    SMVP_CUDA(dev_alloc(row, total));
    SMVP_CUDA(dev_alloc(col, total));
    SMVP_CUDA(dev_alloc(val, total));
    if (nnz > 0)
        SMVP_LAUNCH(filter_scatter_kernel, grid_for(nnz), 256, 0, 0, d_row, d_col, d_val, nnz, row_lo, row_hi, col_lo, col_hi,
                    row_shift, col_shift, (const uint32_t *)pos.get(), row.get(), col.get(), val.get());
    SMVP_CUDA(cudaDeviceSynchronize());
    *o_row = row.release();
    *o_col = col.release();
    *o_val = val.release();
    return SMVP_OK;
}

extern "C" int smvp_coo_histogram_device(const int32_t *d_row, const int32_t *d_col, int64_t nnz, int by_col, int32_t nkeys,
                                         uint32_t *d_counts)
{
    if (nnz < 0 || nkeys < 0 || !d_counts || (nnz > 0 && (!d_row || !d_col)))
        return SMVP_E_ARG;
    SMVP_TRY(histogram_i32(by_col ? d_col : d_row, nnz, d_counts, nkeys, 0));
    SMVP_CUDA(cudaDeviceSynchronize());
    return SMVP_OK;
}

extern "C" int smvp_vector_add_device(double *d_y, const double *d_a, int64_t n, void *stream)
{
    if (n < 0 || (n > 0 && (!d_y || !d_a)))
        return SMVP_E_ARG;
    if (n > 0)
        SMVP_LAUNCH(vector_add_kernel, grid_for(n), 256, 0, (cudaStream_t)stream, d_y, d_a, n);
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

extern "C" int smvp_copy_device(void *d_dst, const void *d_src, int64_t bytes, void *stream)
{
    if (bytes < 0 || (bytes > 0 && (!d_dst || !d_src)))
        return SMVP_E_ARG;
    if (bytes > 0)
        SMVP_CUDA(cudaMemcpyAsync(d_dst, d_src, (size_t)bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return SMVP_OK;
}

extern "C" int smvp_push_device(void *d_dst, const void *d_src, int64_t bytes, int ctas, void *stream)
{
    if (bytes < 0 || ctas < 1 || (bytes % 8) != 0 || (bytes > 0 && (!d_dst || !d_src)))
        return SMVP_E_ARG;
    if (bytes == 0)
        return SMVP_OK;
    // 16-byte vectors need both pointers 16-byte aligned; otherwise peel one double in front
    char *dst = (char *)d_dst;
    const char *src = (const char *)d_src;
    if ((((uintptr_t)dst) & 15) != (((uintptr_t)src) & 15))
        return smvp_copy_device(d_dst, d_src, bytes, stream); // mutually misaligned: let the copy engines do it
    int64_t head = (((uintptr_t)dst) & 15) ? 8 : 0;
    if (head > bytes)
        head = bytes;
    if (head)
        SMVP_CUDA(cudaMemcpyAsync(dst, src, (size_t)head, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    const int64_t body = bytes - head;
    const int64_t n16 = body / 16;
    const int tail = (int)((body % 16) / 8);
    SMVP_LAUNCH(push_kernel, (unsigned)ctas, 512, 0, (cudaStream_t)stream, (double2 *)(dst + head), (const double2 *)(src + head), n16,
                (double *)(dst + head + 16 * n16), (const double *)(src + head + 16 * n16), tail);
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

extern "C" int smvp_push_fanout_device(void *const *d_dst_list, int n_dst, const void *d_src, int64_t bytes, int ctas, void *stream)
{
    if (bytes < 0 || ctas < 1 || (bytes % 8) != 0 || n_dst < 1 || n_dst > 8 || !d_dst_list || (bytes > 0 && !d_src))
        return SMVP_E_ARG;
    if (bytes == 0)
        return SMVP_OK;
    const char *src = (const char *)d_src;
    bool aligned = true;
    for (int k = 0; k < n_dst; k++)
    {
        if (!d_dst_list[k])
            return SMVP_E_ARG;
        aligned = aligned && ((((uintptr_t)d_dst_list[k]) & 15) == (((uintptr_t)src) & 15));
    }
    if (!aligned) // mutually misaligned: one copy-engine transfer per destination
    {
        for (int k = 0; k < n_dst; k++)
            SMVP_TRY(smvp_copy_device(d_dst_list[k], d_src, bytes, stream));
        return SMVP_OK;
    }
    int64_t head = (((uintptr_t)src) & 15) ? 8 : 0;
    if (head > bytes)
        head = bytes;
    PushFan fan;
    fan.n = n_dst;
    const int64_t body = bytes - head;
    const int64_t n16 = body / 16;
    const int tail = (int)((body % 16) / 8);
    for (int k = 0; k < 8; k++)
    {
        char *dst = k < n_dst ? (char *)d_dst_list[k] : nullptr;
        fan.dst[k] = (double2 *)(dst ? dst + head : nullptr);
        fan.dst_tail[k] = (double *)(dst ? dst + head + 16 * n16 : nullptr);
        if (dst && head)
            SMVP_CUDA(cudaMemcpyAsync(dst, src, (size_t)head, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    }
    SMVP_LAUNCH(push_fanout_kernel, (unsigned)ctas, 512, 0, (cudaStream_t)stream, fan, (const double2 *)(src + head), n16,
                (const double *)(src + head + 16 * n16), tail);
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

extern "C" int smvp_push_tma_device(void *const *d_dst_list, int n_dst, const void *d_src, int64_t bytes, int ctas, void *stream)
{
    if (bytes < 0 || ctas < 1 || (bytes % 8) != 0 || n_dst < 1 || n_dst > 8 || !d_dst_list || (bytes > 0 && !d_src))
        return SMVP_E_ARG;
    if (bytes == 0)
        return SMVP_OK;
    const char *src = (const char *)d_src;
    for (int k = 0; k < n_dst; k++)
        if (!d_dst_list[k] || ((((uintptr_t)d_dst_list[k]) & 15) != (((uintptr_t)src) & 15)))
            return smvp_push_fanout_device(d_dst_list, n_dst, d_src, bytes, ctas, stream); // bulk copies need 16-byte alignment
    int64_t head = (((uintptr_t)src) & 15) ? 8 : 0;
    if (head > bytes)
        head = bytes;
    const int64_t body16 = ((bytes - head) / 16) * 16, tail = bytes - head - body16;
    PushTma fan;
    fan.n = n_dst;
    for (int k = 0; k < 8; k++)
        fan.dst[k] = k < n_dst ? (char *)d_dst_list[k] + head : nullptr;
    for (int k = 0; k < n_dst; k++)
    {
        if (head)
            SMVP_CUDA(cudaMemcpyAsync(d_dst_list[k], src, (size_t)head, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        if (tail)
            SMVP_CUDA(cudaMemcpyAsync((char *)d_dst_list[k] + head + body16, src + head + body16, (size_t)tail, cudaMemcpyDeviceToDevice,
                                      (cudaStream_t)stream));
    }
    if (body16 > 0)
    {
        constexpr int SMEM = PUSH_TMA_STAGES * PUSH_TMA_CHUNK;
        static thread_local int configured_dev = -1;
        int dev = 0;
        SMVP_CUDA(cudaGetDevice(&dev));
        if (configured_dev != dev)
        {
            SMVP_CUDA(cudaFuncSetAttribute(push_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
            // same L1 / shared-memory split as the merge-path SpMV (which needs ~200 KB of shared memory per SM): an SM
            // hosts CTAs of two kernels at once only under one split
            if (env_tristate("SMVP_PUSH_CARVEOUT") != -1)
                SMVP_CUDA(cudaFuncSetAttribute(push_tma_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                               (int)cudaSharedmemCarveoutMaxShared));
            configured_dev = dev;
        }
        const int64_t nchunks = ceil_div64(body16, PUSH_TMA_CHUNK);
        SMVP_LAUNCH(push_tma_kernel, (unsigned)(ctas < nchunks ? ctas : nchunks), 32, SMEM, (cudaStream_t)stream, fan, src + head, body16);
    }
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

extern "C" int smvp_sum_ordered_device(double *d_out, const double *d_parts, int nparts, int64_t stride, int64_t n, void *stream)
{
    if (n < 0 || nparts < 1 || stride < 0 || (n > 0 && (!d_out || !d_parts)))
        return SMVP_E_ARG;
    if (n > 0)
    {
        SMVP_LAUNCH(sum_ordered_kernel, grid_for(n), 256, 0, (cudaStream_t)stream, d_out, d_parts, nparts, stride, n);
        SMVP_CUDA(cudaGetLastError());
    }
    return SMVP_OK;
}

extern "C" int smvp_sum_ordered_ptrs_device(double *d_out, const double *const *d_part_list, int nparts, int64_t n, void *stream)
{
    if (n < 0 || nparts < 1 || nparts > 16 || !d_part_list || (n > 0 && !d_out))
        return SMVP_E_ARG;
    PartPtrs parts;
    parts.n = nparts;
    for (int k = 0; k < 16; k++)
    {
        parts.p[k] = k < nparts ? d_part_list[k] : nullptr;
        if (k < nparts && n > 0 && (!parts.p[k] || (((uintptr_t)parts.p[k]) & 15)))
            return SMVP_E_ARG; // 16-byte aligned parts (128-bit loads)
    }
    if (n > 0 && (((uintptr_t)d_out) & 15))
        return SMVP_E_ARG;
    if (n > 0)
    {
        SMVP_LAUNCH(sum_ordered_ptrs_kernel, grid_for(n, 2), 256, 0, (cudaStream_t)stream, d_out, parts, n);
        SMVP_CUDA(cudaGetLastError());
    }
    return SMVP_OK;
}

extern "C" int smvp_flush_l2(int64_t bytes, void *stream)
{
    static thread_local void *buf = nullptr;
    static thread_local int64_t cap = 0;
    if (bytes <= 0)
        return SMVP_E_ARG;
    if (cap < bytes)
    {
        cudaFree(buf);
        buf = nullptr;
        cap = 0;
        SMVP_CUDA(cudaMalloc(&buf, (size_t)bytes));
        cap = bytes;
    }
    SMVP_CUDA(cudaMemsetAsync(buf, 0, (size_t)bytes, (cudaStream_t)stream));
    return SMVP_OK;
}

extern "C" void smvp_device_free(void *d_ptr) { cudaFree(d_ptr); }
