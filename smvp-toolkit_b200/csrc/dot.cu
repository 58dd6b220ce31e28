// dot.cu -- the reduction of the fused inner product (the *_axpby_dot entry points, DESIGN.md §5.7).
//
// The multiply kernels leave one partial per work unit; this kernel sums them in a tree fixed by their number alone:
//   level 1: CTA b of ceil(n / 8192) takes partials [8192 b, 8192 (b+1)); thread t adds partials 8192 b + 256 i + t,
//            i = 0 .. 31, left to right from +0.0, and the 256 thread sums are added in a pairwise tree (cta_tree_sum);
//   level 2: the last CTA to finish adds the CTA sums t, t + 256, ... left to right from +0.0 in thread t, then the
//            same pairwise tree, and stores *out.
// One launch whatever n: the CTA sums meet through a counter that the last CTA resets, so the pass can be replayed
// from a CUDA graph.  Depth of the tree (the bound in smvp_cuda.h): at most 48 + ceil(n / 2^21) additions.
#include "common.cuh"

namespace smvp
{

constexpr int DOT_THREADS = 256;
constexpr int DOT_PER_THREAD = 32;
constexpr int64_t DOT_CHUNK = DOT_THREADS * DOT_PER_THREAD; // partials per CTA of level 1

static int64_t dot_ctas(int64_t units) { return units > 0 ? ceil_div64(units, DOT_CHUNK) : 1; }

__global__ void __launch_bounds__(DOT_THREADS) dot_reduce_kernel(const double *__restrict__ part, int64_t n,
                                                                 double *__restrict__ cta_sum, unsigned int *__restrict__ counter,
                                                                 double *__restrict__ out)
{
    __shared__ bool last;
    const int t = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * DOT_CHUNK + t;
    double s = 0.0;
#pragma unroll 8
    for (int i = 0; i < DOT_PER_THREAD; i++)
    {
        const int64_t k = base + (int64_t)i * DOT_THREADS;
        if (k < n)
            s = __dadd_rn(s, __ldcg(part + k)); // L2: the multiply kernels wrote these
    }
    s = cta_tree_sum<DOT_THREADS>(s);
    if (t == 0)
    {
        cta_sum[blockIdx.x] = s;
        __threadfence();
        last = atomicAdd(counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last)
        return;
    __threadfence();
    double s2 = 0.0;
    for (int64_t k = t; k < (int64_t)gridDim.x; k += DOT_THREADS)
        s2 = __dadd_rn(s2, __ldcg(cta_sum + k));
    s2 = cta_tree_sum<DOT_THREADS>(s2);
    if (t == 0)
    {
        *out = s2;
        *counter = 0u; // ready for the next pass
    }
}

// layout: [0, units) partials | [units, units + ctas) CTA sums | counter in the last double
int dot_scratch(DevPtr<double> *buf, int64_t *cap, int64_t *device_bytes, int64_t units, cudaStream_t s)
{
    const int64_t need = units + dot_ctas(units) + 1;
    if (*buf && *cap >= need)
        return SMVP_OK;
    SMVP_CUDA(cudaStreamSynchronize(s)); // an earlier dot pass on this handle may still use the old scratch
    DevPtr<double> grown;
    SMVP_CUDA(dev_alloc(grown, need));
    SMVP_CUDA(cudaMemsetAsync(grown.get(), 0, sizeof(double) * (size_t)need, s));
    *buf = std::move(grown);
    *device_bytes += 8 * (need - *cap);
    *cap = need;
    return SMVP_OK;
}

int dot_reduce(double *buf, int64_t cap, int64_t units, double *out, cudaStream_t s)
{
    const int64_t ctas = dot_ctas(units);
    if (ctas > 0x7fffffffLL)
        return SMVP_E_TOOBIG;
    SMVP_LAUNCH(dot_reduce_kernel, (unsigned)ctas, DOT_THREADS, 0, s, (const double *)buf, units, buf + units,
                reinterpret_cast<unsigned int *>(buf + cap - 1), out);
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

} // namespace smvp
