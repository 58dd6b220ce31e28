// api.cu -- the small C-ABI entry points that are not kernels: error text, device probe,
// launch counter and the iteration statistics of struct _time_data_ (main-cli.c:87-95, :428-456).
#include "common.cuh"

#include <math.h>

using namespace smvp;

extern "C" const char *smvp_strerror(int code)
{
    switch (code)
    {
    case SMVP_OK:
        return "ok";
    case SMVP_E_ARG:
        return "invalid argument";
    case SMVP_E_ALLOC:
        return "allocation failed";
    case SMVP_E_CUDA:
        return "CUDA error (no device, or a runtime/launch failure; see smvp_last_cuda_error)";
    case SMVP_E_RANGE:
        return "matrix coordinate out of range";
    case SMVP_E_TOOBIG:
        return "problem too large for int32 offsets";
    case SMVP_E_PATTERN:
        return "entry not stored in the matrix (a value update cannot add entries)";
    default:
        return "unknown error";
    }
}

extern "C" const char *smvp_last_cuda_error(void) { return g_last_cuda_error; }

extern "C" int smvp_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess)
        return cuda_fail(e, "cudaGetDeviceCount", __FILE__, __LINE__);
    return n;
}

// page-locked host buffers for x and y (plain C callers need no CUDA header): what makes the overlapped transfers of
// smvp_csr_mult effective
extern "C" void *smvp_host_alloc(int64_t bytes)
{
    void *p = nullptr;
    if (bytes < 0 || cudaHostAlloc(&p, (size_t)(bytes > 0 ? bytes : 1), cudaHostAllocDefault) != cudaSuccess)
    {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" void smvp_host_free(void *p)
{
    if (p)
        cudaFreeHost(p);
}

extern "C" int64_t smvp_launch_count(void) { return (int64_t)g_launches.load(); }

namespace smvp
{
const char *env_str(const char *name)
{
    const char *e = getenv(name);
    return e && e[0] ? e : nullptr;
}

bool env_set(const char *name) { return getenv(name) != nullptr; }

int env_int(const char *name, int dflt, int lo, int hi)
{
    const char *e = env_str(name);
    if (!e)
        return dflt;
    const long long v = atoll(e);
    return v < lo ? lo : (v > hi ? hi : (int)v);
}

int env_tristate(const char *name)
{
    const char *e = env_str(name);
    return (e && e[0] == '1') ? 1 : (e && e[0] == '0') ? -1 : 0;
}

int timed_loop(int iters, double *ms_each, bool batched, const std::function<int(cudaStream_t)> &pass,
               const std::function<int(cudaStream_t, int)> &multi)
{
    if (iters < 1)
        return SMVP_E_ARG;
    if (env_int("SMVP_EXACT_ITER_TIMES", 0, INT32_MIN, INT32_MAX) == 1 || iters < 4)
        batched = false;
    Event e0, e1;
    SMVP_CUDA(cudaEventCreate(out(e0)));
    SMVP_CUDA(cudaEventCreate(out(e1)));
    if (batched)
    {
        // one untimed pass first: the first launch of a kernel loads its module (milliseconds), which would otherwise be
        // charged to iteration 0 of a loop whose passes last microseconds.  Every pass rewrites all of y.
        SMVP_TRY(pass(0));
        if (multi)
            SMVP_TRY(multi(0, 1));
        SMVP_CUDA(cudaStreamSynchronize(0));
    }
    // exact passes on the legacy stream, as before
    const int exact = batched ? 1 : iters;
    for (int it = 0; it < exact; it++)
    {
        cudaEventRecord(e0.get(), 0);
        const int rc = pass(0);
        cudaEventRecord(e1.get(), 0);
        if (rc != SMVP_OK)
            return rc;
        SMVP_CUDA(cudaEventSynchronize(e1.get()));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0.get(), e1.get());
        if (ms_each)
            ms_each[it] = (double)ms;
    }
    if (!batched)
        return SMVP_OK;

    // ---- the remaining passes: graphs of `batch` passes replayed back to back on a private stream
    const int rest = iters - 1;
    int batch = env_int("SMVP_LOOP_BATCH", 50, 1, INT32_MAX);
    if ((rest + batch - 1) / batch > 1024)
        batch = (rest + 1023) / 1024; // bounds the number of events
    if (batch > rest)
        batch = rest;
    const int nfull = rest / batch, tail = rest % batch;
    const int nev = nfull + (tail ? 1 : 0) + 1;
    Stream s;
    Graph g[2];
    GraphExec ge[2];
    std::unique_ptr<Event[]> ev(new (std::nothrow) Event[nev]);
    long long captured[2] = {0, 0};
    if (!ev)
        return SMVP_E_ALLOC;
    SMVP_CUDA(cudaStreamCreateWithFlags(out(s), cudaStreamNonBlocking));
    for (int k = 0; k < nev; k++)
        SMVP_CUDA(cudaEventCreate(out(ev[k])));
    for (int k = 0; k < 2; k++)
    {
        const int n = k == 0 ? batch : tail;
        if (n == 0 || (k == 0 && nfull == 0) || multi)
            continue;
        const long long before = g_launches.load();
        SMVP_CUDA(cudaStreamBeginCapture(s.get(), cudaStreamCaptureModeThreadLocal));
        int prc = SMVP_OK;
        for (int b = 0; b < n && prc == SMVP_OK; b++)
            prc = pass(s.get());
        const cudaError_t ee = cudaStreamEndCapture(s.get(), out(g[k]));
        captured[k] = g_launches.load() - before;
        g_launches.fetch_sub(captured[k]); // nothing ran yet: replays are counted below
        if (prc != SMVP_OK)
            return prc;
        SMVP_CUDA(ee);
        SMVP_CUDA(cudaGraphInstantiate(out(ge[k]), g[k].get(), 0));
    }
    int e = 0;
    SMVP_CUDA(cudaEventRecord(ev[e++].get(), s.get()));
    for (int k = 0; k < nfull; k++)
    {
        if (multi)
            SMVP_TRY(multi(s.get(), batch));
        else
        {
            SMVP_CUDA(cudaGraphLaunch(ge[0].get(), s.get()));
            g_launches.fetch_add(captured[0]);
        }
        SMVP_CUDA(cudaEventRecord(ev[e++].get(), s.get()));
    }
    if (tail)
    {
        if (multi)
            SMVP_TRY(multi(s.get(), tail));
        else
        {
            SMVP_CUDA(cudaGraphLaunch(ge[1].get(), s.get()));
            g_launches.fetch_add(captured[1]);
        }
        SMVP_CUDA(cudaEventRecord(ev[e++].get(), s.get()));
    }
    SMVP_CUDA(cudaStreamSynchronize(s.get()));
    int it = 1;
    for (int k = 0; k + 1 < nev; k++)
    {
        float ms = 0.f;
        SMVP_CUDA(cudaEventElapsedTime(&ms, ev[k].get(), ev[k + 1].get()));
        const int n = k < nfull ? batch : tail;
        for (int b = 0; b < n; b++, it++)
            if (ms_each)
                ms_each[it] = (double)ms / n;
    }
    return SMVP_OK;
}
} // namespace smvp

// total / mean / min / max and the POPULATION standard deviation the reference intends
// (calcStDevDouble, main-cli.c:114-130: sqrt(sum((t - mean)^2) / n); its accumulators are
// uninitialised there, U11 -- zero is the intended start).
extern "C" int smvp_time_stats(const double *ms_each, int n, smvp_time_stats_t *out)
{
    if (!out || n < 0 || (n > 0 && !ms_each))
        return SMVP_E_ARG;
    double total = 0.0, mn = 0.0, mx = 0.0;
    for (int i = 0; i < n; i++)
    {
        total += ms_each[i];
        if (i == 0 || ms_each[i] < mn)
            mn = ms_each[i];
        if (i == 0 || ms_each[i] > mx)
            mx = ms_each[i];
    }
    const double mean = n > 0 ? total / n : 0.0;
    double ss = 0.0;
    for (int i = 0; i < n; i++)
        ss += (ms_each[i] - mean) * (ms_each[i] - mean);
    out->time_total = total;
    out->time_avg = mean;
    out->time_stdev = n > 0 ? sqrt(ss / n) : 0.0;
    out->time_min = mn;
    out->time_max = mx;
    return SMVP_OK;
}
