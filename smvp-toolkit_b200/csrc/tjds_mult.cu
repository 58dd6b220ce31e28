// tjds_mult.cu -- y = A x in TJDS on sm_100a.  Replaces the loop at main-cli.c:1013-1020
//
//     for d in diagonals: for j in start_pos[d] .. start_pos[d+1]:  y[row_ind[j]] += val[j] * x_perm[j - start_pos[d]]
//
// (the reference indexes x by ROW there, U7; with its x = ones that is invisible -- the intended
// index, the slot of the entry's column, is used here).
//
// Layout fact the kernels exploit: slot p of EVERY diagonal belongs to the same (permuted) column, and
// columns are sorted by length, so "thread p walks diagonals 0 .. len[p]-1 at offset p" reads val and
// row_ind fully coalesced (consecutive threads, consecutive addresses, per diagonal), keeps x_perm[p]
// in a register, and lanes of a warp have near-equal trip counts.  One launch covers all diagonals
// (never one launch per diagonal: power-law matrices have 1e5..1e6 of them).
//
//  ATOMIC         scatter with fp64 atomicAdd (RED.E.ADD.F64) into y.
//  DETERMINISTIC  same walk, but every product is split exactly into two signed 64-bit fixed-point
//                 words (scaled per row by a bound known before the multiply) and accumulated with
//                 INTEGER atomics.  Integer addition is associative, so the result is bit-identical
//                 run to run whatever order the hardware schedules the adds in; a final pass converts
//                 the 96-bit sums to fp64 (one rounding of the sum of the products truncated at
//                 2^-94 of the row bound).  Cost: two 8-byte reductions per entry instead of one, 16 B/row of
//                 accumulators to clear and read back.
#include "common.cuh"

#include <string.h>

namespace smvp
{

// The matrix streams are read with plain __ldg.  Measured on B200 and removed: ld.global.nc.L1::no_allocate streams
// lose (atomic 3.19 vs 3.12 ms, deterministic 4.12 vs 3.83 ms on the 369^3 stencil); ld.global.nc.L2::256B changed nothing.

constexpr int32_t EXP_LOW_NONE = 0x7fffffff;  // "no row bound seen" for the running minimum
constexpr int32_t EXP_NONFINITE = 0x40000000; // "an Inf or NaN was seen": above every real exponent
constexpr int TJDS_W = 32;           // bits kept in the low word
constexpr int TJDS_FRAC = 62 + TJDS_W; // value = V * 2^(T_r - TJDS_FRAC), |sum V| < 2^TJDS_FRAC

// x_exp is taken over the slots p < nslots only: the columns that hold entries, which perm puts first.  An x entry
// that A x never reads (an empty column) must not raise the row bounds of the deterministic variants (and truncate
// every row), nor send the pass to the atomic kernel when it is Inf or NaN.
__global__ void __launch_bounds__(256) tjds_permute_x_kernel(const double *__restrict__ x, const int32_t *__restrict__ perm,
                                                             int32_t cols, int32_t nslots, double *__restrict__ x_perm,
                                                             int32_t *__restrict__ x_exp)
{
    int32_t e = INT32_MIN;
    for (int32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < cols; p += gridDim.x * blockDim.x)
    {
        const double v = x[perm[p]];
        x_perm[p] = v;
        if (p >= nslots)
            continue;
        if (!isfinite(v))
            e = EXP_NONFINITE; // the deterministic variant needs finite inputs: such an x is routed to the atomic kernel
        else if (v != 0.0)
            e = max(e, ilogb(v) + 1); // |v| < 2^e
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        e = max(e, __shfl_xor_sync(0xffffffffu, e, o));
    if ((threadIdx.x & 31) == 0 && e != INT32_MIN)
        atomicMax(x_exp, e);
}

// ---- work plan: power-law matrices have columns with 1e5..1e6 entries; one thread walking such a
// column alone would serialise the whole multiply.  The (diagonal, slot) plane is therefore cut into
// segments of TJDS_SEG consecutive diagonals; segment g only needs the first L[g*TJDS_SEG] slots (the
// columns longer than g*TJDS_SEG), i.e. ceil(L/256) CTAs.  blocks[b] = {segment, first slot} is a flat
// table over all segments, built once per handle, so one launch covers everything and no thread walks
// more than TJDS_SEG entries.
//
// SKEWED WALK (round 2).  Round 1 paid one L2 read-modify-write per nonzero (ncu: 372.7 M RED sectors, the L2
// reduction path was the limiter, profiles/r01_tjds_atomic_stencil369.txt).  In a banded matrix the entries of one
// ROW sit in neighbouring columns, and the rank of that row inside column c+1 is one less than inside column c:
// (slot q, diagonal d) and (slot q-1, diagonal d+1) hold the same row.  A thread that walks the plane along that
// anti-diagonal -- slot q-i at diagonal d+i -- therefore meets RUNS of the same row, sums them in a register and
// issues one reduction per run (27-point stencil: runs of 3, a third of the reductions).  The walk is exactly as
// coalesced as the straight one (at every step consecutive threads read consecutive slots of one diagonal); the
// price is that x_perm[slot] changes per step (an L1-resident 8-byte load instead of a register).  Whether the
// matrix has such runs is probed once per handle (tjds_skew_probe_kernel); matrices without them (R-MAT) keep the
// straight walk.  SMVP_TJDS_SKEW=0/1 forces it.
constexpr int TJDS_SEG = 32;

__global__ void __launch_bounds__(256) tjds_seg_count_kernel(const int32_t *__restrict__ start_pos, int32_t ndiag, int32_t nseg,
                                                             int32_t extra, uint32_t *__restrict__ seg_nblocks)
{
    const int32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nseg)
        return;
    const int32_t d = g * TJDS_SEG;
    const int32_t L = start_pos[d + 1] - start_pos[d];
    seg_nblocks[g] = (uint32_t)(((int64_t)L + extra + 255) / 256);
}

__global__ void __launch_bounds__(256) tjds_seg_fill_kernel(const uint32_t *__restrict__ seg_first, const int32_t *__restrict__ start_pos,
                                                            int32_t nseg, int32_t extra, int2 *__restrict__ blocks)
{
    // one CTA per segment: writes that segment's run of the table
    const int32_t g = blockIdx.x;
    const int32_t d = g * TJDS_SEG;
    const int32_t L = start_pos[d + 1] - start_pos[d];
    const int32_t nb = (int32_t)(((int64_t)L + extra + 255) / 256);
    const uint32_t first = seg_first[g];
    for (int32_t i = threadIdx.x; i < nb; i += blockDim.x)
        blocks[first + i] = make_int2(g, i * 256);
}

// fraction of (slot q, diagonal d) entries whose row equals that of (slot q-1, diagonal d+1), sampled over the first
// diagonal pairs: out[0] = pairs looked at, out[1] = pairs that match
__global__ void __launch_bounds__(256) tjds_skew_probe_kernel(const int32_t *__restrict__ start_pos, const int32_t *__restrict__ row_ind,
                                                              int32_t ndiag, unsigned long long *__restrict__ out)
{
    const int32_t d = blockIdx.y;
    if (d + 1 >= ndiag)
        return;
    const int32_t s0 = start_pos[d], s1 = start_pos[d + 1], s2 = start_pos[d + 2];
    const int32_t n = min(s1 - s0 - 1, s2 - s1); // q in [1, n]
    if (n <= 0)
        return;
    const int32_t want = 1 << 18; // sampled in runs of 32 consecutive slots (one coalesced request each)
    const int32_t runs = (n + 31) / 32, stride = max(1, runs / (want / 32));
    unsigned int seen = 0, hit = 0;
    for (int32_t r = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); r * stride < runs; r += gridDim.x * (blockDim.x / 32))
    {
        const int32_t q = 1 + r * stride * 32 + (threadIdx.x & 31);
        if (q <= n)
        {
            seen++;
            hit += __ldg(row_ind + s0 + q) == __ldg(row_ind + s1 + q - 1);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
        seen += __shfl_xor_sync(0xffffffffu, seen, o);
        hit += __shfl_xor_sync(0xffffffffu, hit, o);
    }
    if ((threadIdx.x & 31) == 0 && seen)
    {
        atomicAdd(out, (unsigned long long)seen);
        atomicAdd(out + 1, (unsigned long long)hit);
    }
}

// One CTA = 256 consecutive slots x up to TJDS_SEG diagonals.  Step i of thread t looks at diagonal d_begin + i, slot
// first + t - (SKEW ? i : 0).  The segment's start_pos entries are staged in shared memory (they are warp-uniform).
template <int UNROLL, bool SKEW>
__global__ void __launch_bounds__(256) tjds_atomic_kernel(const int2 *__restrict__ blocks, const int32_t *__restrict__ start_pos,
                                                          const int32_t *__restrict__ row_ind, const double *__restrict__ val,
                                                          const double *__restrict__ x_perm, double *__restrict__ y, int32_t nslots,
                                                          int32_t diag_limit)
{
    __shared__ int32_t s_sp[TJDS_SEG + 1];
    const int2 blk = __ldg(blocks + blockIdx.x);
    const int32_t d_begin = blk.x * TJDS_SEG;
    const int32_t nd = min(TJDS_SEG, diag_limit - d_begin); // diagonals of this segment to walk
    if (nd <= 0)
        return;
    if ((int32_t)threadIdx.x <= nd)
        s_sp[threadIdx.x] = __ldg(start_pos + d_begin + threadIdx.x);
    __syncthreads();
    const int32_t q0 = blk.y + (int32_t)threadIdx.x;
    double xq = 0.0;
    if (!SKEW)
    {
        if (q0 >= nslots)
            return;
        xq = __ldg(x_perm + q0);
    }
    double acc = 0.0;
    int32_t acc_row = -1;
    for (int32_t i0 = 0; i0 < nd; i0 += UNROLL)
    {
        int32_t r[UNROLL];
        double v[UNROLL], xv[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; u++)
        {
            const int32_t i = i0 + u;
            r[u] = -1;
            v[u] = 0.0;
            xv[u] = xq;
            if (i < nd)
            {
                const int32_t sp = s_sp[i], q = SKEW ? q0 - i : q0;
                if ((uint32_t)q < (uint32_t)(s_sp[i + 1] - sp))
                {
                    const int32_t j = sp + q;
                    r[u] = __ldg(row_ind + j);
                    v[u] = __ldg(val + j);
                    if (SKEW)
                        xv[u] = __ldg(x_perm + q);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; u++)
        {
            if (r[u] >= 0)
            {
                const double p = __dmul_rn(v[u], xv[u]);
                if (!SKEW)
                    atomicAdd(y + r[u], p); // a column never holds a row twice: nothing to merge on the straight walk
                else if (r[u] == acc_row)
                    acc = __dadd_rn(acc, p);
                else
                {
                    if (acc_row >= 0)
                        atomicAdd(y + acc_row, acc);
                    acc_row = r[u];
                    acc = p;
                }
            }
        }
    }
    if (acc_row >= 0)
        atomicAdd(y + acc_row, acc);
}

// Tiny matrices (the reference's sample-data files): the `-n` loop itself runs on the device, ONE CTA repeating the
// whole multiply `passes` times (zero-fill of y, straight walk with atomicAdd, block barrier) -- see
// csr_tiny_loop_kernel in csr_mult.cu for the rationale.  Plain loads after each barrier: every pass re-reads the
// arrays (from L1) and re-accumulates y.  Only reachable from the batched `-n` loop of smvp_tjds_mult, atomic variant.
constexpr int TJDS_TINY_THREADS = 512;
__global__ void __launch_bounds__(TJDS_TINY_THREADS) tjds_tiny_loop_kernel(const int32_t *start_pos, const int32_t *slot_len,
                                                                           const int32_t *row_ind, const double *val, const double *x_perm,
                                                                           double *y, int32_t rows, int32_t nslots, int32_t diag_limit,
                                                                           int passes)
{
    for (int p = 0; p < passes; p++)
    {
        for (int32_t r = threadIdx.x; r < rows; r += TJDS_TINY_THREADS)
            y[r] = 0.0;
        __syncthreads();
        for (int32_t q = threadIdx.x; q < nslots; q += TJDS_TINY_THREADS)
        {
            const int32_t len = min(slot_len[q], diag_limit);
            const double xq = x_perm[q];
            for (int32_t d = 0; d < len; d++)
            {
                const int32_t j = start_pos[d] + q;
                atomicAdd(y + row_ind[j], __dmul_rn(val[j], xq));
            }
        }
        __syncthreads();
    }
}

// ---- deterministic variant --------------------------------------------------------------------
// row_exp[r] = ea_r + cb_r where |a_rj| < 2^ea_r for every entry of row r and the row holds at most
// 2^cb_r entries.  With |x_c| < 2^ex every partial sum of row r is below 2^(row_exp[r] + ex) = 2^T_r.
__global__ void __launch_bounds__(256) tjds_row_bound_kernel(const int32_t *__restrict__ row_ind, const double *__restrict__ val,
                                                             int64_t nnz, int32_t *__restrict__ row_maxexp, uint32_t *__restrict__ row_cnt,
                                                             int32_t *__restrict__ flags)
{
    bool bad = false;
    int32_t rmin = 0x7fffffff, rmax = -1;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nnz; j += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t r = row_ind[j];
        const double v = val[j];
        rmin = min(rmin, r);
        rmax = max(rmax, r);
        atomicAdd(row_cnt + r, 1u);
        if (!isfinite(v))
            bad = true;
        else if (v != 0.0)
            atomicMax(row_maxexp + r, ilogb(v) + 1);
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0)
        atomicOr(flags, 1); // flags[0] bit 0: the matrix holds an Inf or NaN
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
        rmin = min(rmin, __shfl_xor_sync(0xffffffffu, rmin, o));
        rmax = max(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
    }
    if ((threadIdx.x & 31) == 0 && rmax >= 0)
    {
        atomicMin(flags + 3, rmin); // flags[3], flags[4]: first / last row that holds an entry (the column block of one GPU
        atomicMax(flags + 4, rmax); // out of N of a banded matrix touches ~1/N of the rows)
    }
}

__global__ void __launch_bounds__(256) tjds_row_exp_kernel(int32_t *__restrict__ row_exp, const uint32_t *__restrict__ row_cnt, int32_t rows,
                                                           int32_t *__restrict__ flags)
{
    const int32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    int32_t out = EXP_NONE;
    if (r < rows)
    {
        const uint32_t c = row_cnt[r];
        const int32_t cb = c <= 1 ? 0 : 32 - __clz(c - 1); // ceil(log2(c))
        const int32_t e = row_exp[r];
        out = (e == EXP_NONE) ? EXP_NONE : e + cb;
        row_exp[r] = out;
        if (c > 0 && e == EXP_NONE)
            atomicOr(flags, 2); // flags[0] bit 1: a row holds entries but no nonzero value
    }
    int32_t lo = out == EXP_NONE ? EXP_LOW_NONE : out;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
        out = max(out, __shfl_xor_sync(0xffffffffu, out, o));
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    }
    if ((threadIdx.x & 31) == 0 && out != EXP_NONE)
    {
        atomicMax(flags + 1, out); // flags[1]: largest row bound (pre-set to EXP_NONE)
        atomicMin(flags + 2, lo);  // flags[2]: smallest row bound (pre-set to EXP_LOW_NONE)
    }
}

// exact split of one fp64 product into (hi, lo) fixed-point words for a row with bound 2^T
__device__ __forceinline__ void fixed_split(double prod, int32_t T, long long *hi, long long *lo)
{
    *hi = 0;
    *lo = 0;
    if (prod == 0.0)
        return;
    const long long bits = __double_as_longlong(prod);
    const int32_t be = (int32_t)((bits >> 52) & 0x7ff);
    unsigned long long m = (unsigned long long)bits & 0xfffffffffffffULL;
    int32_t e; // prod = m * 2^e
    if (be == 0)
        e = -1074;
    else
    {
        m |= 1ULL << 52;
        e = be - 1075;
    }
    const int32_t s = e - (T - TJDS_FRAC); // V = m * 2^s, |V| < 2^TJDS_FRAC
    unsigned long long hm, lm;
    if (s >= TJDS_W)
    {
        hm = m << (s - TJDS_W);
        lm = 0;
    }
    else if (s >= 0)
    {
        hm = m >> (TJDS_W - s);
        lm = (m << s) & ((1ULL << TJDS_W) - 1ULL);
    }
    else if (s > -64)
    {
        const unsigned long long t = m >> (-s); // bits below 2^(T-94) are dropped (far below fp64 resolution of the row)
        hm = t >> TJDS_W;
        lm = t & ((1ULL << TJDS_W) - 1ULL);
    }
    else
    {
        hm = 0;
        lm = 0;
    }
    const bool neg = bits < 0;
    *hi = neg ? -(long long)hm : (long long)hm;
    *lo = neg ? -(long long)lm : (long long)lm;
}

// Fast exact split for the common exponent range: with S = 2^(TJDS_FRAC - T) (a normal fp64 power of two),
//   s = prod * S           exact (power-of-two scaling, |s| < 2^TJDS_FRAC; a result below 2^-1022 truncates to 0 anyway)
//   hi = trunc(s * 2^-W)   F2I toward zero
//   lo = trunc(s - hi*2^W) the fma is exact: hi has at most 53 significant bits and the difference is the low part of s
// Same (hi, lo) as fixed_split -- magnitude truncated toward zero, both words signed like the product -- in three
// fp64 operations and three conversions instead of ~40 integer instructions (round 1: 3.0 G warp instructions per
// SpMV, issue-bound; profiles/r01_tjds_det_stencil369.txt).
__device__ __forceinline__ void fixed_split_fast(double prod, double S, long long *hi, long long *lo)
{
    const double s = __dmul_rn(prod, S);
    const long long h = __double2ll_rz(__dmul_rn(s, 1.0 / 4294967296.0));
    *hi = h;
    *lo = __double2ll_rz(__fma_rn(__ll2double_rn(h), -4294967296.0, s));
}
// T for which 2^(TJDS_FRAC - T) is a normal fp64: TJDS_FRAC - T in [-1022, 1023]
__device__ __forceinline__ bool fast_scale_ok(int32_t T) { return T >= TJDS_FRAC - 1023 && T <= TJDS_FRAC + 1022; }
__device__ __forceinline__ double pow2_f64(int32_t e) { return __hiloint2double((1023 + e) << 20, 0); }

// Same walk as tjds_atomic_kernel; a run of equal rows accumulates its (hi, lo) words in registers (integer, exact:
// |sum hi| < 2^62 by the row bound, a run adds at most TJDS_SEG lo words of 32 bits) and is flushed with two integer
// reductions.  Integer addition is associative, so neither the run boundaries nor the scheduling change the result.
// FAST: the host has checked (tjds_det_route) that every row bound T lies in the range of fixed_split_fast and that
// no visited row lacks an exponent, so the per-entry "is the product zero / which split" tests and the 60-instruction
// general split disappear from the loop.  Both instantiations produce the same words, hence the same bits of y.
// WORDS = 2 (SMVP_TJDS_DETERMINISTIC): a product keeps its bits down to 2^(T - 94), the accumulated words are converted
//            with one rounding (fixed_to_double): y is the correctly rounded row sum when no product has bits below
//            that grid, and within count * 2^(T - 94) of it otherwise (the exact contract is in smvp_cuda.h).
// WORDS = 1 (SMVP_TJDS_DETERMINISTIC_FAST): only the high word, scaled to 2^(T - 62): a product loses the bits below 2^-62
//            of its row's bound (2^-9 of what one fp64 addition at that magnitude rounds away); the sum of the integers
//            is still associative, so the result is just as reproducible; one 8-byte reduction and one conversion per
//            run instead of two, half the accumulator traffic.  The bound is normwise (see smvp_cuda.h).
// Tried and dropped (profiles/r02_logs/r02_tjds_sweep4.log): prefetch.global.L2 of the next round (3.62 -> 3.87 ms),
// ld.global.nc.L1::no_allocate streams (3.62 -> 3.75 ms), 5 or 7 CTAs per SM (4.1 / 3.9 ms), 3-deep rounds at 8 CTAs (4.0 ms).
constexpr int TJDS_MAX_UNROLL = 8;
template <int UNROLL, bool SKEW, bool FAST, int MINB, int WORDS>
__global__ void __launch_bounds__(256, MINB) tjds_det_kernel(const int2 *__restrict__ blocks, const int32_t *__restrict__ start_pos,
                                                       const int32_t *__restrict__ row_ind, const double *__restrict__ val,
                                                       const double *__restrict__ x_perm, const int32_t *__restrict__ row_exp,
                                                       const int32_t *__restrict__ x_exp, unsigned long long *__restrict__ acc,
                                                       int32_t rows, int32_t nslots, int32_t diag_limit)
{
    static_assert(UNROLL <= TJDS_MAX_UNROLL, "s_sp padding");
    __shared__ int32_t s_sp[TJDS_SEG + TJDS_MAX_UNROLL + 1];
    const int2 blk = __ldg(blocks + blockIdx.x);
    const int32_t d_begin = blk.x * TJDS_SEG;
    const int32_t nd = min(TJDS_SEG, diag_limit - d_begin);
    if (nd <= 0)
        return;
    // entries past the last diagonal repeat its end: such a diagonal is empty, so the loop needs no "i < nd" test
    if ((int32_t)threadIdx.x <= TJDS_SEG + TJDS_MAX_UNROLL)
        s_sp[threadIdx.x] = __ldg(start_pos + d_begin + min((int32_t)threadIdx.x, nd));
    __syncthreads();
    const int32_t q0 = blk.y + (int32_t)threadIdx.x;
    double xq = 0.0;
    if (!SKEW)
    {
        if (q0 >= nslots)
            return;
        xq = __ldg(x_perm + q0);
    }
    const int32_t ex = __ldg(x_exp);
    long long hi_acc = 0, lo_acc = 0;
    int32_t acc_row = -1, T = 0;
    double S = 0.0;
    auto flush = [&]() {
        if (hi_acc != 0)
            atomicAdd(acc + acc_row, (unsigned long long)hi_acc); // hi words [0, rows), lo words [rows, 2 rows):
        if (WORDS == 2 && lo_acc != 0)
            atomicAdd(acc + (int64_t)rows + acc_row, (unsigned long long)lo_acc); // a warp's reductions stay contiguous
    };
    constexpr int FRAC = WORDS == 2 ? TJDS_FRAC : TJDS_FRAC - TJDS_W; // scale of the word(s) kept
    for (int32_t i0 = 0; i0 < nd; i0 += UNROLL)
    {
        int32_t r[UNROLL];
        double v[UNROLL], xv[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; u++)
        {
            // unconditional loads: a slot outside the diagonal reads entry 0 (in bounds, cached) and is marked dead
            const int32_t i = i0 + u;
            const int32_t sp = s_sp[i], q = SKEW ? q0 - i : q0;
            const bool live = (uint32_t)q < (uint32_t)(s_sp[i + 1] - sp);
            const int32_t j = live ? sp + q : 0;
            r[u] = __ldg(row_ind + j);
            v[u] = __ldg(val + j);
            xv[u] = SKEW ? __ldg(x_perm + (live ? q : 0)) : xq;
            if (!live)
                r[u] = -1;
        }
#pragma unroll
        for (int u = 0; u < UNROLL; u++)
        {
            double p = __dmul_rn(v[u], xv[u]);
            if (FAST)
            {
                if (r[u] >= 0 && r[u] != acc_row)
                {
                    if (acc_row >= 0)
                        flush();
                    acc_row = r[u];
                    hi_acc = lo_acc = 0;
                    S = pow2_f64(FRAC - (__ldg(row_exp + acc_row) + ex));
                }
                if (r[u] < 0)
                    p = 0.0; // dead slot: adds nothing to the current run
                if (WORDS == 2)
                {
                    long long hi, lo;
                    fixed_split_fast(p, S, &hi, &lo);
                    hi_acc += hi;
                    lo_acc += lo;
                }
                else
                    hi_acc += __double2ll_rz(__dmul_rn(p, S)); // == the high word of the two-word split
            }
            else if (r[u] >= 0 && p != 0.0)
            {
                if (r[u] != acc_row)
                {
                    if (acc_row >= 0)
                        flush();
                    acc_row = r[u];
                    hi_acc = lo_acc = 0;
                    T = __ldg(row_exp + acc_row) + ex;
                    S = fast_scale_ok(T) ? pow2_f64(TJDS_FRAC - T) : 0.0;
                }
                long long hi, lo;
                if (S != 0.0)
                    fixed_split_fast(p, S, &hi, &lo);
                else
                    fixed_split(p, T, &hi, &lo);
                hi_acc += hi;
                if (WORDS == 2)
                    lo_acc += lo;
            }
        }
    }
    if (acc_row >= 0)
        flush();
}

// Calls store(i) for the rows i in [0, n) of y, store returning the row's dot term.  Dot: one row per thread, so that
// the work unit is the CTA's 256 rows whatever the grid; their terms are added in a pairwise tree into part[blockIdx.x].
// The other modes: a grid-stride loop.
template <YStore M, typename F>
__device__ __forceinline__ void for_rows_of_y(int32_t n, double *__restrict__ part, F &&store)
{
    if constexpr (M == YStore::Dot)
    {
        const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        double d = 0.0;
        if (i < n)
            d = __dadd_rn(d, store(i));
        d = cta_tree_sum<256>(d);
        if (threadIdx.x == 0)
            part[blockIdx.x] = d;
    }
    else
        for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
            store(i);
}

// V * 2^E with V = hi * 2^W + lo, rounded ONCE to nearest even fp64, subnormal results included (they round at
// 2^-1074).  Converting hi on its own and adding lo would round twice when hi has more than 53 significant bits (a row
// sum near its bound).  Common case, E >= -1022: V = H * 2^W + L with 0 <= L < 2^W; a = fl(H) and H - a are exact
// (|H - a| <= 2^10), so V = a * 2^W + r with r = (H - a) * 2^W + L exact in fp64 (|r| < 2^43): the one fp64 addition
// rounds V once, and |fl(V)| >= 1 makes the scaling by 2^E exact.  Below that the result may be subnormal and is rounded
// from V as a 128-bit integer: its leading 53 bits are kept (fewer for a subnormal result), the dropped bits round; with
// q the kept bits and 2^k the weight of the lowest, the fp64 bit pattern is ((k + 1074) << 52) + q for normal and
// subnormal results alike (a carry of q into bit 53 moves the exponent).  Rows with T < -928 take this path, and their
// normal results do round here.  A subnormal result is in fact always exact: every product is a multiple of 2^-1074,
// so a grid 2^E finer than that truncates nothing, and a coarser one has E > -1074.  Its rounding branch (and
// shift > 96) only keep the function correct for any (hi, lo, E).  The row bound keeps the result below the overflow
// threshold (tjds_det_route).
__device__ __forceinline__ double fixed_to_double(long long hi, long long lo, int32_t E)
{
    if (E >= -1022)
    {
        const long long H = hi + (lo >> TJDS_W), L = lo & ((1LL << TJDS_W) - 1);
        const double a = __ll2double_rn(H);
        const long long r = (H - __double2ll_rz(a)) * (1LL << TJDS_W) + L;
        return __dmul_rn(__dadd_rn(__dmul_rn(a, 4294967296.0), __ll2double_rn(r)), pow2_f64(E));
    }
    const __int128 v = (__int128)hi * ((__int128)1 << TJDS_W) + lo;
    if (v == 0)
        return 0.0;
    const bool neg = v < 0;
    const unsigned __int128 m = (unsigned __int128)(neg ? -v : v);
    const unsigned long long mh = (unsigned long long)(m >> 64), ml = (unsigned long long)m;
    const int32_t n = mh ? 128 - __clzll((long long)mh) : 64 - __clzll((long long)ml); // bits of m
    const int32_t shift = max(n - 53, -1074 - E);                                     // low bits of m dropped
    unsigned long long q;
    if (shift <= 0)
        q = ml << -shift; // m < 2^53: exact
    else if (shift > 96)
        q = 0; // m * 2^E < 2^-1075: rounds to zero
    else
    {
        q = (unsigned long long)(m >> shift);
        const unsigned __int128 rem = m - ((unsigned __int128)q << shift), half = (unsigned __int128)1 << (shift - 1);
        q += (rem > half || (rem == half && (q & 1))) ? 1 : 0;
    }
    const unsigned long long bits = ((unsigned long long)(E + shift + 1074) << 52) + q;
    return __longlong_as_double((long long)(neg ? bits | (1ULL << 63) : bits));
}

// row_rank != NULL: the accumulators and row_exp are in popularity-rank order (relabelled handle), y is not.
// Returns the row's dot term (store_row).  Dot: the work unit is the CTA's 256 rows of y; their dot terms are added in a
// pairwise tree.
template <YStore M>
__device__ __forceinline__ double tjds_det_finalize_row(int32_t row, const long long *__restrict__ acc, const int32_t *__restrict__ row_exp,
                                                        const int32_t *__restrict__ x_exp, int32_t rows, double *__restrict__ y,
                                                        const int32_t *__restrict__ row_rank, int words, int32_t r_lo, int32_t r_hi,
                                                        double alpha, double beta, const double *__restrict__ w)
{
    // accumulators exist (are cleared and filled) only for rows [r_lo, r_hi) of the index space the kernels use
    const int32_t r = row_rank ? row_rank[row] : row;
    if (r < r_lo || r >= r_hi)
        return store_row<M>(y, row, 0.0, alpha, beta, w);
    const long long hi = acc[r];
    const long long lo = words == 2 ? acc[(int64_t)rows + r] : 0; // one word: the value is hi * 2^(T - 62), i.e. lo = 0 below
    double out = 0.0;
    if (hi != 0 || lo != 0)
        out = fixed_to_double(hi, lo, row_exp[r] + *x_exp - TJDS_FRAC);
    return store_row<M>(y, row, out, alpha, beta, w);
}
template <YStore M>
__global__ void __launch_bounds__(256) tjds_det_finalize_kernel(const long long *__restrict__ acc, const int32_t *__restrict__ row_exp,
                                                                const int32_t *__restrict__ x_exp, int32_t rows, double *__restrict__ y,
                                                                const int32_t *__restrict__ row_rank, int words, int32_t r_lo, int32_t r_hi,
                                                                double alpha, double beta, const double *__restrict__ w,
                                                                double *__restrict__ part)
{
    const int32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    double d = 0.0;
    if (row < rows)
        d = tjds_det_finalize_row<M>(row, acc, row_exp, x_exp, rows, y, row_rank, words, r_lo, r_hi, alpha, beta, w);
    if constexpr (M == YStore::Dot)
    {
        d = cta_tree_sum<256>(d);
        if (threadIdx.x == 0)
            part[blockIdx.x] = d;
    }
}

// y[r] = y_rel[rank[r]]: the atomic variant of a relabelled handle sums in rank order.  Axpby / Dot: y[r] = alpha *
// y_rel[rank[r]] + beta * y[r] (axpby, common.cuh), and row_rank == NULL stands for the identity (the atomic sums of a
// natural-order handle, which land in a scratch vector under the epilogue).
template <YStore M>
__global__ void __launch_bounds__(256) tjds_unrank_y_kernel(const double *__restrict__ y_rel, const int32_t *__restrict__ row_rank,
                                                            int32_t rows, double *__restrict__ y, double alpha, double beta,
                                                            const double *__restrict__ w, double *__restrict__ part)
{
    for_rows_of_y<M>(rows, part, [&](int32_t r) {
        const int32_t k = M == YStore::Plain || row_rank ? __ldg(row_rank + r) : r; // Plain: only relabelled handles
        return store_row<M>(y, r, __ldg(y_rel + k), alpha, beta, w);
    });
}

// ---- transposed product y = A^T x --------------------------------------------------------------------------------
// Slot q of every diagonal belongs to column perm[q], and the d-th entry of a column is its d-th by row, so
//     (A^T x)[perm[q]] = sum_d val[start_pos[d] + q] * x[row_ind[start_pos[d] + q]]
// is a GATHER along the slot: the streams of tjds_atomic_kernel, no atomics, the terms in ascending row order.  The
// handle's segment table (tjds_plan) cuts a column into chunks of TJDS_SEG entries; thread (segment g, slot q) sums its
// chunk left to right from +0.0.  A column of at most TJDS_SEG entries (every column of the 27-point stencil) is done
// there, bit-identical to the sequential transposed loop, and a pass is one launch.  The chunk sums of a longer column
// go to tr_part[tr_seg_off[g] + q] (one coalesced store per warp) and tjds_transpose_combine_kernel adds them in
// segment order.  The table is walked straight whatever walk A x uses: a skewed table only has extra slots past the
// end of each segment's first diagonal, and those threads find nothing to do.  row_ind is read, never row_rel.
// Axpby / Dot: every store of a column's value s goes through the epilogue (store_row), empty columns too (s = +0.0).
// Dot: a CTA of either kernel is a work unit.  A thread adds the dot terms of the columns it stores in the order it stores
// them, and the CTA's threads are added in a pairwise tree into dot_part[unit].
constexpr int TJDS_TR_UNROLL = 8; // entries whose loads are issued before the first of them is used
template <YStore M>
__global__ void __launch_bounds__(256) tjds_transpose_kernel(const int2 *__restrict__ blocks, const int32_t *__restrict__ start_pos,
                                                             const int32_t *__restrict__ row_ind, const double *__restrict__ val,
                                                             const int32_t *__restrict__ perm, const double *__restrict__ x,
                                                             double *__restrict__ y, double *__restrict__ part,
                                                             const uint32_t *__restrict__ seg_off, int32_t ndiag, int32_t nslots,
                                                             int32_t cols, int32_t nlong, double alpha, double beta,
                                                             const double *__restrict__ dot_w, double *__restrict__ dot_part)
{
    static_assert(TJDS_SEG % TJDS_TR_UNROLL == 0, "s_sp holds TJDS_SEG + 1 entries");
    __shared__ int32_t s_sp[TJDS_SEG + 1];
    double d = 0.0; // Dot: this thread's dot terms
    // empty columns (slots nslots .. cols-1) get +0.0, spread over the whole grid
    for (int64_t p = (int64_t)nslots + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < cols; p += (int64_t)gridDim.x * blockDim.x)
        d = __dadd_rn(d, store_row<M>(y, __ldg(perm + p), 0.0, alpha, beta, dot_w));
    const int2 blk = __ldg(blocks + blockIdx.x);
    const int32_t d_begin = blk.x * TJDS_SEG;
    const int32_t nd = min(TJDS_SEG, ndiag - d_begin);
    // entries past the segment's last diagonal repeat its end: such a diagonal is empty
    if ((int32_t)threadIdx.x <= TJDS_SEG)
        s_sp[threadIdx.x] = __ldg(start_pos + d_begin + min((int32_t)threadIdx.x, nd));
    __syncthreads();
    const int32_t q = blk.y + (int32_t)threadIdx.x;
    const bool has = q < s_sp[1] - s_sp[0];
    if (M != YStore::Dot && !has)
        return; // the column at this slot ends before the segment (or the slot is past the table's diagonals)
    double s = 0.0;
    for (int32_t i0 = 0; has && i0 < nd; i0 += TJDS_TR_UNROLL)
    {
        int32_t r[TJDS_TR_UNROLL];
        double v[TJDS_TR_UNROLL], xv[TJDS_TR_UNROLL];
#pragma unroll
        for (int u = 0; u < TJDS_TR_UNROLL; u++)
        {
            const int32_t i = i0 + u, sp = s_sp[i];
            const bool live = q < s_sp[i + 1] - sp;
            r[u] = live ? __ldg(row_ind + sp + q) : -1;
            v[u] = live ? __ldg(val + sp + q) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < TJDS_TR_UNROLL; u++)
            xv[u] = r[u] >= 0 ? __ldg(x + r[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < TJDS_TR_UNROLL; u++)
            if (r[u] >= 0)
                s = __dadd_rn(s, __dmul_rn(v[u], xv[u]));
    }
    if (has && q >= nlong) // a column of at most TJDS_SEG entries lives in segment 0 alone
        d = __dadd_rn(d, store_row<M>(y, __ldg(perm + q), s, alpha, beta, dot_w));
    else if (has)
        part[(int64_t)__ldg(seg_off + blk.x) + q] = s;
    if constexpr (M == YStore::Dot)
    {
        d = cta_tree_sum<256>(d);
        if (threadIdx.x == 0)
            dot_part[blockIdx.x] = d;
    }
}
// y[perm[q]] = tr_part partials of long column q added left to right from +0.0, chunk 0 first.  Slots [0, nwide) hold
// more than TJDS_SEG chunks (a power-law column can hold ~1e6 entries, ~3e4 chunks): a warp loads 32 chunk sums per
// round, TJDS_TR_ROUNDS rounds ahead, and every lane adds them in order from shuffles (the additions are the serial
// part, the loads are not).  Slots [nwide, nlong) take one thread each.
constexpr int TJDS_TR_ROUNDS = 4;
template <YStore M>
__global__ void __launch_bounds__(256) tjds_transpose_combine_kernel(const double *__restrict__ part, const uint32_t *__restrict__ seg_off,
                                                                     const int32_t *__restrict__ slot_len, const int32_t *__restrict__ perm,
                                                                     int32_t nlong, int32_t nwide, double *__restrict__ y, double alpha,
                                                                     double beta, const double *__restrict__ dot_w,
                                                                     double *__restrict__ dot_part)
{
    double d = 0.0; // Dot: this thread's dot term
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, wide_threads = (int64_t)nwide * 32;
    if (t < wide_threads)
    {
        // whole warps: wide_threads is a multiple of 32
        const int32_t q = (int32_t)(t >> 5), lane = threadIdx.x & 31;
        const int32_t nch = (__ldg(slot_len + q) + TJDS_SEG - 1) / TJDS_SEG;
        double s = 0.0;
        for (int32_t g0 = 0; g0 < nch; g0 += 32 * TJDS_TR_ROUNDS)
        {
            double v[TJDS_TR_ROUNDS];
#pragma unroll
            for (int k = 0; k < TJDS_TR_ROUNDS; k++)
            {
                const int32_t g = g0 + 32 * k + lane;
                v[k] = g < nch ? __ldg(part + __ldg(seg_off + g) + q) : 0.0;
            }
#pragma unroll
            for (int k = 0; k < TJDS_TR_ROUNDS; k++)
#pragma unroll 8
                for (int l = 0; l < 32; l++)
                {
                    const double c = __shfl_sync(0xffffffffu, v[k], l);
                    if (g0 + 32 * k + l < nch)
                        s = __dadd_rn(s, c);
                }
        }
        if (lane == 0)
            d = __dadd_rn(d, store_row<M>(y, __ldg(perm + q), s, alpha, beta, dot_w));
        if (M != YStore::Dot)
            return;
    }
    else
    {
        const int64_t qq = (int64_t)nwide + (t - wide_threads);
        if (M != YStore::Dot && qq >= nlong)
            return;
        if (qq < nlong)
        {
            const int32_t q = (int32_t)qq;
            const int32_t nch = (__ldg(slot_len + q) + TJDS_SEG - 1) / TJDS_SEG;
            double s = 0.0;
#pragma unroll 4
            for (int32_t g = 0; g < nch; g++)
                s = __dadd_rn(s, __ldg(part + __ldg(seg_off + g) + q));
            d = __dadd_rn(d, store_row<M>(y, __ldg(perm + q), s, alpha, beta, dot_w));
        }
    }
    if constexpr (M == YStore::Dot)
    {
        d = cta_tree_sum<256>(d);
        if (threadIdx.x == 0)
            dot_part[blockIdx.x] = d;
    }
}
// y = alpha * (+0.0) + beta * y: the scaled, accumulating transposed product of a handle without entries (Axpby, Dot)
template <YStore M>
__global__ void __launch_bounds__(256) tjds_axpby_empty_kernel(double *__restrict__ y, int32_t n, double alpha, double beta,
                                                               const double *__restrict__ w, double *__restrict__ part)
{
    for_rows_of_y<M>(n, part, [&](int32_t i) { return store_row<M>(y, i, 0.0, alpha, beta, w); });
}

// partials segment g holds: the long columns (slots [0, nlong), nlong = length of diagonal TJDS_SEG) in segment 0, the
// columns that reach its first diagonal in every later one
__global__ void __launch_bounds__(256) tjds_transpose_count_kernel(const int32_t *__restrict__ start_pos, int32_t nseg,
                                                                   uint32_t *__restrict__ count)
{
    const int32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nseg)
        return;
    const int32_t d = g == 0 ? TJDS_SEG : g * TJDS_SEG;
    count[g] = (uint32_t)(start_pos[d + 1] - start_pos[d]);
}

// the row indices the kernels scatter through: the relabelled copy when that plan is in use (relabel.cu)
static inline const int32_t *mult_rows(const smvp_tjds *A) { return A->relabel_state == 1 ? A->row_rel.get() : A->row_ind.get(); }

// decides the walk (once per handle) and builds the block table for it.  Synchronous.
static int tjds_plan(smvp_tjds *A, cudaStream_t s)
{
    if (A->seg_blocks || A->ndiag == 0)
        return SMVP_OK;
    int32_t skew = A->skew;
    if (skew == 0)
    {
        skew = env_tristate("SMVP_TJDS_SKEW");
        if (skew == 0 && A->ndiag >= 2)
        {
            DevPtr<unsigned long long> probe;
            SMVP_CUDA(dev_alloc(probe, 2));
            SMVP_CUDA(cudaMemsetAsync(probe.get(), 0, 2 * sizeof(unsigned long long), s));
            const int pairs = A->ndiag - 1 < 8 ? A->ndiag - 1 : 8;
            SMVP_LAUNCH(tjds_skew_probe_kernel, dim3(64, pairs), 256, 0, s, (const int32_t *)A->start_pos.get(),
                        (const int32_t *)A->row_ind.get(), A->ndiag, probe.get());
            unsigned long long h[2] = {0, 0};
            SMVP_CUDA(cudaMemcpyAsync(h, probe.get(), sizeof(h), cudaMemcpyDeviceToHost, s));
            SMVP_CUDA(cudaStreamSynchronize(s));
            // worth it when at least a quarter of the looked-at entries continue a run (the x_perm load per step has
            // to be paid for by saved reductions)
            skew = (h[0] >= 1024 && 4 * h[1] >= h[0]) ? 1 : -1;
        }
        else if (skew == 0)
            skew = -1;
    }
    const int32_t extra = skew == 1 ? TJDS_SEG - 1 : 0; // the skewed walk of the last block leans TJDS_SEG-1 slots back
    const int32_t nseg = (A->ndiag + TJDS_SEG - 1) / TJDS_SEG;
    DevPtr<uint32_t> seg_nb, d_total;
    SMVP_CUDA(dev_alloc(seg_nb, nseg));
    SMVP_CUDA(dev_alloc(d_total, 1));
    SMVP_LAUNCH(tjds_seg_count_kernel, (unsigned)ceil_div64(nseg, 256), 256, 0, s, (const int32_t *)A->start_pos.get(), A->ndiag, nseg,
                extra, seg_nb.get());
    SMVP_TRY(exclusive_scan_u32(seg_nb.get(), seg_nb.get(), nseg, d_total.get(), s));
    uint32_t total = 0;
    SMVP_CUDA(cudaMemcpyAsync(&total, d_total.get(), sizeof(total), cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaStreamSynchronize(s));
    if (total > 0x7fffffffu)
        return SMVP_E_TOOBIG;
    DevPtr<int2> blocks;
    SMVP_CUDA(dev_alloc(blocks, total));
    SMVP_LAUNCH(tjds_seg_fill_kernel, (unsigned)nseg, 256, 0, s, (const uint32_t *)seg_nb.get(), (const int32_t *)A->start_pos.get(),
                nseg, extra, blocks.get());
    SMVP_CUDA(cudaStreamSynchronize(s));
    SMVP_CUDA(cudaGetLastError());
    A->skew = skew;
    A->seg_blocks = std::move(blocks);
    A->num_seg_blocks = (int32_t)total;
    return SMVP_OK;
}

// The row bounds of the deterministic variants, from the current values: row_exp[rows] and the matrix flags
// (smvp_tjds::det_flags) into det_flags.  Synchronous.
static int tjds_row_bounds(const smvp_tjds *A, int32_t *row_exp, int32_t det_flags[5], cudaStream_t s)
{
    DevPtr<int32_t> flags;
    DevPtr<uint32_t> cnt;
    SMVP_CUDA(dev_alloc(cnt, A->rows));
    SMVP_CUDA(dev_alloc(flags, 5));
    const int32_t h0[5] = {0, EXP_NONE, EXP_LOW_NONE, 0x7fffffff, -1};
    SMVP_CUDA(cudaMemcpyAsync(flags.get(), h0, sizeof(h0), cudaMemcpyHostToDevice, s));
    SMVP_CUDA(cudaMemsetAsync(cnt.get(), 0, sizeof(uint32_t) * (size_t)A->rows, s));
    // EXP_NONE = 0x80808080 is a byte pattern, so a memset fills it
    SMVP_CUDA(cudaMemsetAsync(row_exp, 0x80, sizeof(int32_t) * (size_t)A->rows, s));
    if (A->nnz > 0)
    {
        int64_t blocks = ceil_div64(A->nnz, 256 * 4);
        const int64_t cap = (int64_t)device_props().sms * 16;
        if (blocks > cap)
            blocks = cap;
        // after the relabel decision: row_exp lives in the index space the kernels use
        SMVP_LAUNCH(tjds_row_bound_kernel, (unsigned)blocks, 256, 0, s, mult_rows(A), (const double *)A->val.get(), A->nnz,
                    row_exp, cnt.get(), flags.get());
    }
    if (A->rows > 0)
        SMVP_LAUNCH(tjds_row_exp_kernel, (unsigned)ceil_div64(A->rows, 256), 256, 0, s, row_exp, (const uint32_t *)cnt.get(),
                    A->rows, flags.get());
    SMVP_CUDA(cudaMemcpyAsync(det_flags, flags.get(), 5 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaStreamSynchronize(s));
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

static int tjds_prepare_det(smvp_tjds *A, cudaStream_t s)
{
    if (A->row_exp)
        return SMVP_OK;
    DevPtr<int32_t> row_exp;
    DevPtr<long long> acc;
    SMVP_CUDA(dev_alloc(row_exp, A->rows));
    SMVP_CUDA(dev_alloc(acc, 2 * (int64_t)A->rows));
    int32_t det_flags[5];
    static_assert(sizeof(det_flags) == sizeof(A->det_flags), "flags layout");
    SMVP_TRY(tjds_row_bounds(A, row_exp.get(), det_flags, s));
    memcpy(A->det_flags, det_flags, sizeof(det_flags));
    A->row_exp = std::move(row_exp);
    A->acc = std::move(acc);
    A->det_route = 0; // depends on the matrix flags just computed
    return SMVP_OK;
}

// After smvp_tjds_update_values has written new values: the row bounds and matrix flags again, into the handle's own
// row_exp, and the route of the current x decided again at the next pass.  Nothing to do while the deterministic state
// does not exist yet.  On failure that state is dropped, so the next deterministic pass builds it as on a new handle.
int tjds_update_det(smvp_tjds *A, cudaStream_t s)
{
    if (!A->row_exp)
        return SMVP_OK;
    A->det_route = 0;
    int32_t det_flags[5];
    const int rc = tjds_row_bounds(A, A->row_exp.get(), det_flags, s);
    if (rc != SMVP_OK)
    {
        A->row_exp.reset();
        A->acc.reset();
        return rc;
    }
    memcpy(A->det_flags, det_flags, sizeof(det_flags));
    return SMVP_OK;
}

// Which kernel serves SMVP_TJDS_DETERMINISTIC for the current x.  The exact integer accumulation needs finite inputs
// and products that cannot overflow; an x or a matrix holding Inf / NaN (the loader accepts them, strtod) or exponents
// whose sum may leave the fp64 range is routed to the atomic kernel, which propagates them the way the reference's
// loop does.  Decided on the host from two scalars: the matrix flags (tjds_prepare_det) and x_exp, which
// smvp_tjds_set_x_device copies into pinned memory behind an event -- one event wait per x, none per pass.
static int tjds_det_route(smvp_tjds *A)
{
    if (A->x_exp_pending)
    {
        SMVP_CUDA(cudaEventSynchronize(A->x_exp_event.get()));
        A->x_exp_pending = 0;
        A->det_route = 0;
    }
    if (A->det_route == 0)
    {
        const int32_t ex = A->x_exp_host ? *A->x_exp_host : EXP_NONE, er = A->det_flags[1];
        bool ok = !(A->det_flags[0] & 1) && ex != EXP_NONFINITE;
        if (ok && ex != EXP_NONE && er != EXP_NONE && (int64_t)ex + er > 1000)
            ok = false; // a product may overflow to Inf
        A->det_route = ok ? 1 : -1;
        // the short loop (tjds_det_kernel<.., FAST>) needs every visited row's bound inside the range of the fast split
        // and no visited row without an exponent (all-zero rows), and an x that is not all zero
        const int32_t lo_r = A->det_flags[2];
        A->det_fast = (ok && !(A->det_flags[0] & 2) && ex != EXP_NONE && er != EXP_NONE && lo_r != EXP_LOW_NONE &&
                       (int64_t)lo_r + ex >= TJDS_FRAC - 1023 && (int64_t)er + ex <= TJDS_FRAC - TJDS_W + 1022 &&
                       !env_set("SMVP_TJDS_DET_GENERAL"))
                          ? 1
                          : -1;
    }
    return SMVP_OK;
}

// plan and scratch of the transposed product (once per handle).  Synchronous.
static int tjds_transpose_prepare(smvp_tjds *A, cudaStream_t s)
{
    if (A->tr_ready || A->ndiag == 0)
        return SMVP_OK;
    SMVP_TRY(tjds_plan(A, s));
    if (A->ndiag > TJDS_SEG)
    {
        const int32_t nseg = (A->ndiag + TJDS_SEG - 1) / TJDS_SEG;
        const int32_t wide = TJDS_SEG * TJDS_SEG; // columns longer than this have more than TJDS_SEG chunks
        int32_t h[4] = {0, 0, 0, 0};
        SMVP_CUDA(cudaMemcpyAsync(h, A->start_pos.get() + TJDS_SEG, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        if (A->ndiag > wide)
            SMVP_CUDA(cudaMemcpyAsync(h + 2, A->start_pos.get() + wide, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        DevPtr<uint32_t> d_total, seg_off;
        DevPtr<double> part;
        SMVP_CUDA(dev_alloc(d_total, 1));
        SMVP_CUDA(dev_alloc(seg_off, nseg));
        SMVP_LAUNCH(tjds_transpose_count_kernel, (unsigned)ceil_div64(nseg, 256), 256, 0, s, (const int32_t *)A->start_pos.get(), nseg,
                    seg_off.get());
        SMVP_TRY(exclusive_scan_u32(seg_off.get(), seg_off.get(), nseg, d_total.get(), s));
        uint32_t total = 0;
        SMVP_CUDA(cudaMemcpyAsync(&total, d_total.get(), sizeof(total), cudaMemcpyDeviceToHost, s));
        SMVP_CUDA(cudaStreamSynchronize(s));
        SMVP_CUDA(cudaGetLastError());
        SMVP_CUDA(dev_alloc(part, total));
        A->tr_seg_off = std::move(seg_off);
        A->tr_part = std::move(part);
        A->tr_nlong = h[1] - h[0];
        A->tr_nwide = h[3] - h[2];
        A->device_bytes += 4 * (int64_t)nseg + 8 * (int64_t)total;
    }
    A->tr_ready = 1;
    return SMVP_OK;
}

constexpr Axpby AXPBY_PLAIN = {1.0, 0.0};

// work units of a transposed dot pass: the CTAs of the gather and of the combine kernel, or of the empty-handle kernel
static int64_t tjds_transpose_units(const smvp_tjds *A)
{
    if (A->ndiag == 0)
        return ceil_div64(A->cols, 256);
    const int64_t combine = A->ndiag > TJDS_SEG ? ceil_div64(32 * (int64_t)A->tr_nwide + (A->tr_nlong - A->tr_nwide), 256) : 0;
    return A->num_seg_blocks + combine;
}

// the most work units a dot pass of the handle can have: A x (256-row blocks) and, once its plan exists, A^T x -- the
// scratch is sized for both, so it grows at most once, at the first transposed dot call after an A x one
static int64_t tjds_dot_units_max(const smvp_tjds *A)
{
    const int64_t ax = ceil_div64(A->rows, 256);
    const int64_t atx = A->cols > 0 && (A->tr_ready || A->ndiag == 0) ? tjds_transpose_units(A) : 0;
    return ax > atx ? ax : atx;
}

// one transposed pass, asynchronous on s; tjds_transpose_prepare has run and A->cols > 0.  dot != NULL: a dot pass, its
// partials in dot->part (tjds_transpose_units of them)
static int tjds_transpose_pass(smvp_tjds *A, const double *d_x, double *d_y, const Axpby &ab, const DotOut *dot, cudaStream_t s)
{
    const YStore mode = store_mode(dot, false, ab);
    if (A->ndiag == 0 && mode == YStore::Plain) // no entries: every column is empty
    {
        SMVP_CUDA(cudaMemsetAsync(d_y, 0, sizeof(double) * (size_t)A->cols, s));
        return SMVP_OK;
    }
    const double *w = dot ? dot->w : nullptr;
    double *part = dot ? dot->part : nullptr;
    with_store<YStore::Plain, YStore::Axpby, YStore::Dot>(mode, [&](auto S) {
        constexpr YStore M = decltype(S)::value;
        if constexpr (M != YStore::Plain)
            if (A->ndiag == 0)
            {
                int64_t blocks = ceil_div64(A->cols, 256);
                const int64_t cap = (int64_t)device_props().sms * 8;
                if (M != YStore::Dot) // a grid-stride loop: 4 entries per thread, at most 8 CTAs per SM
                    blocks = ceil_div64(A->cols, 256 * 4) < cap ? ceil_div64(A->cols, 256 * 4) : cap;
                SMVP_LAUNCH(tjds_axpby_empty_kernel<M>, (unsigned)blocks, 256, 0, s, d_y, A->cols, ab.alpha, ab.beta, w, part);
                return (int)SMVP_OK;
            }
        SMVP_LAUNCH(tjds_transpose_kernel<M>, (unsigned)A->num_seg_blocks, 256, 0, s, (const int2 *)A->seg_blocks.get(),
                    (const int32_t *)A->start_pos.get(), (const int32_t *)A->row_ind.get(), (const double *)A->val.get(),
                    (const int32_t *)A->perm.get(), d_x, d_y, A->tr_part.get(), (const uint32_t *)A->tr_seg_off.get(), A->ndiag,
                    A->nslots, A->cols, A->tr_nlong, ab.alpha, ab.beta, w, part);
        if (A->ndiag > TJDS_SEG)
        {
            const int64_t threads = 32 * (int64_t)A->tr_nwide + (A->tr_nlong - A->tr_nwide);
            SMVP_LAUNCH(tjds_transpose_combine_kernel<M>, (unsigned)ceil_div64(threads, 256), 256, 0, s,
                        (const double *)A->tr_part.get(), (const uint32_t *)A->tr_seg_off.get(), (const int32_t *)A->slot_len.get(),
                        (const int32_t *)A->perm.get(), A->tr_nlong, A->tr_nwide,
                        d_y, ab.alpha, ab.beta, w, M == YStore::Dot ? part + A->num_seg_blocks : nullptr);
        }
        return (int)SMVP_OK;
    });
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

} // namespace smvp

using namespace smvp;

extern "C" int smvp_tjds_mult_transpose_device(smvp_tjds *A, const double *d_x, double *d_y, void *stream)
{
    if (!A || (A->rows > 0 && !d_x) || (A->cols > 0 && !d_y))
        return SMVP_E_ARG;
    if (A->cols == 0)
        return SMVP_OK;
    cudaStream_t s = (cudaStream_t)stream;
    SMVP_TRY(tjds_transpose_prepare(A, s));
    return tjds_transpose_pass(A, d_x, d_y, AXPBY_PLAIN, nullptr, s);
}

extern "C" int smvp_tjds_mult_transpose_device_axpby(smvp_tjds *A, double alpha, const double *d_x, double beta, double *d_y,
                                                     void *stream)
{
    if (!A || (A->rows > 0 && !d_x) || (A->cols > 0 && !d_y))
        return SMVP_E_ARG;
    if (d_y && d_y == d_x)
        return SMVP_E_ARG; // y would be read and written while the kernels gather it as x
    if (A->cols == 0)
        return SMVP_OK;
    cudaStream_t s = (cudaStream_t)stream;
    SMVP_TRY(tjds_transpose_prepare(A, s));
    return tjds_transpose_pass(A, d_x, d_y, Axpby{alpha, beta}, nullptr, s);
}

extern "C" int smvp_tjds_mult_transpose_device_axpby_dot(smvp_tjds *A, double alpha, const double *d_x, double beta, double *d_y,
                                                         const double *d_w, double *d_dot, void *stream)
{
    if (!A || (A->rows > 0 && !d_x) || (A->cols > 0 && !d_y) || !d_dot)
        return SMVP_E_ARG;
    if (d_y && d_y == d_x)
        return SMVP_E_ARG; // y would be read and written while the kernels gather it as x
    if ((d_w && d_w == d_y) || d_dot == d_x || d_dot == d_y || d_dot == d_w)
        return SMVP_E_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    if (A->cols > 0)
        SMVP_TRY(tjds_transpose_prepare(A, s));
    const int64_t units = A->cols > 0 ? tjds_transpose_units(A) : 0;
    SMVP_TRY(dot_scratch(&A->dot_buf, &A->dot_cap, &A->device_bytes, tjds_dot_units_max(A), s));
    const DotOut dot = {d_w, A->dot_buf.get()};
    if (A->cols > 0)
        SMVP_TRY(tjds_transpose_pass(A, d_x, d_y, Axpby{alpha, beta}, &dot, s));
    return dot_reduce(A->dot_buf.get(), A->dot_cap, units, d_dot, s);
}

extern "C" int smvp_tjds_mult_transpose(smvp_tjds *A, const double *x_host, double *y_host, int iters, double *ms_each)
{
    if (!A || iters < 1 || (A->rows > 0 && !x_host) || (A->cols > 0 && !y_host))
        return SMVP_E_ARG;
    if (!A->d_xt)
        SMVP_CUDA(dev_alloc(A->d_xt, A->rows));
    if (!A->d_yt)
        SMVP_CUDA(dev_alloc(A->d_yt, A->cols));
    if (A->rows > 0)
        SMVP_CUDA(cudaMemcpy(A->d_xt.get(), x_host, sizeof(double) * (size_t)A->rows, cudaMemcpyHostToDevice));
    SMVP_TRY(tjds_transpose_prepare(A, 0));
    const bool small = (int64_t)A->rows + A->cols + A->nnz < SMVP_SMALL_LOOP_ITEMS;
    if (A->cols > 0)
        SMVP_TRY(timed_loop(iters, ms_each, small, [&](cudaStream_t s) {
            return tjds_transpose_pass(A, A->d_xt.get(), A->d_yt.get(), AXPBY_PLAIN, nullptr, s);
        }));
    else if (ms_each)
        for (int it = 0; it < iters; it++)
            ms_each[it] = 0.0;
    if (A->cols > 0)
        SMVP_CUDA(cudaMemcpy(y_host, A->d_yt.get(), sizeof(double) * (size_t)A->cols, cudaMemcpyDeviceToHost));
    return SMVP_OK;
}

extern "C" int smvp_tjds_set_x_device(smvp_tjds *A, const double *d_x, void *stream)
{
    if (!A || (A->cols > 0 && !d_x))
        return SMVP_E_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    if (!A->x_exp)
        SMVP_CUDA(dev_alloc(A->x_exp, 1));
    if (!A->x_exp_host)
        SMVP_CUDA(cudaHostAlloc((void **)(int32_t **)out(A->x_exp_host), sizeof(int32_t), cudaHostAllocDefault));
    if (!A->x_exp_event)
        SMVP_CUDA(cudaEventCreateWithFlags(out(A->x_exp_event), cudaEventDisableTiming));
    SMVP_CUDA(cudaMemsetAsync(A->x_exp.get(), 0x80, sizeof(int32_t), s)); // 0x80808080: below every real exponent
    if (A->cols > 0)
    {
        int64_t blocks = ceil_div64(A->cols, 256);
        const int64_t cap = (int64_t)device_props().sms * 8;
        if (blocks > cap)
            blocks = cap;
        SMVP_LAUNCH(tjds_permute_x_kernel, (unsigned)blocks, 256, 0, s, d_x, (const int32_t *)A->perm.get(), A->cols, A->nslots,
                    A->x_perm.get(), A->x_exp.get());
    }
    SMVP_CUDA(cudaMemcpyAsync(A->x_exp_host.get(), A->x_exp.get(), sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    SMVP_CUDA(cudaEventRecord(A->x_exp_event.get(), s));
    A->x_exp_pending = 1;
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

// effective number of diagonals to walk: all, or the reference's shipped truncation (see smvp_cuda.h)
static int32_t tjds_effective_limit(const smvp_tjds *A, int32_t diag_limit)
{
    if (diag_limit <= 0)
        return A->ndiag;
    int32_t lim = diag_limit < A->ndiag ? diag_limit : A->ndiag;
    if (lim == A->ndiag && A->ndiag > 0 && A->last_diag_len == 1)
        lim = A->ndiag - 1; // the shipped loop never sees a singleton last diagonal (main-cli.c:957-966)
    return lim;
}

// plans, auxiliary arrays and the host-side routing decision: everything that may synchronise, so that the pass
// itself only enqueues work (and can be captured in a CUDA graph)
static int tjds_prepare(smvp_tjds *A, int variant, const Axpby &ab, cudaStream_t s, bool dot = false)
{
    if (A->rows == 0)
        return SMVP_OK;
    if (!A->x_exp)
        return SMVP_E_ARG; // smvp_tjds_set_x_device has not been called
    SMVP_TRY(tjds_plan(A, s));
    SMVP_TRY(tjds_relabel_plan(A, s));
    if (variant != SMVP_TJDS_ATOMIC)
    {
        SMVP_TRY(tjds_prepare_det(A, s));
        SMVP_TRY(tjds_det_route(A));
    }
    // the atomic sums of a natural-order handle land in a scratch vector under the epilogue (relabelled handles use y_rel);
    // a dot pass always runs the epilogue
    if ((!ab.plain() || dot) && A->relabel_state != 1 && (variant == SMVP_TJDS_ATOMIC || A->det_route != 1) && !A->y_sum)
    {
        SMVP_CUDA(dev_alloc(A->y_sum, A->rows));
        A->device_bytes += 8 * (int64_t)A->rows;
    }
    return SMVP_OK;
}

#define SMVP_TJDS_ARGS_COMMON                                                                                    \
    (const int2 *)A->seg_blocks.get(), (const int32_t *)A->start_pos.get(), mult_rows(A), (const double *)A->val.get(), \
        (const double *)A->x_perm.get()

// one pass, asynchronous on s; tjds_prepare has run (with the same ab and dot).  dot != NULL: the per-row kernel that
// stores y (unrank or det-finalize) also leaves the dot partials of its 256-row blocks in dot->part.
static int tjds_pass(smvp_tjds *A, double *d_y, int variant, int32_t diag_limit, const Axpby &ab, cudaStream_t s,
                     const DotOut *dot = nullptr)
{
    const int32_t lim = tjds_effective_limit(A, diag_limit);
    const YStore mode = store_mode(dot, false, ab);
    const bool ranked = A->relabel_state == 1, skew = A->skew == 1, epi = mode != YStore::Plain;
    const double *dot_w = dot ? dot->w : nullptr;
    double *part = dot ? dot->part : nullptr;
    const unsigned blocks = (unsigned)A->num_seg_blocks;
    if (variant == SMVP_TJDS_ATOMIC || A->det_route != 1)
    {
        double *y_caller = d_y;
        if (ranked)
            d_y = A->y_rel.get(); // sums land in rank order; tjds_unrank_y_kernel puts them back
        else if (epi)
            d_y = A->y_sum.get(); // sums land beside y; tjds_unrank_y_kernel (identity rank) applies the epilogue
        SMVP_CUDA(cudaMemsetAsync(d_y, 0, sizeof(double) * (size_t)A->rows, s));
        if (blocks > 0 && lim > 0)
        {
            if (skew)
                SMVP_LAUNCH((tjds_atomic_kernel<4, true>), blocks, 256, 0, s, SMVP_TJDS_ARGS_COMMON, d_y, A->nslots, lim);
            else
                SMVP_LAUNCH((tjds_atomic_kernel<4, false>), blocks, 256, 0, s, SMVP_TJDS_ARGS_COMMON, d_y, A->nslots, lim);
        }
        if (ranked || epi)
        {
            // Dot: one row per thread; the others: a grid-stride loop, 4 rows per thread, at most 8 CTAs per SM
            int64_t ub = ceil_div64(A->rows, 256);
            const int64_t cap = (int64_t)device_props().sms * 8;
            if (mode != YStore::Dot)
                ub = ceil_div64(A->rows, 256 * 4) < cap ? ceil_div64(A->rows, 256 * 4) : cap;
            const int32_t *rank = ranked ? (const int32_t *)A->row_rank.get() : nullptr;
            with_store<YStore::Plain, YStore::Axpby, YStore::Dot>(mode, [&](auto S) {
                SMVP_LAUNCH(tjds_unrank_y_kernel<decltype(S)::value>, (unsigned)ub, 256, 0, s, (const double *)d_y, rank, A->rows, y_caller,
                            ab.alpha, ab.beta, dot_w, part);
                return (int)SMVP_OK;
            });
        }
    }
    else
    {
        const int words = variant == SMVP_TJDS_DETERMINISTIC_FAST ? 1 : 2;
        // only the rows that hold entries have accumulators to clear and convert (tjds_prepare_det found the range)
        const int32_t r_lo = A->det_flags[4] >= 0 ? A->det_flags[3] : 0, r_hi = A->det_flags[4] + 1;
        for (int w = 0; w < words && r_hi > r_lo; w++)
            SMVP_CUDA(cudaMemsetAsync(A->acc.get() + (size_t)w * (size_t)A->rows + r_lo, 0, sizeof(long long) * (size_t)(r_hi - r_lo),
                                      s));
        if (blocks > 0 && lim > 0)
        {
            // CTAs per SM: 6 for the two-word kernel (40 registers).  The one-word kernel of the skewed fast walk runs at 8
            // (32 registers, at the price of ONE 4-byte spill outside the loop): 3.0 - 3.1 ms against 3.85 ms at 6 CTAs
            // without the spill (profiles/r02_logs/r02_tjds_sweep5.log) -- the kernel is latency-bound, residency wins.
            // The other swept configurations are in DESIGN.md §5.3.
            with_flag(skew, [&](auto SK) {
                return with_flag(A->det_fast == 1, [&](auto FA) {
                    constexpr bool SKEW = decltype(SK)::value, FAST = decltype(FA)::value;
                    if (words == 2)
                        SMVP_LAUNCH((tjds_det_kernel<4, SKEW, FAST, 6, 2>), blocks, 256, 0, s, SMVP_TJDS_ARGS_COMMON,
                                    (const int32_t *)A->row_exp.get(), (const int32_t *)A->x_exp.get(),
                                    (unsigned long long *)A->acc.get(), A->rows, A->nslots, lim);
                    else
                        SMVP_LAUNCH((tjds_det_kernel<4, SKEW, FAST, SKEW && FAST ? 8 : 6, 1>), blocks, 256, 0, s,
                                    SMVP_TJDS_ARGS_COMMON, (const int32_t *)A->row_exp.get(), (const int32_t *)A->x_exp.get(),
                                    (unsigned long long *)A->acc.get(), A->rows, A->nslots, lim);
                    return (int)SMVP_OK;
                });
            });
        }
        with_store<YStore::Plain, YStore::Axpby, YStore::Dot>(mode, [&](auto S) {
            SMVP_LAUNCH(tjds_det_finalize_kernel<decltype(S)::value>, (unsigned)ceil_div64(A->rows, 256), 256, 0, s,
                        (const long long *)A->acc.get(), (const int32_t *)A->row_exp.get(), (const int32_t *)A->x_exp.get(), A->rows,
                        d_y, ranked ? (const int32_t *)A->row_rank.get() : nullptr, words, r_lo, r_hi, ab.alpha, ab.beta, dot_w, part);
            return (int)SMVP_OK;
        });
    }
    SMVP_CUDA(cudaGetLastError());
    return SMVP_OK;
}

// d_dot != NULL: a dot pass (smvp_tjds_mult_device_axpby_dot), *d_dot = sum of w[r] * y_new[r] (w = d_w, or y_new)
static int tjds_mult_any(smvp_tjds *A, const Axpby &ab, double *d_y, int variant, int32_t diag_limit, void *stream,
                         const double *d_w = nullptr, double *d_dot = nullptr)
{
    if (!A || (A->rows > 0 && !d_y))
        return SMVP_E_ARG;
    if (variant != SMVP_TJDS_ATOMIC && variant != SMVP_TJDS_DETERMINISTIC && variant != SMVP_TJDS_DETERMINISTIC_FAST)
        return SMVP_E_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    if (!d_dot)
    {
        if (A->rows == 0)
            return SMVP_OK;
        SMVP_TRY(tjds_prepare(A, variant, ab, s));
        return tjds_pass(A, d_y, variant, diag_limit, ab, s);
    }
    const int64_t units = ceil_div64(A->rows, 256); // 256-row blocks of the kernel that stores y
    SMVP_TRY(tjds_prepare(A, variant, ab, s, true));
    SMVP_TRY(dot_scratch(&A->dot_buf, &A->dot_cap, &A->device_bytes, tjds_dot_units_max(A), s));
    if (A->rows > 0)
    {
        const DotOut dot = {d_w, A->dot_buf.get()};
        SMVP_TRY(tjds_pass(A, d_y, variant, diag_limit, ab, s, &dot));
    }
    return dot_reduce(A->dot_buf.get(), A->dot_cap, units, d_dot, s);
}

extern "C" int smvp_tjds_mult_device(smvp_tjds *A, double *d_y, int variant, int32_t diag_limit, void *stream)
{
    return tjds_mult_any(A, AXPBY_PLAIN, d_y, variant, diag_limit, stream);
}

extern "C" int smvp_tjds_mult_device_axpby(smvp_tjds *A, double alpha, double beta, double *d_y, int variant, int32_t diag_limit,
                                           void *stream)
{
    return tjds_mult_any(A, Axpby{alpha, beta}, d_y, variant, diag_limit, stream);
}

extern "C" int smvp_tjds_mult_device_axpby_dot(smvp_tjds *A, double alpha, double beta, double *d_y, const double *d_w, double *d_dot,
                                               int variant, int32_t diag_limit, void *stream)
{
    if (!A || !d_dot || (d_w && d_w == d_y) || d_dot == d_y || d_dot == d_w)
        return SMVP_E_ARG;
    return tjds_mult_any(A, Axpby{alpha, beta}, d_y, variant, diag_limit, stream, d_w, d_dot);
}

extern "C" int smvp_tjds_mult(smvp_tjds *A, const double *x_host, double *y_host, int iters, double *ms_each, int variant,
                              int32_t diag_limit)
{
    if (!A || iters < 1 || (A->cols > 0 && !x_host) || (A->rows > 0 && !y_host))
        return SMVP_E_ARG;
    if (variant != SMVP_TJDS_ATOMIC && variant != SMVP_TJDS_DETERMINISTIC && variant != SMVP_TJDS_DETERMINISTIC_FAST)
        return SMVP_E_ARG;
    if (!A->d_x)
        SMVP_CUDA(dev_alloc(A->d_x, A->cols));
    if (!A->d_y)
        SMVP_CUDA(dev_alloc(A->d_y, A->rows));
    if (A->cols > 0)
        SMVP_CUDA(cudaMemcpy(A->d_x.get(), x_host, sizeof(double) * (size_t)A->cols, cudaMemcpyHostToDevice));
    // x is permuted once, before the loop, as the reference does at build time (main-cli.c:907-923)
    SMVP_TRY(smvp_tjds_set_x_device(A, A->d_x.get(), nullptr));
    SMVP_TRY(tjds_prepare(A, variant, AXPBY_PLAIN, 0));
    // the zero-fill of y / of the accumulators is part of the pass and therefore INSIDE the timed bracket (the
    // reference keeps its vectorInit outside, main-cli.c:1008): conservative.
    const bool small = (int64_t)A->rows + A->cols + A->nnz < SMVP_SMALL_LOOP_ITEMS;
    const bool tiny = variant == SMVP_TJDS_ATOMIC && A->relabel_state != 1 && A->nnz <= 16384 && A->rows <= 4096 && A->cols <= 4096 &&
                      !env_set("SMVP_NO_TINY_LOOP");
    std::function<int(cudaStream_t, int)> multi;
    if (tiny)
        multi = [&](cudaStream_t s, int n) {
            SMVP_LAUNCH(tjds_tiny_loop_kernel, 1, TJDS_TINY_THREADS, 0, s, (const int32_t *)A->start_pos.get(),
                        (const int32_t *)A->slot_len.get(), (const int32_t *)A->row_ind.get(), (const double *)A->val.get(),
                        (const double *)A->x_perm.get(), A->d_y.get(), A->rows, A->nslots, tjds_effective_limit(A, diag_limit), n);
            SMVP_CUDA(cudaGetLastError());
            return (int)SMVP_OK;
        };
    if (A->rows > 0)
        SMVP_TRY(timed_loop(
            iters, ms_each, small, [&](cudaStream_t s) { return tjds_pass(A, A->d_y.get(), variant, diag_limit, AXPBY_PLAIN, s); },
            multi));
    else if (ms_each)
        for (int it = 0; it < iters; it++)
            ms_each[it] = 0.0;
    if (A->rows > 0)
        SMVP_CUDA(cudaMemcpy(y_host, A->d_y.get(), sizeof(double) * (size_t)A->rows, cudaMemcpyDeviceToHost));
    return SMVP_OK;
}

extern "C" int smvp_tjds_info(const smvp_tjds *A, smvp_tjds_info_t *out)
{
    if (!A || !out)
        return SMVP_E_ARG;
    out->rows = A->rows;
    out->cols = A->cols;
    out->nnz = A->nnz;
    out->ndiag = A->ndiag;
    out->ref_diag_limit = A->ref_diag_limit;
    out->input_order = A->input_order;
    out->bytes_per_mult = 12 * A->nnz + 4 * ((int64_t)A->ndiag + 1) + 8 * (int64_t)A->cols + 8 * (int64_t)A->rows;
    out->device_bytes = A->device_bytes;
    out->launches_per_mult[SMVP_TJDS_ATOMIC] = A->relabel_state == 1 ? 2 : 1;
    out->launches_per_mult[SMVP_TJDS_DETERMINISTIC] = 2;
    out->launches_per_mult[SMVP_TJDS_DETERMINISTIC_FAST] = 2;
    out->y_relabel = A->relabel_state;
    out->skewed_walk = A->skew;
    out->det_route = A->det_route;
    return SMVP_OK;
}
