// merge_warp_body.cuh -- the statements of the warp-autonomous merge-path kernel (csr_mult.cu), included as the body of
// csr_merge_warp_kernel (SMVP_MERGE_DOT 0) and of csr_merge_warp_dot_kernel (SMVP_MERGE_DOT 1).  The includer provides
// the template flags WARPS, IPT, FANOUT, RANKED, UNI, EPI and the kernel parameters; with SMVP_MERGE_DOT also dot_w and
// part.  The dot pass's statements are preprocessor sections rather than `if (DOT)` branches of an inlined __device__
// function because the plain kernel's machine code must stay as it is, and it does not: inlining the body, or even one
// unused local declared in the kernel, changes how ptxas allocates registers in it (cuobjdump -sass).  With
// SMVP_MERGE_DOT 0 the included text is exactly the plain kernel's.
    // Small grids (early_dependents != 0): let the fix-up kernel, launched with programmatic stream serialization, be
    // scheduled NOW; it parks at griddepcontrol.wait until this grid has completed and flushed.  In the batched `-n` loop
    // of a matrix like memplus that hides the second launch's latency (a pass lasts as long as a launch).
    if (early_dependents)
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // processes tiles [tile_begin, num_tiles): a sub-range lets the host overlap the copy-out of finished rows.
    // One stage per warp: deeper rings lost to more resident warps in every sweep.
    using Shape = MergeShape<32, IPT>;
    extern __shared__ __align__(128) unsigned char stage_mem[];
    __shared__ __align__(8) uint64_t full_bar[WARPS];

    // UNI: the warp index and the tile coordinates below are broadcast from lane 0.  The values are the same in every lane
    // anyway, but the broadcast lets the compiler PROVE it and keep the whole tile bookkeeping (and the operands of the
    // bulk copies) in uniform registers instead of electing a lane and converting per copy.  Measured on B200
    // (profiles/r01_logs/diet_bisect.log): stencil configuration 2.78 -> 2.69 ms, but the R-MAT configuration 5.67 ->
    // 6.39 ms, so it is a per-configuration choice (MergeStencil::UNI, MergeSkewed::UNI).
#define SMVP_BCAST(v) (UNI ? __shfl_sync(0xffffffffu, (v), 0) : (v))
    const int lane = threadIdx.x & 31, w = SMVP_BCAST((int)(threadIdx.x >> 5));
    const int64_t total = (int64_t)rows + nnz;
    unsigned char *base = stage_mem + (size_t)w * Shape::SMEM_BYTES;
    uint64_t *my_bar = &full_bar[w];
    uint64_t policy = 0;
    if (lane == 0)
    {
        mbar_init(my_bar, 1);
        fence_mbar_init();
        policy = l2_evict_first_policy();
    }
    __syncwarp();

    const uint64_t pol_last = RANKED ? l2_evict_last_policy() : 0, pol_first = RANKED ? l2_evict_first_policy() : 0;
    const int32_t warp_stride = (int32_t)gridDim.x * WARPS;
    auto issue = [&](const TileView &v) { // lane 0 only
        mbar_expect_tx(my_bar, v.vb + v.cb + v.rb);
        if (v.vb)
            bulk_g2s(base, val + v.va, v.vb, my_bar, policy);
        if (v.cb)
            bulk_g2s(base + v.vb, col_ind + v.ca, v.cb, my_bar, policy);
        if (v.rb)
            bulk_g2s(base + v.vb + v.cb, row_ptr + v.ra, v.rb, my_bar, policy);
    };

    int32_t t = tile_begin + (int32_t)blockIdx.x * WARPS + w;
    int32_t cur_r0 = 0, cur_r1 = 0; // merge coordinates of the tile in flight: the only tile state kept across the loop
    if (t < num_tiles)
    {
        cur_r0 = SMVP_BCAST(__ldg(tile_row + t));
        cur_r1 = SMVP_BCAST(__ldg(tile_row + t + 1));
        if (lane == 0)
            issue(make_tile(cur_r0, cur_r1, t, Shape::TILE, total));
    }
    uint32_t parity = 0;

    while (t < num_tiles)
    {
        // per-tile scalars: only what the walk needs stays live (the rest of the TileView dies here)
        int32_t n0, tile_r0, rows_t, nnz_t, items_t;
        uint32_t sval, scol, srow; // shared-window byte addresses of TILE-LOCAL nonzero 0 / row 0
        {
            const TileView v = make_tile(cur_r0, cur_r1, t, Shape::TILE, total);
            n0 = (int32_t)v.n0;
            tile_r0 = v.r0;
            rows_t = v.rows_t;
            nnz_t = v.nnz_t;
            items_t = v.items_t;
            const uint32_t b = smem_u32(base);
            sval = b + 8u * (uint32_t)(n0 - v.va);
            scol = b + v.vb + 4u * (uint32_t)(n0 - v.ca);
            srow = b + v.vb + v.cb + 4u * (uint32_t)(v.r0 + 1 - v.ra);
        }
        auto row_end = [&](int32_t i) -> int32_t { return lds_s32(srow + 4u * (uint32_t)i) - n0; };

        mbar_wait(my_bar, parity);
        parity ^= 1u;

        // ---- my first merge item: interpolate, gallop, bisect (2 probes on regular matrices)
        int32_t d = lane * IPT;
        if (d > items_t)
            d = items_t;
        int32_t lo = d > nnz_t ? d - nnz_t : 0, hi = d < rows_t ? d : rows_t;
        if (lo < hi)
        {
            // first guess by interpolation.  The divisor is the FULL tile size (a compile-time constant: multiply-shift
            // instead of a 25-instruction integer division); only the matrix's last tile is shorter, and there the guess
            // is merely a little low before the gallop corrects it.
            int32_t g = (int32_t)(((uint32_t)d * (uint32_t)rows_t) / (uint32_t)Shape::TILE); // < 2^20: 32-bit is exact
            g = g < lo ? lo : (g > hi - 1 ? hi - 1 : g);
            int32_t step = 1;
            if (row_end(g) <= d - g - 1)
            {
                lo = g + 1;
                while (lo < hi)
                {
                    const int32_t m = (lo + step - 1 < hi - 1) ? lo + step - 1 : hi - 1;
                    if (row_end(m) <= d - m - 1)
                    {
                        lo = m + 1;
                        step <<= 1;
                    }
                    else
                    {
                        hi = m;
                        break;
                    }
                }
            }
            else
            {
                hi = g;
                while (lo < hi)
                {
                    const int32_t m = (hi - step > lo) ? hi - step : lo;
                    if (!(row_end(m) <= d - m - 1))
                    {
                        hi = m;
                        step <<= 1;
                    }
                    else
                    {
                        lo = m + 1;
                        break;
                    }
                }
            }
            while (lo < hi)
            {
                const int32_t mid = (lo + hi) >> 1;
                if (row_end(mid) <= d - mid - 1)
                    lo = mid + 1;
                else
                    hi = mid;
            }
        }
        const int32_t i0 = lo, j0 = d - lo;
        int32_t d_next = (lane + 1) * IPT;
        if (d_next > items_t)
            d_next = items_t;
        int32_t j_next = __shfl_down_sync(0xffffffffu, j0, 1);
        if (lane == 31)
            j_next = nnz_t;
        const int32_t i_next = d_next - j_next;
        const int32_t cnt = j_next - j0;

        // ---- all my gathers first, in three phases pinned by volatile asm: the column indices, then every x gather of
        // the lane (IPT independent loads in flight together -- left alone, the compiler reuses one register pair and
        // waits for each load before issuing the next), then the products.  (Pinning the lane's two shared-window bases
        // in registers with an opaque move saves an address instruction per load but makes the 14-item configurations
        // spill; the nested "live slot / row end" walk this one replaced is in profiles/r01_logs/diet_bisect.log.)
        // EPI: y of my first row end (tile row i0; row 0 of the tile is the fix-up kernel's), loaded before the gathers so
        // that its latency hides behind them; further row ends of the lane (short rows) load y at their store
        double y_first = 0.0;
        if (EPI && beta != 0.0 && i0 < i_next && i0 != 0)
            y_first = ld_y_early(y + (int64_t)tile_r0 + i0);
#if SMVP_MERGE_DOT
        double w_first = 0.0; // w of that row, loaded beside it
        if (dot_w && i0 < i_next && i0 != 0)
            w_first = __ldg(dot_w + (int64_t)tile_r0 + i0);
#endif
        double prod[IPT];
        {
            int32_t cq[IPT];
            uint32_t cbase = scol + 4u * (uint32_t)j0, vbase = sval + 8u * (uint32_t)j0;
            // (every slot gets a defined value: leaving the dead ones undefined makes the compiler carry the previous
            // tile's registers through the loop and spill them)
#pragma unroll
            for (int q = 0; q < IPT; q++)
                cq[q] = q < cnt ? lds_s32(cbase + 4u * q) : 0;
#pragma unroll
            for (int q = 0; q < IPT; q++)
            {
                prod[q] = 0.0;
                if (q < cnt)
                    prod[q] = RANKED ? ldg_x_ranked(x, cq[q], hot_l1, hot_l2, pol_last, pol_first) : ldg_x_pinned(x, cq[q]);
            }
#pragma unroll
            for (int q = 0; q < IPT; q++)
                if (q < cnt)
                    prod[q] = __dmul_rn(lds_f64(vbase + 8u * q), prod[q]);
        }

        double sum = 0.0, first_sum = 0.0;
#if SMVP_MERGE_DOT
        double dl = 0.0; // this lane's dot terms, in the order it stores its rows
#endif
        bool has_first = false;
        {
            // Walk.  `until` = nonzeros of mine before my next row end (relative to j0, so each test is against a constant;
            // "no further row end of mine" = never).  Dead slots (q >= cnt) hold +0.0, and a partial sum that starts at
            // +0.0 can never become -0.0, so adding them is exact: the loop needs no "is this slot live" test, and the row
            // ends that follow my last nonzero are flushed by the same test at the first dead slot.
            int32_t row = i0;
            int32_t until = (row < i_next ? row_end(row) : 0x7fffffff) - j0;
#pragma unroll
            for (int q = 0; q < IPT; q++)
            {
                if (until <= q) // rare: a row end (or a run of empty rows) sits before item q
                {
                    do
                    {
                        if (!has_first)
                        {
                            has_first = true;
                            first_sum = sum;
                        }
#if SMVP_MERGE_DOT
                        else
                            store_axpby_dot(y, (int64_t)tile_r0 + row, sum, alpha, beta, dot_w, dl);
#else
                        else
                            store_y<FANOUT, EPI>(y, fan, (int64_t)tile_r0 + row, sum, alpha, beta);
#endif
                        sum = 0.0;
                        row++;
                        until = (row < i_next ? row_end(row) : 0x7fffffff) - j0;
                    } while (until <= q);
                }
                sum = __dadd_rn(sum, prod[q]);
            }
            // every row end of mine has at most IPT - 1 of my nonzeros before it, so the loop above has seen them all;
            // this is only a safety net
            while (row < i_next)
            {
                if (!has_first)
                {
                    has_first = true;
                    first_sum = sum;
                }
#if SMVP_MERGE_DOT
                else
                    store_axpby_dot(y, (int64_t)tile_r0 + row, sum, alpha, beta, dot_w, dl);
#else
                else
                    store_y<FANOUT, EPI>(y, fan, (int64_t)tile_r0 + row, sum, alpha, beta);
#endif
                sum = 0.0;
                row++;
            }
        }

        // ---- the stage is consumed: refill it for my next tile while the warp stitches
        __syncwarp();
        const int32_t tn = t + warp_stride;
        if (tn < num_tiles && tn > t)
        {
            cur_r0 = SMVP_BCAST(__ldg(tile_row + tn));
            cur_r1 = SMVP_BCAST(__ldg(tile_row + tn + 1));
            if (lane == 0)
                issue(make_tile(cur_r0, cur_r1, tn, Shape::TILE, total));
        }

        // ---- stitch rows cut by lane boundaries: segmented inclusive scan of (carry row, carry sum)
        const int32_t key = i_next; // the row my trailing partial belongs to
        double scan = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const int32_t pk = __shfl_up_sync(0xffffffffu, key, o);
            const bool take = lane >= o && pk == key;
            const double pv = __shfl_up_sync(0xffffffffu, scan, o);
            if (take)
                scan = __dadd_rn(pv, scan);
        }
        const double prev_scan = __shfl_up_sync(0xffffffffu, scan, 1);
        const int32_t prev_key = __shfl_up_sync(0xffffffffu, key, 1);
        if (has_first)
        {
            if (lane > 0 && prev_key == i0)
                first_sum = __dadd_rn(prev_scan, first_sum);
            // the tile's first row may have started in earlier tiles: its partial goes to the fix-up
            // kernel, which adds the carries and writes y -- and, under the epilogue, is the only one to read that
            // row of y.  Without the epilogue y is only ever WRITTEN here (never read), so it may be a write-only
            // mapping such as an NVSwitch multicast address.
            if (i0 == 0)
                head_val[t] = first_sum;
#if SMVP_MERGE_DOT
            else
            {
                const double v = axpby(alpha, first_sum, beta, y_first);
                y[(int64_t)tile_r0 + i0] = v;
                dl = __dadd_rn(dl, __dmul_rn(dot_w ? w_first : v, v));
            }
#else
            else if (EPI)
                y[(int64_t)tile_r0 + i0] = axpby(alpha, first_sum, beta, y_first);
            else
                store_y<FANOUT, false>(y, fan, (int64_t)tile_r0 + i0, first_sum, alpha, beta);
#endif
        }
        if (lane == 31)
            carry_val[t] = scan; // partial of the row that continues into the next tile
#if SMVP_MERGE_DOT
        dl = warp_tree_sum(dl); // the lanes in a pairwise tree: the tile's partial (the fix-up adds its first row)
        if (lane == 0)
            part[t] = dl;
#endif
        if (tn <= t)
            break; // 32-bit overflow guard
        t = tn;
    }
#undef SMVP_BCAST
