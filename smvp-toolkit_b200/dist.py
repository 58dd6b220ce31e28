"""Multi-GPU partitioning of the CSR / TJDS path: one process per GPU, torch.distributed for the plumbing.

The reference is single-process and single-threaded (SURVEY.md 8e); the path shards naturally with
exactly one exchange step per format:

  CSR   contiguous ROW blocks balanced by nnz; x replicated; each rank multiplies its rows; every rank
        must end with the full y.  Two exchanges:
          "multicast"  fused: y lives in symmetric memory with an NVSwitch multicast mapping and the
                       multiply kernels store their rows straight to the multicast address, so the
                       switch replicates each 8-byte result into every peer's y while the SpMV is still
                       streaming; a device-side barrier closes the step.  No separate collective.
          "p2p"        fused, unicast: same, but the kernels store each row into every rank's y through the
                       peer mappings of the symmetric-memory buffer (fan-out of N stores per row).
                       Measured on B200 (tools/probe_symm.py): coalesced peer stores run at ~700 GB/s,
                       multicast stores at ~340 GB/s per sender, so p2p wins for N = 2 and multicast
                       (egress 1/N of the data instead of (N-1)/N) from N = 4 on.
          "copy"       pipelined: the rank's row block is cut into sub-blocks (nnz-balanced); while the SpMV
                       of sub-block k+1 streams the matrix on the SMs, the copy engines push the finished
                       rows of sub-block k into every peer's y over NVLink (cudaMemcpyAsync to the peer
                       mappings, no SM involved).  The exchange then costs one sub-block's copy instead
                       of the whole allgather.  At N = 8 the allgather itself is NVLink-ingress bound
                       (each GPU must receive 7/8 of y: 352 MB = 0.55 ms measured), so large aligned
                       transfers matter more than fusing: in-kernel 8-byte stores reach only a third of
                       that rate.
          "pipeline"   "copy" with two y buffers: the copy engines push step k's rows while step k+1 already
                       multiplies (x is constant over the -n loop and the reference reports only the last
                       y, main-cli.c:401, so consecutive iterations are independent).  Every step's y still
                       reaches every rank -- one step later -- and finish() drains the pipe; the steady-state
                       cost per step is max(SpMV, exchange) instead of their sum.
          "nccl"       baseline: the y blocks are all-gathered by NCCL after the multiply.
  TJDS  contiguous COLUMN blocks balanced by nnz; each rank builds a local TJDS over its columns and
        needs only its slice of x; partial y vectors are combined by NCCL reduce-scatter (sum, fp64).

The partition arithmetic (`balanced_bounds`) and the two operators are backend-agnostic: the
world_size-2 gloo tests drive them on CPU with an injected local multiply.
"""
import json
import os

import numpy as np


def bind_host_near_gpu(index):
    """Pins this process to the CPUs of the NUMA node its GPU hangs off (sysfs), so that the page-locked host vectors it
    allocates afterwards are local to that GPU's PCIe root.  torchrun starts one process per GPU without any binding;
    with 8 ranks on a two-socket host half of the host<->device traffic would otherwise cross the socket interconnect.
    Returns the node, or None when the platform does not say (VMs often report -1)."""
    try:
        import torch

        p = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:  # noqa: BLE001  (no sysfs, no permission, properties missing: leave the process where it is)
        return None


def balanced_bounds(prefix, total_keys, parts):
    """Boundaries 0 = b_0 <= ... <= b_parts = total_keys with b_g = lower_bound(prefix, g*total/parts),
    where prefix(k) = number of nonzeros with key < k (SURVEY.md 8e: r_g = lower_bound(row_ptr, g*nnz/G))."""
    total = int(prefix(total_keys))
    bounds = [0]
    for g in range(1, parts):
        target = total * g // parts
        lo, hi = bounds[-1], total_keys
        while lo < hi:
            mid = (lo + hi) // 2
            if prefix(mid) < target:
                lo = mid + 1
            else:
                hi = mid
        bounds.append(lo)
    bounds.append(total_keys)
    return bounds


def bounds_from_counts(counts, parts):
    """Same, from an explicit per-key count array (numpy int)."""
    csum = np.concatenate([[0], np.cumsum(np.asarray(counts, dtype=np.int64))])
    return balanced_bounds(lambda k: csum[k], len(counts), parts)


def allgather_v(dist, y_full, bounds, rank):
    """All-gather of uneven contiguous blocks of y_full (block g = y_full[bounds[g]:bounds[g+1]]), in place."""
    views = [y_full[bounds[g]:bounds[g + 1]] for g in range(len(bounds) - 1)]
    if dist.get_backend() == "nccl":
        dist.all_gather(views, views[rank])
    else:  # gloo (CPU tests): one broadcast per block
        for g, v in enumerate(views):
            if v.numel() > 0:
                dist.broadcast(v, src=g)


def allgather_padded(dist, y_pad, y_full, bounds, rank, per):
    """All-gather of uneven blocks through ONE NCCL all_gather_into_tensor on equal padded slots (block g lives in
    y_pad[g*per : g*per + rows_g]), followed by the compaction into the contiguous y_full.  This is the NCCL baseline the
    fused exchanges are compared with (round 1 used dist.all_gather on a list of uneven views, which makes torch stage
    through a temporary: a straw man)."""
    dist.all_gather_into_tensor(y_pad, y_pad[rank * per:(rank + 1) * per])
    for g in range(len(bounds) - 1):
        n = bounds[g + 1] - bounds[g]
        if n > 0:
            y_full[bounds[g]:bounds[g + 1]].copy_(y_pad[g * per:g * per + n], non_blocking=True)


def reduce_scatter_ordered(dist, eng, y_owned, y_partial, scratch, rank, world, stream=None):
    """y_owned = block `rank` of the sum over ranks of y_partial, added in RANK ORDER by our own kernel
    (smvp_sum_ordered_device) after an all-to-all of the blocks: the bits do not depend on NCCL's algorithm, protocol or
    channel count, which is what makes the deterministic TJDS variant reproducible run to run at N > 1 (SURVEY.md 8e)."""
    per = y_owned.numel()
    if dist.get_backend() == "nccl":
        dist.all_to_all_single(scratch, y_partial)
        eng.sum_ordered_device(y_owned, scratch, world, per, per, stream)
    else:  # gloo (CPU tests) has no all-to-all: gather every partial, add my block in rank order
        parts = [y_partial.new_empty(y_partial.shape) for _ in range(world)]
        dist.all_gather(parts, y_partial)
        acc = parts[0][rank * per:(rank + 1) * per].clone()
        for k in range(1, world):
            acc = acc + parts[k][rank * per:(rank + 1) * per]
        y_owned.copy_(acc)


def reduce_scatter_sum(dist, y_owned, y_partial, rank):
    """y_owned = block `rank` of sum over ranks of y_partial (len(y_partial) == world * len(y_owned))."""
    if dist.get_backend() == "nccl":
        dist.reduce_scatter_tensor(y_owned, y_partial, op=dist.ReduceOp.SUM)
    else:  # gloo has no reduce-scatter: all-reduce, keep my block
        dist.all_reduce(y_partial, op=dist.ReduceOp.SUM)
        n = y_owned.numel()
        y_owned.copy_(y_partial[rank * n:(rank + 1) * n])


def row_block_spmv(dist, local_mult, bounds, rank, x, y_full):
    """The row-partitioned product, backend-agnostic: y_full[block] = local_mult(x) on every rank, then the
    blocks are all-gathered.  local_mult maps the replicated x to this rank's rows of y."""
    y_full[bounds[rank]:bounds[rank + 1]] = local_mult(x)
    allgather_v(dist, y_full, bounds, rank)
    return y_full


def col_block_spmv(dist, local_mult, bounds, rank, world, x, rows, ordered=False, eng=None):
    """The column-partitioned product, backend-agnostic: partial = local_mult(x[my columns]) has `rows`
    entries on every rank; the partials are summed and scattered (rank g owns rows [g*p, (g+1)*p)).
    ordered=True: the sum is taken in rank order (reduce_scatter_ordered) instead of by the backend's reduction."""
    import torch

    per = -(-rows // world)
    partial = torch.zeros(per * world, dtype=torch.float64, device=x.device)
    partial[:rows] = local_mult(x[bounds[rank]:bounds[rank + 1]])
    owned = torch.zeros(per, dtype=torch.float64, device=x.device)
    if ordered:
        reduce_scatter_ordered(dist, eng, owned, partial, torch.empty_like(partial), rank, world)
    else:
        reduce_scatter_sum(dist, owned, partial, rank)
    return owned


# ------------------------------------------------------------------------------------ matrix sources
class StencilSource:
    """27-point stencil on an nx*ny*nz grid (BASELINE.json configs[2]); shards are generated on the device."""

    def __init__(self, eng, nx, ny, nz, value_mode=None, seed=0):
        self.eng, self.nx, self.ny, self.nz = eng, nx, ny, nz
        self.rows = self.cols = nx * ny * nz
        self.value_mode = eng.VAL_STENCIL if value_mode is None else value_mode
        self.seed = seed
        self.nnz = self.row_prefix(self.rows)
        self.desc = "27-point stencil %dx%dx%d" % (nx, ny, nz)

    def row_prefix(self, r):
        return self.eng.synth_stencil27_prefix(self.nx, self.ny, self.nz, r)

    col_prefix = row_prefix  # structurally symmetric

    def row_block(self, r0, r1):
        """(row_local, col_global, val, order) of rows [r0, r1)."""
        return self.eng.synth_stencil27(self.nx, self.ny, self.nz, r0, r1, self.value_mode, self.seed)

    def col_block(self, c0, c1):
        """(row_global, col_local, val) of columns [c0, c1).  The {26,-1} stencil matrix is symmetric, so the
        column block is the row block with the two index arrays swapped (it arrives (col,row)-sorted)."""
        if self.value_mode != self.eng.VAL_STENCIL:
            raise ValueError("col_block by symmetry needs the symmetric {26,-1} values")
        r, c, v = self.eng.synth_stencil27(self.nx, self.ny, self.nz, c0, c1, self.value_mode, self.seed)
        return c, r, v


class RmatSource:
    """R-MAT 2^scale square matrix (BASELINE.json configs[3]/[4]).  Every rank generates the same deduplicated
    edge list on its own device (counter-based RNG) and cuts its block out of it."""

    def __init__(self, eng, scale, nedges, seed=42):
        import torch

        self.eng = eng
        self.rows = self.cols = 1 << scale
        self.row, self.col, self.val = eng.synth_rmat(scale, nedges, seed=seed)
        self.nnz = self.row.n
        self.desc = "R-MAT scale %d, %d draws, %d unique" % (scale, nedges, self.nnz)
        self._prefix = {}
        self._torch = torch

    def _csum(self, by_col):
        if by_col not in self._prefix:
            torch = self._torch
            counts = torch.zeros(self.rows + 1, dtype=torch.int32, device="cuda")
            self.eng.coo_histogram_device(self.row, self.col, self.nnz, by_col, self.rows, counts)
            csum = torch.zeros(self.rows + 1, dtype=torch.int64, device="cuda")
            csum[1:] = torch.cumsum(counts[:-1].to(torch.int64), 0)
            self._prefix[by_col] = csum.cpu().numpy()
        return self._prefix[by_col]

    def row_prefix(self, r):
        return int(self._csum(False)[r])

    def col_prefix(self, c):
        return int(self._csum(True)[c])

    def row_block(self, r0, r1):
        return self.eng.coo_filter_device(self.row, self.col, self.val, self.nnz, r0, r1, 0, self.cols, r0, 0)

    def col_block(self, c0, c1):
        return self.eng.coo_filter_device(self.row, self.col, self.val, self.nnz, 0, self.rows, c0, c1, 0, c0)

    def release(self):
        for a in (self.row, self.col, self.val):
            a.free()


def _measured_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture, if any."""
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(kernel_key)
    except Exception:
        return None


# ------------------------------------------------------------------------------------ operators
class RowBlockCsr:
    """y = A x with A in CSR, rows cut into nnz-balanced blocks over `world` ranks."""

    def __init__(self, eng, source, rank, world, variant=0, exchange="nccl", release_source=False, sub_blocks=4):
        import torch

        self.eng, self.rank, self.world, self.variant, self.exchange = eng, rank, world, variant, exchange
        self.M, self.N = source.rows, source.cols
        self.bounds = balanced_bounds(source.row_prefix, self.M, world)
        self.r0, self.r1 = self.bounds[rank], self.bounds[rank + 1]
        # sub-blocks (only the "copy" exchange uses more than one)
        # "copy" hides the exchange behind the next SUB-BLOCK; "pipeline" hides it behind the next STEP and needs none
        nsub = sub_blocks if (world > 1 and exchange == "copy") else 1
        base = source.row_prefix(self.r0)
        if nsub > 1:
            rel = balanced_bounds(lambda k: source.row_prefix(self.r0 + k) - base, self.r1 - self.r0, nsub)
            self.sub_bounds = [self.r0 + b for b in rel]
        else:
            self.sub_bounds = [self.r0, self.r1]
        self.subs = []
        self.local_nnz = 0
        for g in range(len(self.sub_bounds) - 1):
            a0, a1 = self.sub_bounds[g], self.sub_bounds[g + 1]
            r, c, v = source.row_block(a0, a1)
            self.local_nnz += r.n
            self.subs.append(eng.CsrMatrix.build_device(r, c, v, a1 - a0, self.N, r.n))
            for a in (r, c, v):
                a.free()
        self.A = self.subs[0]
        if hasattr(source, "release") and release_source:
            source.release()
        self.global_nnz = source.nnz
        self.global_bytes_per_mult = 12 * source.nnz + 4 * (self.M + 1) + 8 * self.N + 8 * self.M
        self.local_bytes_per_mult = (12 * self.local_nnz + 4 * (self.r1 - self.r0 + 1) + 8 * self.N +
                                     8 * (self.r1 - self.r0))
        self.symm = None
        self.y_fan = None
        self.peer_views, self.copy_stream, self.sub_events = None, None, None
        self.y_src, self.y_pad = None, None
        self.scheme, self.tuning = None, None
        self.spmv_events = None  # (start, end) CUDA events around the SpMV launch of the step in progress
        self.nbuf, self.k = 1, 0
        if world > 1 and exchange in ("multicast", "p2p", "copy", "pipeline"):
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm_mem

            self.nbuf = 2 if exchange == "pipeline" else 1
            self.y_sym = symm_mem.empty(self.nbuf * self.M, dtype=torch.float64,
                                        device=torch.device("cuda", torch.cuda.current_device()))
            self.y_sym.zero_()
            self.y_full = self.y_sym[:self.M]
            self.symm = symm_mem.rendezvous(self.y_sym, dist.group.WORLD.group_name)
            self.y_write = None
            self.mc_base = int(self.symm.multicast_ptr) if self.symm.multicast_ptr else None
            self.peer_ranks = [(rank + j) % world for j in range(1, world)]  # ring order
            if exchange == "multicast":
                if not self.mc_base:
                    raise RuntimeError("this system exposes no NVSwitch multicast mapping; use exchange='p2p' or 'nccl'")
                # write-only view of y: one store here lands in every rank's y_full
                self.y_write = self.mc_base + 8 * self.r0
            elif exchange == "pipeline":
                self._setup_pipeline()
            elif exchange == "copy":
                self.peer_views = [self.symm.get_buffer(k, (self.nbuf * self.M,), torch.float64) for k in self.peer_ranks]
                # SMVP_COPY_STREAMS=1: one stream, the ring steps follow each other (a permutation per step);
                # default: one stream per peer, all copies in flight at once
                nstreams = int(os.environ.get("SMVP_COPY_STREAMS", "0")) or len(self.peer_views)
                pool = [torch.cuda.Stream() for _ in range(min(nstreams, len(self.peer_views)))]
                self.copy_streams = [pool[i % len(pool)] for i in range(len(self.peer_views))]
                self.copy_stream = self.copy_streams[0]
                self.sub_events = [[torch.cuda.Event() for _ in self.subs] for _ in range(self.nbuf)]
            else:
                if world > 8:
                    raise RuntimeError("p2p fan-out supports at most 8 ranks")
                # my block of y inside every rank's buffer, my own first
                ptrs = [int(p) for p in self.symm.buffer_ptrs]
                order = [rank] + [k for k in range(world) if k != rank]
                self.y_fan = [ptrs[k] + 8 * self.r0 for k in order]
        else:
            self.y_write = None
            if world > 1 and exchange == "nccl":
                # equal padded slots for ONE all_gather_into_tensor; the SpMV writes straight into my slot
                self.per = max(self.bounds[g + 1] - self.bounds[g] for g in range(world))
                self.y_pad = torch.zeros(self.per * world, dtype=torch.float64, device="cuda")
            self.y_full = torch.zeros(self.M, dtype=torch.float64, device="cuda")
        if self.y_pad is not None:
            self.y_local = self.y_pad[rank * self.per:rank * self.per + (self.r1 - self.r0)]
        else:
            self.y_local = self.y_full[self.r0:self.r1]
        self.local_rows_out = self.r1 - self.r0
        resolved = self.A.auto_variant if variant == eng.CSR_AUTO else variant
        self.variant_name = {eng.CSR_VECTOR: "vector", eng.CSR_MERGE: "merge"}[resolved]
        self.x = None
        self._source_desc = source.desc

    # ------------------------------------------------------------------ pipelined exchange: schemes and their tuning
    SCHEME_HOW = {
        "ce_unicast": "the copy engines (one peer copy per rank)",
        "ce_multicast": "ONE copy-engine transfer to the NVSwitch multicast address",
        "sm_multicast": "a small high-priority SM kernel (%d CTAs, 128-bit stores) writing to the NVSwitch multicast address",
        "sm_unicast": "a small high-priority SM kernel (%d CTAs) that reads my rows once and stores them into every peer's y",
        "tma_unicast": "%d one-warp CTAs driving the TMA engine (cp.async.bulk global->shared->global): my rows are read once "
                       "and leave for every peer's y as bulk stores over NVLink",
        "tma_multicast": "%d one-warp CTAs driving the TMA engine (cp.async.bulk) with bulk stores to the NVSwitch multicast address",
        "tma_hybrid": "%d one-warp CTAs driving the TMA engine: the first half of my rows goes to the NVSwitch multicast address, "
                      "the second half to every peer by unicast (less ingress than all-multicast, less egress than all-unicast)",
    }

    def _setup_pipeline(self):
        import torch

        nloc = self.r1 - self.r0
        # staging buffers of the multicast schemes: each starts on the same 16-byte phase as its destination
        # y_sym[b * M + r0] (M and r0 may be odd), otherwise the TMA push (bulk copies need source and destination on
        # the same phase) would fall back to the 512-thread store kernel for half of the (rank, buffer) pairs
        self._y_src_raw = [torch.zeros(nloc + 2, dtype=torch.float64, device="cuda") for _ in range(self.nbuf)]
        self.y_src = [self._y_src_raw[b][((b * self.M + self.r0) & 1):][:nloc] for b in range(self.nbuf)]
        self.peer_views = [self.symm.get_buffer(k, (self.nbuf * self.M,), torch.float64) for k in self.peer_ranks]
        self.peer_ptrs = [int(self.symm.buffer_ptrs[k]) for k in self.peer_ranks]
        self.push_stream = torch.cuda.Stream(priority=-1)
        self.ce_streams = [torch.cuda.Stream() for _ in self.peer_ranks]
        self.spmv_done = [torch.cuda.Event() for _ in range(self.nbuf)]
        self.copy_done = [torch.cuda.Event() for _ in range(self.nbuf)]
        self.copy_pending = [False] * self.nbuf
        forced = os.environ.get("SMVP_PIPELINE_SCHEME")  # e.g. sm_multicast:32, ce_unicast
        if forced is None and os.environ.get("SMVP_PIPELINE_MODE"):  # round-1 switches, still honoured
            ctas = int(os.environ.get("SMVP_PUSH_CTAS", "32"))
            forced = ("ce_unicast" if os.environ["SMVP_PIPELINE_MODE"] == "unicast" else
                      ("sm_multicast:%d" % ctas if ctas > 0 else "ce_multicast"))
        self.set_scheme(forced or ("sm_multicast:32" if (self.mc_base and self.world >= 8) else "ce_unicast"))
        self._scheme_forced = forced is not None

    def scheme_candidates(self):
        c = ["ce_unicast", "tma_unicast:16", "tma_unicast:32", "tma_unicast:64", "tma_unicast:128", "sm_unicast:32"]
        if self.mc_base:
            c += ["ce_multicast", "sm_multicast:32", "tma_multicast:32", "tma_multicast:64", "tma_multicast:128", "tma_hybrid:64"]
        return c

    def set_scheme(self, scheme):
        kind, _, arg = scheme.partition(":")
        if kind not in self.SCHEME_HOW or ((kind.endswith("multicast") or kind == "tma_hybrid") and not self.mc_base):
            raise ValueError("unknown or unavailable pipeline scheme %r" % scheme)
        self.scheme, self.scheme_kind, self.scheme_ctas = scheme, kind, int(arg or 0)
        # a push done by a kernel runs BESIDE the next step's SpMV: the persistent merge-path grid leaves one CTA slot
        # per SM free for it (smvp_csr_set_corunner_headroom; measured on one GPU: SpMV 1.34 ms + TMA push 0.42 ms side by
        # side take 1.78 ms without the room, 1.43 ms with it).  Copy-engine schemes need none.
        self.A.set_corunner_headroom(0 if kind.startswith("ce_") else 1)

    def tune_pipeline(self, stream, steps=6):
        """Times `steps` pipelined steps (exchange drained inside) with every scheme this box offers, takes the MAX over
        ranks and keeps the fastest.  Called during warm-up, outside any timed region; every rank ends up with the same
        choice.  Also measures, for the chosen scheme, the SpMV alone and the exchange alone."""
        import torch
        import torch.distributed as dist

        if self.exchange != "pipeline" or self.symm is None:
            return None
        res = {}
        cands = [self.scheme] if self._scheme_forced else self.scheme_candidates()
        for cand in cands:
            self.set_scheme(cand)
            for _ in range(2):
                self.step(stream)
            self.finish(stream)
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                self.step(stream)
            self.finish(stream)
            e1.record(stream)
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res[cand] = float(t[0])
        # the two fastest are run again over a longer region (a scheme may look good for a handful of steps and lose over
        # many: the copy-engine multicast did at 8 ranks, 0.70 ms over 6 steps, 0.88 ms over 50) and the better one stays
        final = {}
        if len(res) > 1:
            for cand in sorted(res, key=res.get)[:2]:
                self.set_scheme(cand)
                for _ in range(2):
                    self.step(stream)
                self.finish(stream)
                torch.cuda.synchronize()
                dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(5 * steps):
                    self.step(stream)
                self.finish(stream)
                e1.record(stream)
                torch.cuda.synchronize()
                t = torch.tensor([e0.elapsed_time(e1) / (5 * steps)], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                final[cand] = float(t[0])
        best = min(final, key=final.get) if final else min(res, key=res.get)
        self.set_scheme(best)
        # the two halves of a step, each alone (same MAX over ranks): what the overlap has to hide
        parts = {}
        for name, fn in (("spmv_alone_ms", lambda: self.A.mult_device(self.x, self._src(0), self.variant, stream)),
                         ("exchange_alone_ms", lambda: self._push(0, stream, on_main=True))):
            fn()
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                fn()
            e1.record(stream)
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            parts[name] = float(t[0])
        self.symm.barrier(channel=0)
        torch.cuda.synchronize()
        self.tuning = {"candidates_ms_per_step": res, "finalists_ms_per_step_long_run": final, "chosen": best, **parts}
        return self.tuning

    def _src(self, b):
        """Where the SpMV of buffer b writes my rows, and what the push reads.  Unicast schemes: straight into my own copy
        of y (my rows need no transfer to myself).  Multicast schemes: a private staging buffer -- the switch writes my
        rows into EVERY rank's y, mine included, and must not race with the kernel that produces them."""
        if self.scheme_kind.endswith("multicast") or self.scheme_kind == "tma_hybrid":
            return self.y_src[b]
        return self.y_sym[b * self.M + self.r0:b * self.M + self.r1]

    def _push(self, b, stream, on_main=False):
        """Sends my rows of buffer b (y_src[b]) into every rank's y_sym[b], then a device-side barrier over all ranks on
        the same stream: once copy_done[b] has passed, step k's y is complete on EVERY rank (per-step completion, not
        just a drain at the end)."""
        import torch

        nbytes = 8 * (self.r1 - self.r0)
        off = 8 * (b * self.M + self.r0)
        src = self._src(b)
        ps = stream if on_main else self.push_stream
        if self.scheme_kind == "ce_unicast":
            if on_main:
                for pv in self.peer_views:
                    pv[b * self.M + self.r0:b * self.M + self.r1].copy_(src, non_blocking=True)
            else:
                for pv, cs in zip(self.peer_views, self.ce_streams):
                    cs.wait_event(self.spmv_done[b])
                    with torch.cuda.stream(cs):
                        pv[b * self.M + self.r0:b * self.M + self.r1].copy_(src, non_blocking=True)
                    ps.wait_stream(cs)
        elif self.scheme_kind == "ce_multicast":
            self.eng.copy_device(self.mc_base + off, src, nbytes, ps)
        elif self.scheme_kind == "sm_multicast":
            self.eng.push_device(self.mc_base + off, src, nbytes, self.scheme_ctas, ps)
        elif self.scheme_kind == "tma_multicast":
            self.eng.push_tma_device([self.mc_base + off], src, nbytes, self.scheme_ctas, ps)
        elif self.scheme_kind == "tma_unicast":
            self.eng.push_tma_device([p + off for p in self.peer_ptrs], src, nbytes, self.scheme_ctas, ps)
        elif self.scheme_kind == "tma_hybrid":
            half = ((self.r1 - self.r0) // 2) & ~1  # rows; even: the second part stays 16-byte aligned
            hb = 8 * half
            if hb > 0:
                self.eng.push_tma_device([self.mc_base + off], src, hb, max(self.scheme_ctas // 2, 1), ps)
            if nbytes > hb:  # second half: every peer and my own copy of y (the staging buffer is not y)
                dsts = [p + off + hb for p in self.peer_ptrs] + [int(self.symm.buffer_ptrs[self.rank]) + off + hb]
                self.eng.push_tma_device(dsts, src[half:], nbytes - hb, max(self.scheme_ctas // 2, 1), ps)
        else:  # sm_unicast: one kernel reads my rows once and stores them into every peer's buffer
            self.eng.push_fanout_device([p + off for p in self.peer_ptrs], src, nbytes, self.scheme_ctas, ps)
        with torch.cuda.stream(ps):
            self.symm.barrier(channel=1 + b)

    @property
    def partition_desc(self):
        how = {"nccl": "all-gathered by ONE NCCL all_gather_into_tensor on equal padded slots + compaction",
               "multicast": "stored by the SpMV kernel to the NVSwitch multicast address of y (fused, no collective) + device "
               "barrier",
               "p2p": "stored by the SpMV kernel into every rank's y through NVLink peer mappings (fused, no collective) "
               "+ device barrier",
               "copy": "pushed to every rank by the copy engines over NVLink, sub-block by sub-block, while the next "
               "sub-block's SpMV runs (%d sub-blocks) + device barrier" % len(self.subs),
               "pipeline": "pushed to every rank by %s, followed by a device barrier over all ranks (two y buffers): step k's "
               "exchange overlaps step k+1's SpMV, a step's y is complete everywhere one step later, the pipe is drained "
               "inside the timed region" % (
                   (self.SCHEME_HOW[self.scheme_kind] % self.scheme_ctas if "%d" in self.SCHEME_HOW[self.scheme_kind]
                    else self.SCHEME_HOW[self.scheme_kind]) if self.scheme else "?"),
               "none": "kept local"}[self.exchange if self.world > 1 else "none"]
        self._exchange_how = how
        return "row blocks balanced by nnz, %d ranks; x replicated; y %s" % (self.world, how)

    def set_x(self, x, stream=None):
        """The x of the following steps (constant over the reference's -n loop): smvp_csr_set_x_device on every
        block, so a handle that relabels its column space permutes x once here and not once per pass."""
        self._x_keep = x
        for A in self.subs:
            A.set_x_device(x, stream)
        self.x = None  # passes use the x declared above

    def _timed_mult(self, A, y, main):
        if self.spmv_events is not None:
            self.spmv_events[0].record(main)
        A.mult_device(self.x, y, self.variant, main)
        if self.spmv_events is not None:
            self.spmv_events[1].record(main)

    def multiply(self, stream=None):
        import torch

        main = stream if stream is not None else torch.cuda.current_stream()
        if self.y_fan is not None:
            if self.spmv_events is not None:
                self.spmv_events[0].record(main)
            self.A.mult_device_fanout(self.x, self.y_fan, self.variant, stream)
            if self.spmv_events is not None:
                self.spmv_events[1].record(main)
        elif self.exchange == "pipeline" and self.symm is not None:
            b = self.k % self.nbuf
            if self.copy_pending[b]:  # the push that still reads this source buffer (two steps ago) must be done
                main.wait_event(self.copy_done[b])
            self.y_local = self._src(b)
            self.y_full = self.y_sym[b * self.M:(b + 1) * self.M]
            self._timed_mult(self.A, self.y_local, main)  # the event bracket opens AFTER the wait: SpMV time only
            self.spmv_done[b].record(main)
            self.push_stream.wait_event(self.spmv_done[b])
            self._push(b, main)
        elif self.peer_views is not None:
            off = 0
            self.y_full = self.y_sym[off:off + self.M]
            self.y_local = self.y_full[self.r0:self.r1]
            if self.spmv_events is not None:
                self.spmv_events[0].record(main)
            for g, A in enumerate(self.subs):
                a0, a1 = off + self.sub_bounds[g], off + self.sub_bounds[g + 1]
                A.mult_device(self.x, self.y_sym[a0:a1], self.variant, main)
                self.sub_events[0][g].record(main)
                for pv, cs in zip(self.peer_views, self.copy_streams):
                    with torch.cuda.stream(cs):
                        cs.wait_event(self.sub_events[0][g])
                        pv[a0:a1].copy_(self.y_sym[a0:a1], non_blocking=True)
            if self.spmv_events is not None:
                self.spmv_events[1].record(main)
        else:
            self._timed_mult(self.A, self.y_write if self.y_write is not None else self.y_local, main)

    def exchange_y(self, stream=None):
        if self.world > 1 and self.exchange == "nccl":
            import torch.distributed as dist

            if dist.get_backend() == "nccl":
                allgather_padded(dist, self.y_pad, self.y_full, self.bounds, self.rank, self.per)
            else:
                self.y_full[self.r0:self.r1] = self.y_local
                allgather_v(dist, self.y_full, self.bounds, self.rank)
        elif self.exchange == "pipeline" and self.symm is not None:
            b = self.k % self.nbuf
            self.copy_done[b].record(self.push_stream)
            self.copy_pending[b] = True
            self.k += 1
        elif self.symm is not None:
            if self.copy_stream is not None:
                import torch

                main = stream if stream is not None else torch.cuda.current_stream()
                for cs in self.copy_streams:
                    main.wait_stream(cs)
            self.symm.barrier(channel=0)  # every rank's stores have landed everywhere

    def finish(self, stream=None):
        """Drain whatever the exchange still has in flight (only "pipeline" defers anything)."""
        if self.exchange == "pipeline" and self.symm is not None:
            import torch

            main = stream if stream is not None else torch.cuda.current_stream()
            main.wait_stream(self.push_stream)

    def last_y(self):
        """The full y of the LAST completed step (after finish()), as this rank holds it."""
        if self.exchange == "pipeline" and self.symm is not None:
            b = (self.k - 1) % self.nbuf
            return self.y_sym[b * self.M:(b + 1) * self.M]
        return self.y_full

    def step(self, stream=None):
        self.multiply(stream)
        self.exchange_y(stream)

    @property
    def e2e_api(self):
        """What one end-to-end step does (read after the steps: the mode may depend on the plan the library chose)."""
        if self.world == 1:
            return "smvp_csr_mult(A, x_host, y_host, iters=1) [C ABI, pinned host buffers]"
        if self._e2e_mode() == "window":
            return ("every rank: smvp_csr_mult(A_block, x_host, y_host_block, iters=1) [C ABI, pinned host buffers]; the "
                    "pipelined pass uploads only the window of x the row block reads and downloads the block's rows; "
                    "the host holds all of y, no device-side exchange of y on this path")
        self.partition_desc
        return ("H2D of each rank's 1/N slice of x -> NCCL all-gather of x -> smvp_csr_mult_device -> %s -> D2H of "
                "each rank's y block" % self._exchange_how)

    def _e2e_mode(self):
        """"window": the host call per rank (uploads the window of x the block reads); "slices": 1/N slice per rank +
        all-gather.  A relabelled block belongs to a power-law matrix and reads (nearly) every column: its window is
        the whole vector, so the slices scheme moves N times less over PCIe there."""
        forced = os.environ.get("SMVP_E2E_MODE")
        if forced in ("window", "slices"):
            return forced
        return "slices" if self.A.x_relabel == 1 else "window"

    def e2e_step(self, hx, hy, stream):
        import ctypes

        if self.world == 1:
            # the reference-facing C-ABI call with host buffers: H2D x, one multiply, D2H y, synchronous
            rc = self.eng.lib().smvp_csr_mult(self.A._h, ctypes.c_void_p(hx.data_ptr()), ctypes.c_void_p(hy.data_ptr()), 1,
                                             None, self.variant)
            if rc != 0:
                raise self.eng.SmvpError(rc, "smvp_csr_mult")
        elif self._e2e_mode() == "window":
            # every rank makes the reference-facing C-ABI call on ITS row block with the whole host vector: the
            # pipelined pass uploads only the window of x the block reads (for a banded matrix 1/N of the vector plus
            # the band; a block that reads every column uploads all of it), multiplies tile range by tile range as the
            # window arrives, and sends each finished range of its rows down to the host.  The host ends up with all
            # of y, one block per rank; the device-side exchange of y is not part of this path (nothing on the
            # devices consumes y here).
            base = hy.data_ptr()
            for g, A in enumerate(self.subs):
                off = 8 * (self.sub_bounds[g] - self.r0)
                rc = self.eng.lib().smvp_csr_mult(A._h, ctypes.c_void_p(hx.data_ptr()), ctypes.c_void_p(base + off), 1, None,
                                                 self.variant)
                if rc != 0:
                    raise self.eng.SmvpError(rc, "smvp_csr_mult")
        else:
            # SMVP_E2E_MODE=slices: every rank uploads only ITS 1/N slice of x over PCIe (the host vector crosses the
            # bus once per step, job-wide), the slices are all-gathered over NVLink, then the device step with its
            # exchange of y, then every rank downloads its block
            import torch
            import torch.distributed as dist

            per = -(-self.N // self.world)
            if getattr(self, "_xpad", None) is None:
                self._xpad = torch.zeros(per * self.world, dtype=torch.float64, device="cuda")
            s0 = self.rank * per
            s1 = min(self.N, s0 + per)
            if s1 > s0:
                self._xpad[s0:s1].copy_(hx[s0:s1], non_blocking=True)
            dist.all_gather_into_tensor(self._xpad, self._xpad[s0:s0 + per])
            self.set_x(self._xpad[:self.N], stream)
            self.step(stream)
            hy.copy_(self.y_local, non_blocking=True)
            stream.synchronize()

    @property
    def kernel_name(self):
        """The kernel a pass runs; the merge variant of a handle with the row-pattern plan runs the pattern kernel
        (the plan is decided at the first pass, so read this after it)."""
        if self.variant_name == "vector":
            return "csr_vector_kernel"
        return "csr_pattern_kernel" if self.A.row_patterns > 0 else "csr_merge_warp_kernel"

    def measured_traffic_bytes(self):
        return _measured_traffic(self.kernel_name)

    def plan_desc(self):
        """What the multiply does beyond the plain kernel (decided by the library from the matrix, reported as is)."""
        if self.variant_name == "merge" and self.A.row_patterns > 0:
            return ("rows share %d column-offset patterns (smvp_csr_info_t.row_patterns): the kernel streams pattern ids "
                    "instead of col_ind, and the values as %s (smvp_csr_info_t.value_bytes = %d: %s)"
                    % (self.A.row_patterns, {2: "fp16", 4: "fp32", 8: "fp64"}.get(self.A.value_bytes, "?"), self.A.value_bytes,
                       "fp64" if self.A.value_bytes == 8 else "every value converts to it and back exactly"))
        if self.A.x_relabel == 1:
            return ("column space relabelled by popularity (smvp_csr_info_t.x_relabel = 1): the kernels read rank-ordered "
                    "column indices and a permuted copy of x formed ONCE per x by smvp_csr_set_x_device, outside the "
                    "steps -- x is constant over the -n loop, the reference permutes x once for TJDS the same way "
                    "(main-cli.c:907-923); e2e pays the permutation every step")
        return "natural column order"

    def free(self):
        for A in self.subs:
            A.free()
        self.y_full = self.y_local = self.peer_views = self.y_sym = self.y_src = self._y_src_raw = self.y_pad = None


class ColBlockTjds:
    """y = A x with A in TJDS, columns cut into nnz-balanced blocks over `world` ranks; partial y reduce-scattered."""

    def __init__(self, eng, source, rank, world, variant=0, exchange="nccl", release_source=False):
        import torch

        self.eng, self.rank, self.world, self.variant, self.exchange = eng, rank, world, variant, exchange
        self.M, self.N = source.rows, source.cols
        self.bounds = balanced_bounds(source.col_prefix, self.N, world)
        self.c0, self.c1 = self.bounds[rank], self.bounds[rank + 1]
        r, c, v = source.col_block(self.c0, self.c1)
        self.local_nnz = r.n
        self.T = eng.TjdsMatrix.build_device(r, c, v, self.M, self.c1 - self.c0, r.n)
        for a in (r, c, v):
            a.free()
        if hasattr(source, "release") and release_source:
            source.release()
        self.global_nnz = source.nnz
        # ndiag of the whole matrix is the max over ranks of the local ndiag
        nd = self.T.ndiag
        if world > 1:
            import torch.distributed as dist

            t = torch.tensor([nd], dtype=torch.int64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            nd = int(t[0])
        self.ndiag = nd
        self.global_bytes_per_mult = 12 * source.nnz + 4 * (nd + 1) + 8 * self.N + 8 * self.M
        self.local_bytes_per_mult = self.T.bytes_per_mult
        self.Mp = -(-self.M // (2 * world)) * 2 * world  # blocks of an even number of rows: 16-byte aligned for 128-bit loads
        self.y_partial = torch.zeros(self.Mp, dtype=torch.float64, device="cuda")
        self.y_owned = torch.zeros(self.Mp // world, dtype=torch.float64, device="cuda")
        # deterministic variant: the N-way sum is done in rank order by our own kernel after an all-to-all of the blocks,
        # so the bits do not depend on NCCL's reduction order (SMVP_TJDS_ORDERED=0/1 forces it off/on for either variant)
        forced = os.environ.get("SMVP_TJDS_ORDERED")
        self.ordered = world > 1 and exchange == "nccl" and (
            forced == "1" or (forced != "0" and variant != eng.TJDS_ATOMIC))
        self.scratch, self.symm, self.part_ptrs = None, None, None
        if self.ordered:
            # the partial y lives in symmetric memory: the owner of a row block pulls that block from every rank over
            # NVLink and adds in rank order (smvp_sum_ordered_ptrs_device), between two device-side barriers.
            # SMVP_TJDS_ORDERED_PULL=0: all-to-all of the blocks (NCCL) + local ordered sum instead.
            if os.environ.get("SMVP_TJDS_ORDERED_PULL", "1") != "0":
                try:
                    import torch.distributed as dist
                    import torch.distributed._symmetric_memory as symm_mem

                    buf = symm_mem.empty(self.Mp, dtype=torch.float64, device=torch.device("cuda", torch.cuda.current_device()))
                    buf.zero_()
                    self.symm = symm_mem.rendezvous(buf, dist.group.WORLD.group_name)
                    self.y_partial = buf
                    per = self.Mp // world
                    self.part_ptrs = [int(self.symm.buffer_ptrs[k]) + 8 * per * rank for k in range(world)]
                except Exception:  # noqa: BLE001  (no peer access on this box)
                    self.symm = None
            if self.symm is None:
                self.scratch = torch.empty(self.Mp, dtype=torch.float64, device="cuda")
        self.local_rows_out = self.Mp // world
        self.variant_name = {eng.TJDS_ATOMIC: "atomic", eng.TJDS_DETERMINISTIC: "deterministic",
                             eng.TJDS_DETERMINISTIC_FAST: "deterministic_fast"}[variant]
        self.kernel_name = "tjds_%s_kernel" % ("atomic" if variant == eng.TJDS_ATOMIC else "det")
        self.partition_desc = ("column blocks balanced by nnz, %d ranks; x sliced; partial y %s" %
                               (world, (("pulled block-wise over NVLink peer mappings" if self.symm is not None else
                                         "exchanged block-wise (NCCL all-to-all)") + " and summed in rank order by our own "
                                        "kernel: reproducible run to run" if self.ordered else
                                        "reduce-scattered over NCCL") if (world > 1 and exchange == "nccl") else "kept local"))
        self.e2e_api = ("smvp_tjds_mult(A, x_host, y_host, iters=1) [C ABI, pinned host buffers]" if world == 1 else
                        "H2D x slice -> smvp_tjds_set_x_device + smvp_tjds_mult_device -> NCCL reduce-scatter -> D2H y block")
        self.x = None
        self.spmv_events = None

    def plan_desc(self):
        if self.T.y_relabel == 1:
            return ("row space relabelled by popularity (smvp_tjds_info_t.y_relabel = 1): the kernels scatter through "
                    "rank-ordered row indices, a last pass inside every step restores the row order of y")
        return "natural row order"

    def set_x(self, x, stream=None):
        self.x = x
        self.T.set_x_device(x[self.c0:self.c1], stream)

    def multiply(self, stream=None):
        if self.spmv_events is not None:
            import torch

            main = stream if stream is not None else torch.cuda.current_stream()
            self.spmv_events[0].record(main)
            self.T.mult_device(self.y_partial, self.variant, 0, stream)
            self.spmv_events[1].record(main)
        else:
            self.T.mult_device(self.y_partial, self.variant, 0, stream)

    def exchange_y(self, stream=None):
        if self.world > 1 and self.exchange == "nccl":
            import torch.distributed as dist

            if self.ordered and self.symm is not None:
                self.symm.barrier(channel=0)  # every rank's partial y is complete
                self.eng.sum_ordered_ptrs_device(self.y_owned, self.part_ptrs, self.Mp // self.world, stream)
                self.symm.barrier(channel=1)  # nobody refills its partial y while a peer still reads it
            elif self.ordered:
                reduce_scatter_ordered(dist, self.eng, self.y_owned, self.y_partial, self.scratch, self.rank, self.world, stream)
            else:
                reduce_scatter_sum(dist, self.y_owned, self.y_partial, self.rank)

    def finish(self, stream=None):
        pass

    def last_y(self):
        """This rank's block of y (rows [rank * Mp/world, ...)) after the exchange; without an exchange the partial y."""
        if self.world > 1 and self.exchange == "nccl":
            return self.y_owned
        return self.y_partial

    def step(self, stream=None):
        self.multiply(stream)
        self.exchange_y(stream)

    def e2e_step(self, hx, hy, stream):
        import ctypes

        if self.world == 1:
            rc = self.eng.lib().smvp_tjds_mult(self.T._h, ctypes.c_void_p(hx.data_ptr()), ctypes.c_void_p(hy.data_ptr()), 1,
                                              None, self.variant, 0)
            if rc != 0:
                raise self.eng.SmvpError(rc, "smvp_tjds_mult")
        else:
            # a column block needs only its own slice of x
            self.x[self.c0:self.c1].copy_(hx[self.c0:self.c1], non_blocking=True)
            self.T.set_x_device(self.x[self.c0:self.c1], stream)
            self.step(stream)
            hy.copy_(self.y_owned, non_blocking=True)
            stream.synchronize()

    def measured_traffic_bytes(self):
        return _measured_traffic(self.kernel_name)

    def free(self):
        self.T.free()
        self.y_partial = self.y_owned = self.scratch = None
