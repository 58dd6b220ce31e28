#!/usr/bin/env python3
"""bench.py -- headline benchmark of the CSR / TJDS SpMV path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload stencil27|rmat] [--format csr|tjds] [--variant ...] [--no-secondary]
                    [--dump-outputs DIR]

Default (N=1): BASELINE.json configs[2], the HBM-roofline run the metric is quoted on --
27-point stencil on a 369^3 grid (50 243 409 rows, 1 349 232 625 nnz, fp64), CSR, one SpMV per step.
N>1: the same matrix cut into nnz-balanced row blocks, x replicated, y all-gathered (strong scaling).

One JSON line on stdout (rank 0).  `value` = effective GB/s = algorithmic bytes of one SpMV
(12 nnz + 4 (M+1) + 8 N + 8 M for CSR; 12 nnz + 4 (ndiag+1) + 8 N + 8 M for TJDS) / step time, inputs
resident in HBM.  `e2e` = the same metric through the host-buffer C-ABI call (x from pinned host
memory, y back to pinned host memory, copies inside the timed region).

The run verifies itself: after the timed region every rank checks the y it holds (`parity`: closed form of the
stencil for x = ones, exact; agreement of two different kernels on the timed x within 1e-12; at N > 1 the blocks of
the all-gathered y bit-identical to their owners' through an exact 64-bit checksum) and the run FAILS otherwise.

`secondary` carries the other BASELINE.json configurations measured in the same process at the same N, a few steps
each: stencil TJDS atomic / deterministic (configs[2] names both formats), R-MAT 2^26 CSR (configs[3]) and R-MAT
TJDS atomic / deterministic (configs[4]), each with its own parity check against the CSR result.

`--impl reference` times the reference's own CPU loop (oracle/_ref when it was built, else the
oracle port) on a bounded sample of the same workload; `config.workload` names the sample it actually ran.

`--dump-outputs DIR` writes the y of the last timed step of every configuration the run times to DIR/<name>.npy
(float64): `y.npy` for the headline, `y_<secondary name>.npy` for the others.  A y longer than its row budget (2^22
rows for the headline, 2^19 for each secondary: under 64 MB in all) is written as a sample of rows drawn with a fixed
seed.  The inputs are seeded too, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import re
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

METRIC = "spmv_effective_bandwidth"
UNIT = "GB/s"
TOL = 1e-12  # relative L2, fp64 (north_star)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=100)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="stencil27", choices=["stencil27", "rmat"])
    p.add_argument("--grid", type=int, default=369, help="stencil27: grid edge (369 -> 50.2M rows, 1.35B nnz)")
    p.add_argument("--scale", type=int, default=26, help="rmat: log2(rows)")
    p.add_argument("--edge-factor", type=int, default=16)
    p.add_argument("--format", default="csr", choices=["csr", "tjds"])
    p.add_argument("--variant", default="auto", choices=["auto", "vector", "merge", "atomic", "deterministic", "fast"])
    p.add_argument("--exchange", default="auto", choices=["auto", "pipeline", "copy", "multicast", "p2p", "nccl", "none"],
                   help="N>1: collective after the multiply (allgather of y for CSR, reduce-scatter for TJDS)")
    p.add_argument("--sub-blocks", type=int, default=4, help="exchange=copy: sub-blocks per rank")
    # 128^3: x is 16.8 MB (beyond any host L2); the unmodified reference spends ~80 s in its own qsort of the 55.7 M
    # entries (main-cli.c:340) before the timed loop -- 200^3 would take 6 minutes of sorting for the same GB/s
    p.add_argument("--cpu-grid", type=int, default=128, help="grid edge of the bounded CPU sample (stencil27)")
    p.add_argument("--cpu-scale", type=int, default=21, help="scale of the bounded CPU sample (rmat)")
    p.add_argument("--cpu-iters", type=int, default=10)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-all-cores", action="store_true", help="skip the extra all-cores CPU figure")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-secondary", action="store_true", help="skip the other BASELINE.json configurations")
    p.add_argument("--secondary-steps", type=int, default=8)
    p.add_argument("--secondary-scale", type=int, default=26, help="R-MAT scale of the secondary configurations")
    p.add_argument("--no-tune", action="store_true", help="N>1: keep the default exchange scheme (no warm-up tuning)")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the y of the last timed step of every configuration to "
                   "DIR/<name>.npy (float64, a seeded sample of rows when y is large)")
    args = p.parse_args()
    for name in ("steps", "secondary_steps", "cpu_iters"):
        if getattr(args, name) < 1:
            p.error("--%s must be at least 1" % name.replace("_", "-"))
    if args.warmup < 0:
        p.error("--warmup must not be negative")
    if args.dump_outputs and args.format == "tjds" and args.gpus > 1 and args.exchange == "none":
        # without the reduce-scatter every rank holds a partial sum over its columns, no rank holds rows of y
        p.error("--dump-outputs with --format tjds at --gpus > 1 needs an exchange (not --exchange none)")
    return args


# --------------------------------------------------------------------------------------- helpers
def load_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self.interval = float(os.environ.get("SMVP_BENCH_SAMPLE_MS", "10")) * 1e-3
        self.stop_flag = threading.Event()
        self.active = threading.Event()  # set for the duration of the timed region: only then are samples kept
        self.ok = False
        try:
            import pynvml

            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            # first calls resolve the NVML entry points (milliseconds, under the GIL): done here, not in the timed region
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag.is_set():
            try:
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if self.active.is_set():
                    self.samples.append(mhz)
                    for bit, name in self.REASONS.items():
                        if r & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.interval)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def csr_bytes(rows, cols, nnz):
    return 12 * nnz + 4 * (rows + 1) + 8 * cols + 8 * rows


def tjds_bytes(rows, cols, nnz, ndiag):
    return 12 * nnz + 4 * (ndiag + 1) + 8 * cols + 8 * rows


DUMP_ROWS = 1 << 22            # --dump-outputs: rows of the headline y (32 MB of float64)
DUMP_ROWS_SECONDARY = 1 << 19  # rows of each of the 7 secondary y (4 MB each)


def dump_rows(rows, limit):
    """The rows of a y that --dump-outputs writes: all of them up to `limit`, else at most `limit` rows drawn with a
    fixed seed, ascending (the same rows for the same arguments in every run)."""
    if rows <= limit:
        return np.arange(rows)
    return np.unique(np.random.default_rng(0).integers(0, rows, limit))


def output_name(config_name):
    """File name of a secondary configuration's y: "R-MAT scale 26 CSR" -> "y_r_mat_scale_26_csr"."""
    return "y_" + re.sub(r"[^0-9a-z]+", "_", config_name.lower()).strip("_")


def save_output(args, name, values):
    os.makedirs(args.dump_outputs, exist_ok=True)
    np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(values, np.float64))


# --------------------------------------------------------------------------------------- CPU arm
def stencil_coo_numpy(g):
    """27-point stencil COO on a g^3 grid, (row,col)-sorted, {26,-1} values -- numpy only (no engine).  Built plane by
    plane straight in (row, col) order: the 27 offsets ascend with (dz, dy, dx), so no sort is needed."""
    from oracle import oracle

    offs = [(dz, dy, dx) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
    rows, cols = [], []
    plane = np.arange(g * g, dtype=np.int64)
    ix, iy = plane % g, plane // g
    for iz in range(g):
        base = plane + iz * g * g
        ok = np.stack([(ix + dx >= 0) & (ix + dx < g) & (iy + dy >= 0) & (iy + dy < g) & (0 <= iz + dz < g)
                       for dz, dy, dx in offs], axis=1)
        col = np.stack([base + dx + g * (dy + g * dz) for dz, dy, dx in offs], axis=1)
        rows.append(np.repeat(base, ok.sum(axis=1)))
        cols.append(col[ok])
    row = np.concatenate(rows)
    col = np.concatenate(cols)
    return oracle.make_coo(row, col, np.where(row == col, 26.0, -1.0))


def rmat_coo_numpy(scale, edge_factor):
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import synth_ref

    return synth_ref.rmat(scale, edge_factor << scale, seed=42)


def cpu_sample_desc(args):
    if args.workload == "stencil27":
        g = args.cpu_grid
        return "27-point stencil %d^3 (%d rows, %d nnz)" % (g, g ** 3, (3 * g - 2) ** 3)
    return "R-MAT scale %d, edge factor %d" % (args.cpu_scale, args.edge_factor)


def cpu_reference_run(args, iters, drop=0):
    """The reference's CPU implementation of the path on a bounded sample of the workload, 1 thread
    (the reference is single-threaded: main-cli.c has no threads, SURVEY.md section 0)."""
    from oracle import oracle

    if args.workload == "stencil27":
        g = args.cpu_grid
        coo = stencil_coo_numpy(g)
        m = n = g ** 3
        sample = "27-point stencil %d^3 (%d rows, %d nnz), %d iterations, x = ones" % (g, m, len(coo), iters)
    else:
        coo = rmat_coo_numpy(args.cpu_scale, args.edge_factor)
        m = n = 1 << args.cpu_scale
        sample = "R-MAT scale %d, edge factor %d (%d rows, %d nnz after dedupe), %d iterations" % (
            args.cpu_scale, args.edge_factor, m, len(coo), iters)
    nnz = len(coo)
    if args.format == "csr":
        nbytes = csr_bytes(m, n, nnz)
        # the verbatim reference leaves row_ptr slots unwritten for empty rows (U3): only usable on
        # matrices without empty rows, i.e. the stencil
        if oracle.ref_available() and args.workload == "stencil27":
            kind = "reference"
            y, ms = oracle.ref_csr_compute(coo, m, iters)
            what = "oracle/_ref/libsmvp_ref.so: the unmodified smvp_csr_compute (main-cli.c:325), its own clock_gettime bracket"
        else:
            kind = "port"
            rp, ci, va = oracle.csr_build(coo, m, n)
            y, ms = oracle.csr_mult_timed(rp, ci, va, np.ones(n), iters)
            what = "oracle/smvp_oracle.c: oracle_csr_mult_timed (restatement of main-cli.c:402-420)"
    else:
        kind = "port"  # the reference's TJDS build is O(nnz*N) (main-cli.c:894-904): not runnable at this size
        t = oracle.tjds_build(coo, m, n)
        nbytes = tjds_bytes(m, n, nnz, t.ndiag)
        y, ms = oracle.tjds_mult_timed(t, np.ones(n), iters)
        what = "oracle/smvp_oracle.c: oracle_tjds_mult_timed (restatement of main-cli.c:1004-1024, all diagonals)"
    ms = np.asarray(ms)[drop:]
    avg_ms = float(ms.mean())
    res = {"value": nbytes / (avg_ms * 1e-3) / 1e9, "unit": UNIT, "cores": 1, "kind": kind,
           "sample": sample + "; " + what, "gflops": 2 * nnz / (avg_ms * 1e-3) / 1e9, "ms_per_step": avg_ms,
           "min_ms": float(ms.min()), "rows": m, "nnz": nnz, "x_bytes": 8 * n, "y": y}
    if args.format == "csr" and not args.no_all_cores:
        # NOT the reference (it is single-threaded): its loop over nnz-balanced row blocks on every core of the box,
        # same sample, so the 1-thread figure can be put in proportion.  Reported beside it, never instead of it.
        cores = os.cpu_count() or 1
        rp, ci, va = oracle.csr_build(coo, m, n)
        _, ms_mt = oracle.csr_mult_timed_mt(rp, ci, va, np.ones(n), max(min(iters, 10), 3) + 2, cores)
        mt = float(np.asarray(ms_mt)[2:].mean())
        res["all_cores"] = {"value": nbytes / (mt * 1e-3) / 1e9, "unit": UNIT, "cores": cores, "kind": "port",
                            "note": "oracle/smvp_oracle.c oracle_csr_mult_timed_mt: the reference loop (main-cli.c:410-416) "
                                    "row-parallel on all host cores; the reference itself is single-threaded"}
    return res


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.time()
    # warm-up iterations are part of the same call; the first `warmup` timings are dropped
    res = cpu_reference_run(args, args.steps + args.warmup, drop=args.warmup)
    if args.dump_outputs:
        save_output(args, "y", res["y"][dump_rows(len(res["y"]), DUMP_ROWS)])
    # config.workload names what THIS arm ran: a bounded sample, not the GPU arm's full-size matrix (the reference's
    # builder cannot run at that size: stack VLA main-cli.c:1426, and one CPU pass over it would take seconds)
    cfg = workload_config(args, None)
    cfg["workload"] = ("%s, fp64, %s -- bounded CPU SAMPLE of the GPU arm's workload (%s); x is %d MB, beyond the "
                       "host's L2" % (cpu_sample_desc(args), args.format.upper(), cfg["workload"], res["x_bytes"] >> 20))
    cfg["same_config_as_gpu_arm"] = False
    cfg["rows"], cfg["nnz"] = res["rows"], res["nnz"]
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "gflops": res["gflops"],
        "cpu_baseline": dict({"value": res["value"], "unit": UNIT, "cores": 1, "kind": res["kind"], "sample": res["sample"]},
                             **({"all_cores": res["all_cores"]} if "all_cores" in res else {})),
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    print_json(line)


def workload_config(args, extra):
    if args.workload == "stencil27":
        g = args.grid
        w = "27-point stencil %d^3 (BASELINE.json configs[2]): %d rows, %d nnz, fp64, %s" % (
            g, g ** 3, (3 * g - 2) ** 3, args.format.upper())
    else:
        w = "R-MAT scale %d edge factor %d (BASELINE.json configs[3]/[4]), fp64, %s" % (args.scale, args.edge_factor,
                                                                                         args.format.upper())
    cfg = {"workload": w, "format": args.format, "variant": args.variant,
           "l2_hygiene": "matrix streams (>= 12 B/nnz) are far larger than the 126 MB L2; no flush needed"}
    if extra:
        cfg.update(extra)
    return cfg


# --------------------------------------------------------------------------------------- GPU arm
class Ctx:
    """What every measurement needs: torch, the engine, the rank layout and the stream."""

    def __init__(self, torch, dist, eng, sdist, world, rank, local_rank):
        self.torch, self.dist, self.eng, self.sdist = torch, dist, eng, sdist
        self.world, self.rank, self.local_rank = world, rank, local_rank
        self.stream = torch.cuda.current_stream()
        self.peak, self.peak_src = load_peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]


def timed_steps(ctx, op, steps, warmup, sample_clocks=True):
    """`warmup` untimed steps, then EXACTLY `steps` steps between a barrier + synchronize on both sides; device time by
    CUDA events on the launching stream, MAX over ranks.  The SpMV launch of every step has its own event bracket
    (opened after any wait for the exchange of an earlier step)."""
    torch, stream = ctx.torch, ctx.stream
    # the poller thread is started BEFORE the warm-up steps (its start-up costs the launching thread milliseconds of GIL and
    # driver time: measured at 2 GPUs, 1.49 ms per step with the thread already running, 1.64 ms when it was started at
    # the first timed step) and only keeps the samples it takes inside the timed region
    # N > 1: only rank 0 polls NVML (its GPU's clocks are the ones reported).  A poll takes milliseconds inside the driver;
    # with every rank polling, each one's hiccup reaches all ranks through the per-step barrier of the exchange
    # (measured at 8 GPUs, tools/probe_steps.py: 0.628 ms per step without the pollers, 0.65 - 0.72 ms with 8 of them)
    sampler = ClockSampler(ctx.local_rank) if (sample_clocks and ctx.rank == 0 and
                                               os.environ.get("SMVP_BENCH_SAMPLE_MS") != "0") else None
    if sampler:
        sampler.start()
    for _ in range(max(warmup, 3)):
        op.step(stream)
    op.finish(stream)
    ctx.barrier()
    launches0 = ctx.eng.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    e_begin, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler:
        sampler.active.set()
    e_begin.record(stream)
    for k in range(steps):
        op.spmv_events = ev[k]
        op.multiply(stream)      # the SpMV kernel(s) of this rank
        op.exchange_y(stream)    # N>1: allgather / reduce-scatter
    op.finish(stream)            # drains a pipelined exchange: still inside the timed region
    e_end.record(stream)
    ctx.barrier()
    op.spmv_events = None
    if sampler:
        sampler.active.clear()
        sampler.stop_flag.set()
        sampler.join()
    launches = ctx.eng.launch_count() - launches0
    total_ms = e_begin.elapsed_time(e_end)
    per_step = np.asarray([a.elapsed_time(b) for a, b in ev])
    kern_ms = float(per_step.mean())
    total_max, kern_max = ctx.max_over_ranks([total_ms, kern_ms])
    return {"ms_per_step": total_max / steps, "kern_ms_local": kern_ms, "kern_ms_max": kern_max, "launches": int(launches),
            "kern_ms_min": float(per_step.min()), "kern_ms_median": float(np.median(per_step)),
            "clocks": sampler.result() if sampler else None}


def dump_output(ctx, args, name, op, limit):
    """--dump-outputs: the y of op's last step (call it before anything else runs op), the rows of dump_rows(M, limit)
    gathered from the ranks that hold them, written by rank 0."""
    if not args.dump_outputs:
        return
    torch = ctx.torch
    if isinstance(op, ctx.sdist.ColBlockTjds):  # rank g holds the g-th of `world` equal slices of the padded y
        per = op.Mp // ctx.world
        row0 = ctx.rank * per
        held = op.last_y()[:max(0, min(per, op.M - row0))]
    else:
        row0 = op.r0
        held = op.last_y()[op.r0:op.r1]
    idx = torch.from_numpy(dump_rows(op.M, limit)).to("cuda")
    mine = (idx >= row0) & (idx < row0 + held.numel())
    vals = torch.full(idx.shape, float("-inf"), dtype=torch.float64, device="cuda")
    vals[mine] = held[idx[mine] - row0]
    if ctx.world > 1:
        ctx.dist.all_reduce(vals, op=ctx.dist.ReduceOp.MAX)  # every row is held by exactly one rank
    if ctx.rank == 0:
        save_output(args, name, vals.cpu().numpy())


def block_checksums(torch, y, bounds):
    """Exact 64-bit checksum of every block of y: the int64 views summed with wrap-around (order-independent)."""
    return torch.stack([y[bounds[g]:bounds[g + 1]].view(torch.int64).sum() for g in range(len(bounds) - 1)])


def stencil_counts(torch, g, r0, r1):
    """Entries per row of the 27-point stencil on a g^3 grid, rows [r0, r1): closed form, independent of the engine."""
    r = torch.arange(r0, r1, dtype=torch.int64, device="cuda")

    def span(i):
        return 3 - (i == 0).to(torch.int64) - (i == g - 1).to(torch.int64) if g > 1 else torch.ones_like(i)

    return span(r % g) * span((r // g) % g) * span(r // (g * g))


def rel_l2(torch, a, b):
    nb = float(torch.linalg.norm(b))
    return float(torch.linalg.norm(a - b)) / (nb if nb > 0 else 1.0)


def check_csr_parity(ctx, op, x, stencil_grid=None):
    """In-run verification of a row-block CSR operator (every rank, after the timed region).  Returns a dict; raises on
    failure.  (1) two different kernels agree on the rows of this rank for the timed x; (2) N > 1: every block of the
    all-gathered y this rank holds is bit-identical to its owner's (exact checksums); (3) stencil with the {26,-1}
    values: x = ones gives y_r = 27 - (entries in row r), exactly, on this rank's rows."""
    torch, eng, stream = ctx.torch, ctx.eng, ctx.stream
    out = {}
    op.step(stream)
    op.finish(stream)
    ctx.barrier()
    y_full = op.last_y()
    mine = y_full[op.r0:op.r1].clone()
    other = eng.CSR_VECTOR if op.variant_name == "merge" else eng.CSR_MERGE
    y2 = torch.empty_like(mine)
    off = 0
    for A, (a0, a1) in zip(op.subs, zip(op.sub_bounds[:-1], op.sub_bounds[1:])):
        A.mult_device(None, y2[off:off + (a1 - a0)], other, stream)
        off += a1 - a0
    torch.cuda.synchronize()
    out["kernel_vs_kernel_rel_l2"] = rel_l2(torch, y2, mine)
    if ctx.world > 1 and op.exchange != "none":
        sums = block_checksums(torch, y_full, op.bounds)
        owners = [torch.empty_like(sums) for _ in range(ctx.world)]
        ctx.dist.all_gather(owners, sums)
        bad = [g for g in range(ctx.world) if int(owners[g][g]) != int(sums[g])]
        out["allgather_blocks_bit_identical"] = not bad
        if bad:
            raise SystemExit("PARITY FAILED: rank %d holds blocks %s of y that differ from their owners'" % (ctx.rank, bad))
    if stencil_grid is not None:
        ones = torch.ones(op.N, dtype=torch.float64, device="cuda")
        op.set_x(ones, stream)
        op.step(stream)
        op.finish(stream)
        ctx.barrier()
        expect = (27 - stencil_counts(torch, stencil_grid, op.r0, op.r1)).to(torch.float64)
        got = op.last_y()[op.r0:op.r1]
        exact = bool(torch.equal(got, expect))
        out["stencil_closed_form_exact"] = exact
        if ctx.world > 1 and op.exchange != "none":
            # the other ranks' rows of the gathered y against the closed form too
            full_expect = (27 - stencil_counts(torch, stencil_grid, 0, op.M)).to(torch.float64)
            exact_all = bool(torch.equal(op.last_y(), full_expect))
            out["stencil_closed_form_exact_all_rows"] = exact_all
            exact = exact and exact_all
        op.set_x(x, stream)
        if not exact:
            raise SystemExit("PARITY FAILED: stencil closed form (x = ones) differs on rank %d" % ctx.rank)
    if out["kernel_vs_kernel_rel_l2"] > TOL:
        raise SystemExit("PARITY FAILED: kernels disagree on rank %d: %.3e" % (ctx.rank, out["kernel_vs_kernel_rel_l2"]))
    worst = ctx.max_over_ranks([out["kernel_vs_kernel_rel_l2"]])[0]
    out["parity_max_rel"] = worst
    return out


def check_tjds_parity(ctx, op, y_csr_full, deterministic):
    """Column-block TJDS against the CSR result of the same matrix and x: this rank's block of y within 1e-12; the
    deterministic variant additionally bit-identical run to run (at N > 1 that includes the exchange)."""
    torch, stream = ctx.torch, ctx.stream
    op.step(stream)
    op.finish(stream)
    ctx.barrier()
    per = op.Mp // ctx.world
    lo = ctx.rank * per
    hi = min(lo + per, op.M)
    got = op.last_y()[:hi - lo].clone()
    err = float(torch.linalg.norm(got - y_csr_full[lo:hi])) / max(float(torch.linalg.norm(y_csr_full)), 1e-300)
    out = {"vs_csr_rel_l2": ctx.max_over_ranks([err])[0]}
    if deterministic:
        op.step(stream)
        op.finish(stream)
        ctx.barrier()
        same = bool(torch.equal(op.last_y()[:hi - lo], got))
        same_all = ctx.max_over_ranks([0.0 if same else 1.0])[0] == 0.0
        out["run_to_run_bit_identical"] = same_all
        if not same_all:
            raise SystemExit("PARITY FAILED: deterministic TJDS differs run to run")
    if out["vs_csr_rel_l2"] > TOL:
        raise SystemExit("PARITY FAILED: TJDS vs CSR %.3e" % out["vs_csr_rel_l2"])
    out["parity_max_rel"] = out["vs_csr_rel_l2"]
    return out


def perf_fields(ctx, t, global_bytes, local_bytes, nnz):
    ms = t["ms_per_step"]
    value = global_bytes / (ms * 1e-3) / 1e9
    achieved = local_bytes / (t["kern_ms_local"] * 1e-3) / 1e9
    return {"ms_per_step": ms, "value": value, "unit": UNIT, "gflops": 2 * nnz / (ms * 1e-3) / 1e9,
            "pct_of_hbm_peak_8000": 100.0 * value / 8000.0 / ctx.world,
            "frac_of_measured_peak": value / ctx.peak / ctx.world,
            "kernel_ms": t["kern_ms_local"], "kernel_ms_min": t["kern_ms_min"], "kernel_ms_median": t["kern_ms_median"],
            "kernel_ms_max_over_ranks": t["kern_ms_max"],
            "kernel_frac_of_measured_peak": achieved / ctx.peak, "gpu_launches": t["launches"]}


def make_csr_op(ctx, gen, args, variant, exch, release_source=False):
    """Row-block CSR with the requested exchange ("auto": the first scheme this box supports, in measured order)."""
    torch, dist, eng, sdist = ctx.torch, ctx.dist, ctx.eng, ctx.sdist
    # "auto", in the order measured on B200 (profiles/): the pipelined push (two y buffers, scheme tuned at warm-up);
    # copy engines pushing finished sub-blocks; in-kernel stores to the NVSwitch multicast address; in-kernel unicast
    # fan-out; SpMV followed by an NCCL all-gather as the fallback of last resort
    candidates = ["pipeline", "copy", "multicast", "p2p", "nccl"] if exch == "auto" else [exch]
    op, err = None, None
    for cand in candidates:
        try:
            op = sdist.RowBlockCsr(eng, gen, ctx.rank, ctx.world, variant, exchange=cand,
                                   release_source=(release_source and cand == candidates[-1]), sub_blocks=args.sub_blocks)
        except Exception as e:  # noqa: BLE001  (e.g. no NVSwitch multicast on this box)
            op, err = None, e
        if ctx.world > 1:
            ok = torch.tensor([1 if op is not None else 0], device="cuda")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok[0]) == 0 and op is not None:
                op.free()
                op = None
        if op is not None:
            return op, cand
    raise err if err is not None else RuntimeError("no exchange could be set up on every rank")


def run_secondary(ctx, args, stencil_gen, y_stencil_csr, x_stencil):
    """The other BASELINE.json configurations at this N, a few steps each, every one verified in the run."""
    torch, eng, sdist = ctx.torch, ctx.eng, ctx.sdist
    out = []
    steps = args.secondary_steps
    exch_tjds = "nccl" if ctx.world > 1 else "none"

    def record(name, cfg_ref, op, t, parity, extra=None):
        if ctx.rank != 0:
            return
        d = {"name": name, "baseline_config": cfg_ref, "n_gpus": ctx.world, "steps": steps, "nnz": op.global_nnz,
             "bytes_per_spmv": op.global_bytes_per_mult, "partition": op.partition_desc, "multiply_plan": op.plan_desc(),
             "parity_checked": True, "parity": parity, "parity_max_rel": parity["parity_max_rel"], "clocks": t["clocks"]}
        d.update(perf_fields(ctx, t, op.global_bytes_per_mult, op.local_bytes_per_mult, op.global_nnz))
        if extra:
            d.update(extra)
        out.append(d)

    # ---- stencil TJDS, atomic and deterministic (configs[2] names both formats)
    tjds_variants = (("atomic", eng.TJDS_ATOMIC), ("deterministic", eng.TJDS_DETERMINISTIC),
                     ("deterministic_fast", eng.TJDS_DETERMINISTIC_FAST))
    for vname, variant in tjds_variants:
        name = "stencil %d^3 TJDS %s" % (args.grid, vname)
        op = sdist.ColBlockTjds(eng, stencil_gen, ctx.rank, ctx.world, variant, exchange=exch_tjds)
        op.set_x(x_stencil, ctx.stream)
        t = timed_steps(ctx, op, steps, 3)
        dump_output(ctx, args, output_name(name), op, DUMP_ROWS_SECONDARY)
        parity = check_tjds_parity(ctx, op, y_stencil_csr, variant != eng.TJDS_ATOMIC)
        record(name, "configs[2]", op, t, parity,
               {"ndiag": op.ndiag, "tjds_plan": dict(zip(("skewed_walk", "det_route"), op.T.plan()))})
        op.free()
        del op
    del y_stencil_csr
    torch.cuda.empty_cache()

    # ---- R-MAT: CSR row blocks + all-gather (configs[3]), TJDS column blocks + reduce-scatter (configs[4])
    scale = args.secondary_scale
    gen = sdist.RmatSource(eng, scale, args.edge_factor << scale)
    N = gen.cols
    x = torch.empty(N, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, N, 12345, ctx.stream)
    op, exch = make_csr_op(ctx, gen, args, eng.CSR_AUTO, "none" if ctx.world == 1 else args.exchange)
    op.set_x(x, ctx.stream)
    tuning = None
    if ctx.world > 1 and exch == "pipeline" and not args.no_tune:
        tuning = op.tune_pipeline(ctx.stream)
    t = timed_steps(ctx, op, steps, 3)
    name = "R-MAT scale %d CSR" % scale
    dump_output(ctx, args, output_name(name), op, DUMP_ROWS_SECONDARY)
    parity = check_csr_parity(ctx, op, x)
    y_csr = op.last_y().clone() if ctx.world > 1 else op.y_full.clone()
    record(name, "configs[3]", op, t, parity,
           {"kernel_variant": op.variant_name, "exchange": exch, "exchange_tuning": tuning})
    op.free()
    del op
    torch.cuda.empty_cache()
    for vname, variant in tjds_variants:
        name = "R-MAT scale %d TJDS %s" % (scale, vname)
        op = sdist.ColBlockTjds(eng, gen, ctx.rank, ctx.world, variant, exchange=exch_tjds)
        op.set_x(x, ctx.stream)
        t = timed_steps(ctx, op, steps, 3)
        dump_output(ctx, args, output_name(name), op, DUMP_ROWS_SECONDARY)
        parity = check_tjds_parity(ctx, op, y_csr, variant != eng.TJDS_ATOMIC)
        record(name, "configs[4]", op, t, parity,
               {"ndiag": op.ndiag, "tjds_plan": dict(zip(("skewed_walk", "det_route"), op.T.plan()))})
        op.free()
        del op
        torch.cuda.empty_cache()
    gen.release()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    import smvp_toolkit_b200 as eng

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun (one rank per GPU)" % args.gpus)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from smvp_toolkit_b200 import dist as sdist

    numa_node = sdist.bind_host_near_gpu(local_rank)  # before any page-locked allocation
    ctx = Ctx(torch, dist, eng, sdist, world, rank, local_rank)
    variant_map = {"auto": eng.CSR_AUTO, "vector": eng.CSR_VECTOR, "merge": eng.CSR_MERGE}
    tj_map = {"auto": eng.TJDS_ATOMIC, "atomic": eng.TJDS_ATOMIC, "deterministic": eng.TJDS_DETERMINISTIC,
              "fast": eng.TJDS_DETERMINISTIC_FAST}
    primary_default = args.workload == "stencil27" and args.format == "csr"

    # ---------------- build the shard of this rank
    t_build0 = time.time()
    if args.workload == "stencil27":
        g = args.grid
        M = N = g ** 3
        gen = sdist.StencilSource(eng, g, g, g)
    else:
        M = N = 1 << args.scale
        gen = sdist.RmatSource(eng, args.scale, args.edge_factor << args.scale)
    exch = "none" if world == 1 else args.exchange
    if args.format == "csr":
        op, exch = make_csr_op(ctx, gen, args, variant_map.get(args.variant, eng.CSR_AUTO), exch)
    else:
        op = sdist.ColBlockTjds(eng, gen, rank, world, tj_map.get(args.variant, eng.TJDS_ATOMIC),
                                exchange="nccl" if exch in ("auto", "pipeline", "copy", "multicast", "p2p", "nccl") else "none")
    torch.cuda.synchronize()
    build_s = time.time() - t_build0
    nnz_total = op.global_nnz
    nbytes = op.global_bytes_per_mult
    stream = ctx.stream

    x = torch.empty(N, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, N, 12345, stream)
    op.set_x(x, stream)

    # ---------------- N>1: pick the exchange scheme of the pipelined push (warm-up, outside the timed region)
    tuning = None
    if world > 1 and args.format == "csr" and exch == "pipeline" and not args.no_tune:
        tuning = op.tune_pipeline(stream)

    # ---------------- warm-up, then the timed region: exactly K steps
    t = timed_steps(ctx, op, args.steps, args.warmup)
    dump_output(ctx, args, "y", op, DUMP_ROWS)
    ms_per_step = t["ms_per_step"]
    value = nbytes / (ms_per_step * 1e-3) / 1e9

    # ---------------- the run verifies itself (every rank; failure aborts the run)
    y_csr_keep = None
    if args.format == "csr":
        parity = check_csr_parity(ctx, op, x, stencil_grid=args.grid if args.workload == "stencil27" else None)
        if primary_default and not args.no_secondary:
            op.step(stream)
            op.finish(stream)
            ctx.barrier()
            y_csr_keep = op.last_y().clone()
    else:
        # TJDS as the primary: verified against a CSR operator of the same matrix built beside it
        ref_op, _ = make_csr_op(ctx, gen, args, eng.CSR_AUTO, "none" if world == 1 else "nccl")
        ref_op.set_x(x, stream)
        ref_op.step(stream)
        ref_op.finish(stream)
        ctx.barrier()
        parity = check_tjds_parity(ctx, op, ref_op.last_y(), tj_map.get(args.variant, eng.TJDS_ATOMIC) != eng.TJDS_ATOMIC)
        ref_op.free()
        del ref_op

    # ---------------- roofline of the dominant kernel (this rank's SpMV launch)
    local_bytes = op.local_bytes_per_mult
    kern_ms = t["kern_ms_local"]
    achieved = local_bytes / (kern_ms * 1e-3) / 1e9
    traffic = (op.measured_traffic_bytes() if (world == 1 and args.workload == "stencil27" and args.grid == 369) else None)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak,
                "traffic": traffic,
                "traffic_source": ("profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per launch from the "
                                   "committed ncu --set full capture of this configuration (not measured in this run)"
                                   if traffic is not None else None),
                "kernel": op.kernel_name, "kernel_ms": kern_ms, "kernel_ms_min": t["kern_ms_min"],
                "kernel_ms_median": t["kern_ms_median"],
                "kernel_ms_note": "CUDA events around the SpMV launch only, opened after any wait for an earlier step's exchange",
                "algorithmic_bytes_per_launch": local_bytes, "peak_source": ctx.peak_src,
                "frac_of_nominal_8000": achieved / 8000.0}
    step_breakdown = None
    if world > 1:
        step_breakdown = {"step_ms": ms_per_step, "spmv_ms": t["kern_ms_max"],
                          "spmv_alone_ms": tuning["spmv_alone_ms"] if tuning else None,
                          "exchange_alone_ms": tuning["exchange_alone_ms"] if tuning else None,
                          "note": "spmv_ms: SpMV launch inside the pipelined steps (max over ranks); *_alone_ms: the same SpMV / "
                                  "the exchange of one step run by themselves during warm-up"}

    # ---------------- end to end: host x -> device -> SpMV (-> exchange) -> host y, every step
    e2e = None
    if not args.no_e2e:
        e2e_steps = max(3, min(args.steps, 20))
        hx = torch.empty(N, dtype=torch.float64).pin_memory()
        hx.copy_(x)
        hy = torch.empty(op.local_rows_out, dtype=torch.float64).pin_memory()
        for _ in range(2):
            op.e2e_step(hx, hy, stream)
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            op.e2e_step(hx, hy, stream)
        ctx.barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        e2e_ms = ctx.max_over_ranks([e2e_ms])[0] / e2e_steps
        # whole-job bytes per step: x crosses PCIe once (each rank uploads its slice), y comes back once
        e2e = {"value": nbytes / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(N * 8),
               "d2h_bytes_per_step": int(M * 8), "ms_per_step": e2e_ms, "steps": e2e_steps, "api": op.e2e_api,
               "host_numa_node_of_rank0": numa_node}
        if args.format == "csr":
            # the rows that came back over PCIe against the device-resident result of the same x
            op.step(stream)
            op.finish(stream)
            ctx.barrier()
            dev = op.last_y()[op.r0:op.r1]
            e2e["host_rows_bit_identical_to_device"] = bool(torch.equal(hy.to("cuda"), dev))
            if not e2e["host_rows_bit_identical_to_device"]:
                raise SystemExit("PARITY FAILED: e2e rows differ from the device-resident step on rank %d" % rank)
        del hx, hy

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, {"rows": M, "cols": N, "nnz": nnz_total, "bytes_per_spmv": nbytes,
                                             "partition": op.partition_desc, "kernel_variant": op.variant_name,
                                             "build_s": build_s, "multiply_plan": op.plan_desc()}),
            "gflops": 2 * nnz_total / (ms_per_step * 1e-3) / 1e9,
            "pct_of_hbm_peak_8000": 100.0 * value / 8000.0 / world,
            "roofline": roofline, "clocks": t["clocks"], "gpu_launches": t["launches"],
            "parity_checked": True, "parity_max_rel": parity["parity_max_rel"], "parity": parity,
        }
        if step_breakdown:
            line["step_breakdown"] = step_breakdown
        if tuning:
            line["exchange_tuning"] = tuning
        if e2e:
            line["e2e"] = e2e
    # the operator is released before the secondary configurations and the CPU leg
    op.free()
    del op
    torch.cuda.empty_cache()
    if primary_default and not args.no_secondary:
        sec = run_secondary(ctx, args, gen, y_csr_keep, x)
        if rank == 0:
            line["secondary"] = sec
    if hasattr(gen, "release"):
        gen.release()
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            res = cpu_reference_run(args, args.cpu_iters)
            line["cpu_baseline"] = {"value": res["value"], "unit": UNIT, "cores": 1, "kind": res["kind"],
                                    "sample": res["sample"], "gflops": res["gflops"]}
            if "all_cores" in res:
                line["cpu_baseline"]["all_cores"] = res["all_cores"]
        print_json(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    # stdout carries exactly ONE JSON line: libraries that chat on fd 1 (NCCL prints its version there) are
    # sent to stderr, and the line is written to the real stdout at the end
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global print_json

    def print_json(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
