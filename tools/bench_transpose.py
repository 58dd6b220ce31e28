#!/usr/bin/env python3
"""Transposed product y = A^T x on the benchmark's two matrices (GPU box), in one process:
    python tools/bench_transpose.py [--grid 369] [--scale 26] [--edge-factor 16] [--steps 20] [--rounds 2]
For the 27-point stencil grid^3 (stencil values: 26 on the diagonal, -1 elsewhere, so A is symmetric) and for R-MAT
2^scale (edge factor 16, seed 42, hashed values -- bench.py's defaults) it times, with CUDA events over `steps`
back-to-back passes after a warm-up, alternating in `rounds` rounds:
    CSR  A x      (AUTO)                        CSR  A^T x   (AUTO, on the handle smvp_csr_transpose built)
    TJDS A x      (atomic, x permuted once)     TJDS A^T x   (smvp_tjds_mult_transpose_device)
and reports ms, the algorithmic bytes of a pass and bytes over time.  TJDS A^T x moves 12 nnz + 4 (ndiag+1) for the
matrix, 8 rows for x, 12 cols for y and perm.  Also: the one-off smvp_csr_transpose time (host clock around the
synchronous call), the HBM the transposed handle holds and the scratch the TJDS transposed product adds, and a
profiled pass that splits the TJDS A^T x time into its two kernels (the combine of the long columns runs only when a
column holds more than 32 entries).  Checks, inside the run: stencil x = ones gives 27 - count; stencil random x:
CSR A^T x and TJDS A^T x are bit-identical to CSR A x (A is symmetric and every sum runs in the same order); R-MAT:
CSR A^T x and TJDS A^T x agree within 1e-12.  Every matrix (>= 16 GB) is far larger than L2, so no flush is needed
between passes."""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch  # noqa: E402

import smvp_toolkit_b200 as eng  # noqa: E402
import synth_ref  # noqa: E402


def timeit(fn, steps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def rel_l2(a, b):
    return float(torch.linalg.norm(a - b) / torch.linalg.norm(b))


def tjds_device_bytes(J):
    import ctypes

    info = eng.engine._TjdsInfo()
    assert eng.lib().smvp_tjds_info(J._h, ctypes.byref(info)) == 0
    return info.device_bytes


def kernel_split(fn):
    """Mean device time per pass of the two transposed TJDS kernels (torch.profiler, 5 passes)."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        n = ("tjds_transpose_combine_kernel" if "tjds_transpose_combine_kernel" in ev.key else
             "tjds_transpose_kernel" if "tjds_transpose_kernel" in ev.key else None)
        if n:
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            out[n] = out.get(n, 0.0) + t / 5 / 1e3  # us -> ms per pass
    return out


def run(name, A, J, x, steps, rounds, checks):
    m, n = A.rows, A.cols
    t0 = time.perf_counter()
    T = A.transpose()
    torch.cuda.synchronize()
    t_transpose = (time.perf_counter() - t0) * 1e3
    y = torch.empty(m, dtype=torch.float64, device="cuda")
    yt = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
    yj = torch.empty(m, dtype=torch.float64, device="cuda")
    yjt = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
    J.set_x_device(x)
    tjds_before = tjds_device_bytes(J)
    J.mult_transpose_device(x, yjt)
    torch.cuda.synchronize()
    tjds_scratch = tjds_device_bytes(J) - tjds_before
    ops = [
        ("CSR  A x    (AUTO)", lambda: A.mult_device(x, y), A.bytes_per_mult),
        ("CSR  A^T x  (AUTO, transposed handle)", lambda: T.mult_device(x, yt), T.bytes_per_mult),
        ("TJDS A x    (atomic)", lambda: J.mult_device(yj, eng.TJDS_ATOMIC), J.bytes_per_mult),
        ("TJDS A^T x", lambda: J.mult_transpose_device(x, yjt), 12 * J.nnz + 4 * (J.ndiag + 1) + 8 * J.rows + 12 * J.cols),
    ]
    print("matrix: %s  rows=%d cols=%d nnz=%d ndiag(TJDS)=%d" % (name, m, n, A.nnz, J.ndiag), flush=True)
    print("  smvp_csr_transpose: %.1f ms (one-off, synchronous); A^T handle holds %.3f GB of HBM (A: %.3f GB); "
          "TJDS A^T x scratch: %.3f MB" % (t_transpose, T.device_bytes / 1e9, A.device_bytes / 1e9, tjds_scratch / 1e6), flush=True)
    times = {label: [] for label, _, _ in ops}
    for rnd in range(rounds):
        for label, fn, nbytes in ops:
            ms = timeit(fn, steps)
            times[label].append(ms)
            print("  round %d  %-40s %8.3f ms  %7.3f GB  %7.1f GB/s" % (rnd, label, ms, nbytes / 1e9, nbytes / ms / 1e6), flush=True)
    print("  T.row_patterns=%d  A.row_patterns=%d" % (T.row_patterns, A.row_patterns), flush=True)
    for label, fn, nbytes in ops:
        ts = times[label]
        print("  summary  %-40s min %8.3f  max %8.3f ms  %7.1f GB/s at min" % (label, min(ts), max(ts), nbytes / min(ts) / 1e6), flush=True)
    split = kernel_split(lambda: J.mult_transpose_device(x, yjt))
    print("  TJDS A^T x per kernel (torch.profiler, profiled run): %s" % ", ".join("%s %.3f ms" % kv for kv in sorted(split.items())),
          flush=True)
    checks(A, T, J, x, y, yt, yjt)
    T.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=369)
    ap.add_argument("--scale", type=int, default=26)
    ap.add_argument("--edge-factor", type=int, default=16)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()
    if args.steps < 20 or args.rounds < 1:
        ap.error("--steps must be at least 20 and --rounds at least 1")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("gpu: %s" % smi, flush=True)

    # ---- 27-point stencil
    nx = args.grid
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    J = eng.TjdsMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    x = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, m, 7)

    def stencil_checks(A, T, J, x, y, yt, yjt):
        A.mult_device(x, y)
        T.mult_device(x, yt)
        J.mult_transpose_device(x, yjt)
        torch.cuda.synchronize()
        same_t = bool(torch.equal(yt.view(torch.int64), y.view(torch.int64)))
        same_j = bool(torch.equal(yjt.view(torch.int64), y.view(torch.int64)))
        counts = torch.as_tensor(synth_ref.stencil27_row_counts(nx, nx, nx)).to("cuda").to(torch.float64)
        ones = torch.ones_like(x)
        T.mult_device(ones, yt)
        J.mult_transpose_device(ones, yjt)
        torch.cuda.synchronize()
        closed_t, closed_j = bool(torch.equal(yt, 27 - counts)), bool(torch.equal(yjt, 27 - counts))
        print("  check: random x -- CSR A^T x bit-identical to A x: %s, TJDS A^T x bit-identical to A x: %s; "
              "x = ones -- closed form 27 - count: CSR %s, TJDS %s" % (same_t, same_j, closed_t, closed_j), flush=True)
        assert same_t and same_j and closed_t and closed_j

    run("stencil27 %d^3" % nx, A, J, x, args.steps, args.rounds, stencil_checks)
    A.free()
    J.free()
    del x
    torch.cuda.empty_cache()

    # ---- R-MAT
    n = 1 << args.scale
    r, c, v = eng.synth_rmat(args.scale, args.edge_factor << args.scale, seed=42)
    A = eng.CsrMatrix.build_device(r, c, v, n, n, r.n)
    J = eng.TjdsMatrix.build_device(r, c, v, n, n, r.n)
    for a in (r, c, v):
        a.free()
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, n, 7)

    def rmat_checks(A, T, J, x, y, yt, yjt):
        T.mult_device(x, yt)
        J.mult_transpose_device(x, yjt)
        torch.cuda.synchronize()
        err = rel_l2(yjt, yt)
        finite = bool(torch.isfinite(yjt).all())
        print("  check: CSR A^T x vs TJDS A^T x rel_l2 %.2e (<= 1e-12), all finite %s" % (err, finite), flush=True)
        assert err <= 1e-12 and finite

    run("R-MAT scale %d edge factor %d" % (args.scale, args.edge_factor), A, J, x, args.steps, args.rounds, rmat_checks)
    A.free()
    J.free()


if __name__ == "__main__":
    main()
