#!/usr/bin/env python3
"""Fused update y = alpha * A x + beta * y against the plain pass and the unfused pair, on the benchmark's matrices:
    python tools/bench_axpby.py [--grid 369] [--scale 26] [--edge-factor 16] [--steps 20] [--rounds 3]
For the 27-point stencil grid^3 (stencil values) and R-MAT 2^scale (edge factor 16, seed 42, hashed values -- bench.py's
defaults) it times, in one process with CUDA events over `steps` back-to-back passes after a warm-up, alternating the
three in `rounds` rounds:
    plain    y = A x                                       (the plain call)
    fused    y = -1 * A x + 1 * y                          (the *_axpby call: the residual b - A x)
    unfused  t = A x, then y.mul_(1).add_(t, alpha=-1)      (a plain pass into a temporary and two torch vector kernels)
for CSR AUTO on both matrices (the row-pattern plan on the stencil, merge-path over relabelled columns on R-MAT) and for
TJDS atomic and deterministic on the stencil.  It prints ms, the bytes of each pass computed from the shapes and bytes
over time, and checks inside the run that the fused result equals the unfused one: bit for bit for CSR and TJDS
deterministic (with alpha = -1 and beta = 1 every rounding of the two agrees), within 1e-12 normwise for TJDS atomic.
Bytes: the plain pass as smvp_*_info_t.bytes_per_mult counts it (the row-pattern plan: 8 nnz + rows + 16 rows, it
streams no column index); fused = plain + 8 rows (the read of y), TJDS atomic in natural order + 16 rows more (its sums
go through a scratch vector); unfused = plain + 24 rows (t read, y read and written; torch's mul_ by 1 is a fourth
pass over y, not counted).  Every matrix (>= 13 GB) is far larger than L2, so no flush is needed between passes."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import smvp_toolkit_b200 as eng  # noqa: E402

ALPHA, BETA = -1.0, 1.0


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


def run(label, rows, plain_bytes, plain, fused, extra_fused_bytes, exact, steps, rounds):
    """plain(out) stores A x into out; fused(y) updates y in place."""
    y = torch.empty(rows, dtype=torch.float64, device="cuda")
    t = torch.empty_like(y)
    y0 = torch.empty_like(y)
    eng.synth_vector(y0, rows, 99)

    def unfused():
        plain(t)
        y.mul_(BETA).add_(t, alpha=ALPHA)

    # correctness first, from the same y0
    yf = y0.clone()
    fused(yf)
    y.copy_(y0)
    unfused()
    torch.cuda.synchronize()
    if exact:
        ok = bool(torch.equal(yf.view(torch.int64), y.view(torch.int64)))
        check = "fused == unfused bit for bit: %s" % ok
    else:
        err = rel_l2(yf, y)
        ok = err <= 1e-12
        check = "fused vs unfused rel_l2 %.2e (<= 1e-12): %s" % (err, ok)
    ops = [("plain", lambda: plain(y), plain_bytes), ("fused", lambda: fused(y), plain_bytes + 8 * rows + extra_fused_bytes),
           ("unfused", unfused, plain_bytes + 24 * rows)]
    y.copy_(y0)
    times = {name: [] for name, _, _ in ops}
    for rnd in range(rounds):
        for name, fn, nbytes in ops:
            ms = timeit(fn, steps)
            times[name].append(ms)
            print("  round %d  %-40s %-8s %8.3f ms  %7.3f GB  %7.1f GB/s" % (rnd, label, name, ms, nbytes / 1e9, nbytes / ms / 1e6),
                  flush=True)
    best = {name: min(ts) for name, ts in times.items()}
    for name, _, nbytes in ops:
        ts = times[name]
        print("  summary  %-40s %-8s min %8.3f  max %8.3f ms  %7.1f GB/s at min" % (label, name, min(ts), max(ts), nbytes / min(ts) / 1e6),
              flush=True)
    print("  result   %-40s fused / unfused %.3f, fused / plain %.3f; %s" % (label, best["fused"] / best["unfused"],
                                                                           best["fused"] / best["plain"], check), flush=True)
    assert ok, label
    del y, t, y0, yf
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=369)
    ap.add_argument("--scale", type=int, default=26)
    ap.add_argument("--edge-factor", type=int, default=16)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if args.steps < 20 or args.rounds < 1:
        ap.error("--steps must be at least 20 and --rounds at least 1")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("gpu: %s" % smi, flush=True)
    print("alpha = %g, beta = %g; steps %d, rounds %d" % (ALPHA, BETA, args.steps, args.rounds), flush=True)

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
    J.set_x_device(x)
    out = torch.empty_like(x)
    A.mult_device(x, out)  # decides the plan
    torch.cuda.synchronize()
    print("matrix: stencil27 %d^3  rows=%d nnz=%d  CSR row_patterns=%d" % (nx, m, A.nnz, A.row_patterns), flush=True)
    csr_bytes = 8 * A.nnz + 17 * m if A.row_patterns > 0 else A.bytes_per_mult
    run("stencil CSR AUTO", m, csr_bytes, lambda o: A.mult_device(x, o),
        lambda o: A.mult_device_axpby(ALPHA, x, BETA, o), 0, True, args.steps, args.rounds)
    for name, variant in (("atomic", eng.TJDS_ATOMIC), ("deterministic", eng.TJDS_DETERMINISTIC)):
        J.mult_device(out, variant)
        torch.cuda.synchronize()
        natural = J.y_relabel != 1
        print("  TJDS %s: y_relabel=%d, det_route=%d" % (name, J.y_relabel, J.plan()[1]), flush=True)
        run("stencil TJDS %s" % name, m, J.bytes_per_mult, lambda o, v=variant: J.mult_device(o, v),
            lambda o, v=variant: J.mult_device_axpby(ALPHA, BETA, o, v),
            16 * m if variant == eng.TJDS_ATOMIC and natural else 0, variant != eng.TJDS_ATOMIC, args.steps, args.rounds)
    A.free()
    J.free()
    del x, out
    torch.cuda.empty_cache()

    # ---- R-MAT
    n = 1 << args.scale
    r, c, v = eng.synth_rmat(args.scale, args.edge_factor << args.scale, seed=42)
    A = eng.CsrMatrix.build_device(r, c, v, n, n, r.n)
    for a in (r, c, v):
        a.free()
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, n, 7)
    out = torch.empty_like(x)
    A.mult_device(x, out)
    torch.cuda.synchronize()
    print("matrix: R-MAT scale %d edge factor %d  rows=%d nnz=%d  CSR x_relabel=%d" % (args.scale, args.edge_factor, n, A.nnz,
                                                                                      A.x_relabel), flush=True)
    # a relabelled pass given d_x permutes x first: declare x once, as a solver with a fixed x would
    A.set_x_device(x)
    run("R-MAT CSR AUTO", n, A.bytes_per_mult, lambda o: A.mult_device(None, o),
        lambda o: A.mult_device_axpby(ALPHA, None, BETA, o), 0, True, args.steps, args.rounds)
    A.free()


if __name__ == "__main__":
    main()
