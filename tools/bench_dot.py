#!/usr/bin/env python3
"""Fused inner product y = alpha * A x + beta * y with w . y in the same pass, against the unfused pair, on the benchmark's
matrices:
    python tools/bench_dot.py [--grid 369] [--scale 26] [--edge-factor 16] [--steps 20] [--rounds 3]
For the 27-point stencil grid^3 (stencil values) and R-MAT 2^scale (edge factor 16, seed 42, hashed values -- bench.py's
defaults) it times, in one process with CUDA events over `steps` back-to-back passes after a warm-up, alternating the
three in `rounds` rounds (alpha = -1, beta = 1, the residual update):
    axpby    the *_axpby call alone
    fused    the *_axpby_dot call (w . y_new into a one-element device tensor)
    unfused  the *_axpby call, then torch.dot(w, y) (w = NULL: torch.dot(y, y))
for CSR AUTO on both matrices (the row-pattern plan on the stencil, merge-path over relabelled columns on R-MAT) and for
TJDS deterministic on the stencil, each with w = x and w = NULL.  It checks inside the run that the fused y equals the
unfused y bit for bit and that the fused dot is within the bound of smvp_cuda.h (k = 1 + d + 49) of torch.dot plus a
generous bound for torch's own order, and prints ms, the bytes of each pass computed from the shapes and bytes over time.
Bytes: the *_axpby pass = plain pass (smvp_*_info_t.bytes_per_mult; the row-pattern plan 8 nnz + 17 rows) + 8 rows for the
read of y; fused = that + 8 rows for w when w != NULL (x is gathered by the pass itself, so most of it should come from L2)
+ 16 bytes per work unit; unfused = axpby + 16 rows (torch.dot reads y and w) or 8 rows (w = NULL).  Every matrix (>= 13 GB)
is far larger than L2, so no flush is needed between passes."""
import argparse
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import smvp_toolkit_b200 as eng  # noqa: E402

ALPHA, BETA = -1.0, 1.0
U = 2.0 ** -53


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


def run(label, rows, axpby_bytes, units, depth, axpby, fused, w, steps, rounds):
    """axpby(y) updates y in place; fused(y, w, d) updates y and stores w . y_new into d[0]."""
    y = torch.empty(rows, dtype=torch.float64, device="cuda")
    y0 = torch.empty_like(y)
    eng.synth_vector(y0, rows, 99)
    d = torch.zeros(1, dtype=torch.float64, device="cuda")
    out = torch.zeros((), dtype=torch.float64, device="cuda")

    def unfused():
        axpby(y)
        torch.dot(y if w is None else w, y, out=out)

    # correctness first, from the same y0
    yf = y0.clone()
    fused(yf, w, d)
    y.copy_(y0)
    unfused()
    torch.cuda.synchronize()
    same_y = bool(torch.equal(yf.view(torch.int64), y.view(torch.int64)))
    ww = y if w is None else w
    s_abs = float(torch.sum(torch.abs(ww * y)))
    k = 1 + depth + 49
    tol = k * U / (1 - k * U) * s_abs + 64 * math.log2(rows) * U * s_abs
    err = abs(float(d[0]) - float(out))
    ok = same_y and err <= tol
    check = "y bit for bit: %s; |dot - torch.dot| %.3e (bound %.3e)" % (same_y, err, tol)
    wb = 0 if w is None else 8 * rows
    ops = [("axpby", lambda: axpby(y), axpby_bytes), ("fused", lambda: fused(y, w, d), axpby_bytes + wb + 16 * units),
           ("unfused", unfused, axpby_bytes + 8 * rows + wb)]
    y.copy_(y0)
    times = {name: [] for name, _, _ in ops}
    for rnd in range(rounds):
        for name, fn, nbytes in ops:
            ms = timeit(fn, steps)
            times[name].append(ms)
            print("  round %d  %-36s %-8s %8.3f ms  %7.3f GB  %7.1f GB/s" % (rnd, label, name, ms, nbytes / 1e9, nbytes / ms / 1e6),
                  flush=True)
    best = {name: min(ts) for name, ts in times.items()}
    for name, _, nbytes in ops:
        ts = times[name]
        print("  summary  %-36s %-8s min %8.3f  max %8.3f ms  %7.1f GB/s at min" % (label, name, min(ts), max(ts), nbytes / min(ts) / 1e6),
              flush=True)
    print("  result   %-36s fused / unfused %.3f, fused - axpby %+.3f ms; %s" % (label, best["fused"] / best["unfused"],
                                                                           best["fused"] - best["axpby"], check), flush=True)
    assert ok, label
    del y, y0, yf
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
    csr_bytes = (8 * A.nnz + 17 * m if A.row_patterns > 0 else A.bytes_per_mult) + 8 * m
    for wname, w in (("w = x", x), ("w = NULL", None)):
        run("stencil CSR AUTO, %s" % wname, m, csr_bytes, -(-m // 32), 5, lambda o: A.mult_device_axpby(ALPHA, x, BETA, o),
            lambda o, ww, d: A.mult_device_axpby_dot(ALPHA, x, BETA, o, ww, d), w, args.steps, args.rounds)
    J.mult_device(out, eng.TJDS_DETERMINISTIC)
    torch.cuda.synchronize()
    print("  TJDS deterministic: y_relabel=%d, det_route=%d" % (J.y_relabel, J.plan()[1]), flush=True)
    for wname, w in (("w = x", x), ("w = NULL", None)):
        run("stencil TJDS deterministic, %s" % wname, m, J.bytes_per_mult + 8 * m, -(-m // 256), 8,
            lambda o: J.mult_device_axpby(ALPHA, BETA, o, eng.TJDS_DETERMINISTIC),
            lambda o, ww, d: J.mult_device_axpby_dot(ALPHA, BETA, o, ww, d, eng.TJDS_DETERMINISTIC), w, args.steps, args.rounds)
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
    units = -(-(n + A.nnz) // 320)  # merge-path tiles, at most (rows + nnz) / (32 * 10)
    for wname, w in (("w = x", x), ("w = NULL", None)):
        run("R-MAT CSR AUTO, %s" % wname, n, A.bytes_per_mult + 8 * n, units, 20, lambda o: A.mult_device_axpby(ALPHA, None, BETA, o),
            lambda o, ww, d: A.mult_device_axpby_dot(ALPHA, None, BETA, o, ww, d), w, args.steps, args.rounds)
    A.free()


if __name__ == "__main__":
    main()
