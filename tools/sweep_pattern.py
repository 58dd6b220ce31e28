#!/usr/bin/env python3
"""Tuning sweep (GPU box) of the row-pattern kernel (csr_pattern_kernel, SMVP_PATTERN_CFG) on the 27-point stencil.
    python tools/sweep_pattern.py [--grid 369] [--cfgs 0-7] [--steps 20] [--rounds 2]
Times, in one process and alternating, every pattern configuration and the merge-path kernel with the plan off
(SMVP_CSR_PATTERN=0, a second handle), with CUDA events over `steps` back-to-back passes.  Per configuration: ms, the
bytes the plan actually streams per pass over the kernel time, and that rate as a share of the device-to-device copy
rate measured in the same call (a 4 GiB torch copy: read + written bytes over its time).  Checks y: bit-identical
between configurations, within 1e-12 of the merge kernel.  The matrix (17 GB in CSR) is larger than L2 by two orders
of magnitude, so no flush is needed between passes."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import smvp_toolkit_b200 as eng  # noqa: E402


def parse_list(s):
    out = []
    for part in s.split(","):
        a, _, b = part.partition("-")
        out += list(range(int(a), int(b or a) + 1))
    return out


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


def copy_peak_gbs(steps):
    n = (4 << 30) // 8
    a = torch.empty(n, dtype=torch.float64, device="cuda").fill_(1.0)
    b = torch.empty_like(a)
    ms = timeit(lambda: b.copy_(a), steps)
    del a, b
    return 2 * n * 8 / ms / 1e6


def build(nx, pattern, x):
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH, seed=1)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    os.environ["SMVP_CSR_PATTERN"] = "1" if pattern else "0"
    A.set_x_device(x)  # the plan is decided here
    torch.cuda.synchronize()
    os.environ.pop("SMVP_CSR_PATTERN")
    return A


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=369)
    ap.add_argument("--cfgs", default="0-7")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks.mem",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("gpu: %s" % smi, flush=True)
    nx = args.grid
    m = nx ** 3
    x = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, m, 999)
    A = build(nx, True, x)
    B = build(nx, False, x)
    y = torch.empty(m, dtype=torch.float64, device="cuda")
    y_ref = torch.empty_like(y)
    B.mult_device(x, y_ref, eng.CSR_MERGE)
    A.mult_device(x, y, eng.CSR_MERGE)
    torch.cuda.synchronize()
    P = A.row_patterns
    assert P > 0 and B.row_patterns == -1, (P, B.row_patterns)
    nnz = A.nnz
    algo = 12 * nnz + 4 * (m + 1) + 16 * m
    tiles = (m + 31) // 32
    streamed = 8 * nnz + m + 16 * m + 8 * tiles  # val, pat_id, x, y, two row_ptr entries per 32-row tile
    print("matrix: stencil27 %d^3 rows=%d nnz=%d patterns=%d | algorithmic bytes %.3f GB, streamed by the plan %.3f GB"
          % (nx, m, nnz, P, algo / 1e9, streamed / 1e9), flush=True)
    y0 = None
    for rnd in range(args.rounds):
        peak = copy_peak_gbs(args.steps)
        print("round %d: copy peak %.1f GB/s (4 GiB device-to-device, read + write)" % (rnd, peak), flush=True)
        ms = timeit(lambda: B.mult_device(x, y_ref, eng.CSR_MERGE), args.steps)
        print("  merge (plan off)    : %7.3f ms  %7.1f GB/s algorithmic" % (ms, algo / ms / 1e6), flush=True)
        for cfg in parse_list(args.cfgs):
            os.environ["SMVP_PATTERN_CFG"] = str(cfg)
            y.fill_(float("nan"))
            ms = timeit(lambda: A.mult_device(x, y, eng.CSR_MERGE), args.steps)
            y0 = y.clone() if y0 is None else y0
            same = bool(torch.equal(y, y0))
            err = float(torch.linalg.norm(y - y_ref) / torch.linalg.norm(y_ref))
            rate = streamed / ms / 1e6
            print("  pattern cfg %d       : %7.3f ms  %7.1f GB/s algorithmic  %7.1f GB/s streamed = %5.1f %% of copy peak"
                  "  bit-identical %s  rel_l2_vs_merge %.1e" % (cfg, ms, algo / ms / 1e6, rate, 100 * rate / peak, same, err),
                  flush=True)
        os.environ.pop("SMVP_PATTERN_CFG")
    A.free()
    B.free()


if __name__ == "__main__":
    main()
