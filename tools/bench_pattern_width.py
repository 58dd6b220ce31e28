#!/usr/bin/env python3
"""Row-pattern multiply at each value width the plan can take, on the benchmark's matrix:
    python tools/bench_pattern_width.py [--grid 369] [--steps 50] [--rounds 3] [--widths 2,4,8]
The 27-point stencil grid^3 is built once per width and round, one handle at a time (freed before the next), with values
chosen so that the plan lands on that width (smvp_csr_info_t.value_bytes):
    2  fp16   the stencil values {26, -1} (bench.py's matrix)
    4  fp32   the same values times (1 + 2^-20), formed on the device before the build: 26 (1 + 2^-20) needs 24
              significant bits, more than fp16's 11 and within fp32's 24
    8  fp64   hashed values (VAL_HASH)
For each it prints the milliseconds of one pass (CUDA events over `steps` back-to-back CSR merge passes after a warm-up),
the bytes the plan streams in that time -- value_bytes * nnz + rows (pattern ids) + 8 cols (x) + 8 rows (y) + two
row_ptr entries per 32-row tile -- and those bytes over the time, beside the device-to-device copy rate (4 GiB, read +
write) measured in the same process, the card's name and power limit.  Every matrix (>= 3.5 GB per pass) is far
larger than L2, so no flush is needed between passes.  Each pass is checked against the vector kernel, which reads the
fp64 values: within 1e-12 normwise (it sums in another order; the bit-for-bit checks against the reference loop are in
tests/test_pattern_width.py)."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import smvp_toolkit_b200 as eng  # noqa: E402

NAMES = {2: "fp16", 4: "fp32", 8: "fp64"}


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


def copy_rate(steps):
    """GB/s of a 4 GiB device-to-device copy, bytes read + written."""
    n = 1 << 29
    a = torch.empty(n, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    ms = timeit(lambda: b.copy_(a), steps)
    del a, b
    torch.cuda.empty_cache()
    return 2 * 8 * n / ms / 1e6


def build(nx, width):
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH if width == 8 else eng.VAL_STENCIL)
    if width == 4:
        torch.as_tensor(v, device="cuda").mul_(1.0 + 2.0 ** -20)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    return A


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=369)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--widths", default="2,4,8")
    args = ap.parse_args(argv)
    widths = [int(w) for w in args.widths.split(",")]
    if args.steps < 20 or args.rounds < 1 or any(w not in NAMES for w in widths):
        ap.error("--steps must be at least 20, --rounds at least 1, --widths a list of 2, 4 and 8")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("gpu: %s" % smi, flush=True)
    nx = args.grid
    m = nx ** 3
    x = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, m, 7)
    y = torch.empty_like(x)
    yv = torch.empty_like(x)
    times = {w: [] for w in widths}
    for rnd in range(args.rounds):
        print("round %d: copy rate %.1f GB/s (4 GiB device-to-device, read + write)" % (rnd, copy_rate(args.steps)), flush=True)
        for w in widths:
            A = build(nx, w)
            A.mult_device(x, y, eng.CSR_MERGE)  # decides the plan and its width
            A.mult_device(x, yv, eng.CSR_VECTOR)
            torch.cuda.synchronize()
            assert A.row_patterns == 27 and A.value_bytes == w, (A.row_patterns, A.value_bytes, w)
            err = float(torch.linalg.norm(y - yv) / torch.linalg.norm(yv))
            assert err <= 1e-12, (w, err)
            nnz = A.nnz
            ms = timeit(lambda: A.mult_device(x, y, eng.CSR_MERGE), args.steps)
            times[w].append(ms)
            streamed = w * nnz + m + 8 * m + 8 * m + 8 * -(-m // 32)
            print("  %s  value_bytes %d  %8.3f ms  %7.3f GB streamed  %7.1f GB/s  rel_l2 vs vector %.1e" %
                  (NAMES[w], w, ms, streamed / 1e9, streamed / ms / 1e6, err), flush=True)
            A.free()
            torch.cuda.empty_cache()
    for w in widths:
        ts = times[w]
        print("summary  %s  min %8.3f  max %8.3f ms" % (NAMES[w], min(ts), max(ts)), flush=True)


if __name__ == "__main__":
    main()
