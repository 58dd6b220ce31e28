#!/usr/bin/env python3
"""A/B of the popularity relabelling (relabel.cu) on an R-MAT matrix (GPU box):
    python tools/sweep_rmat.py --scale 26 [--steps 10]
Builds the same CSR twice (SMVP_CSR_RELABEL=0 / 1), times the merge-path and the vector kernel on both with x declared once (smvp_csr_set_x_device), times the x permutation itself, and checks that the relabelled
y is bit-identical to the plain y."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import smvp_toolkit_b200 as eng  # noqa: E402
from smvp_toolkit_b200 import dist as sdist  # noqa: E402


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=int, default=26)
    ap.add_argument("--edge-factor", type=int, default=16)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--modes", default="0,1")
    ap.add_argument("--no-vector", action="store_true")
    args = ap.parse_args()
    src = sdist.RmatSource(eng, args.scale, args.edge_factor << args.scale)
    M = N = src.rows
    r, c, v = src.row_block(0, M)
    nnz = r.n
    nbytes = 12 * nnz + 4 * (M + 1) + 8 * N + 8 * M
    print("matrix: %s rows=%d nnz=%d bytes/spmv=%d" % (src.desc, M, nnz, nbytes), flush=True)
    x = torch.empty(N, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, N, 999)
    y = torch.empty(M, dtype=torch.float64, device="cuda")
    y_plain = None
    for mode in args.modes.split(","):
        os.environ["SMVP_CSR_RELABEL"] = mode
        A = eng.CsrMatrix.build_device(r, c, v, M, N, nnz)
        t_plan = timeit(lambda: A.set_x_device(x), 1)  # first call decides and builds the plan; then 3 warm + 1
        print("relabel=%s state=%d   set_x %.3f ms" % (mode, A.x_relabel, t_plan), flush=True)
        y.fill_(float("nan"))
        ms = timeit(lambda: A.mult_device(None, y, eng.CSR_MERGE), args.steps)
        tag = ""
        if mode == "0":
            y_plain = y.clone()
        elif y_plain is not None:
            tag = "bit-identical" if torch.equal(y, y_plain) else "DIFFERS from plain"
        print("  merge      : %8.3f ms  %8.1f GB/s  %s" % (ms, nbytes / ms / 1e6, tag), flush=True)
        if not args.no_vector:
            ms = timeit(lambda: A.mult_device(None, y, eng.CSR_VECTOR), args.steps)
            print("  vector     : %8.3f ms  %8.1f GB/s" % (ms, nbytes / ms / 1e6), flush=True)
        ms = timeit(lambda: A.mult_device(x, y, eng.CSR_MERGE), args.steps)
        print("  merge, x passed every call (permutation inside): %8.3f ms" % ms, flush=True)
        A.free()


if __name__ == "__main__":
    main()
