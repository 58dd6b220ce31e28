#!/usr/bin/env python3
"""Tuning sweep (GPU box): TJDS multiply on the 27-point stencil, straight walk vs skewed walk (SMVP_TJDS_SKEW=0/1),
atomic and deterministic.  Checks on the way: atomic within 1e-12 of merge-path CSR, deterministic bit-identical
between the two walks (the integer accumulation is exact, so the walk must not matter) and run to run.
    python tools/sweep_tjds.py --grid 369 [--steps 10]"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import smvp_toolkit_b200 as eng  # noqa: E402


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
    ap.add_argument("--grid", type=int, default=369)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--modes", default="0,1,auto")
    args = ap.parse_args()
    g = args.grid
    m = n = g ** 3
    r, c, v = eng.synth_stencil27(g, g, g, value_mode=eng.VAL_HASH, seed=7)
    nnz = r.n
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, n, 999)
    A = eng.CsrMatrix.build_device(r, c, v, m, n, nnz)
    y_csr = torch.empty(m, dtype=torch.float64, device="cuda")
    A.mult_device(x, y_csr, eng.CSR_MERGE)
    torch.cuda.synchronize()
    A.free()
    y = torch.empty(m, dtype=torch.float64, device="cuda")
    det_keep = {}
    for mode in args.modes.split(","):
        if mode == "auto":
            os.environ.pop("SMVP_TJDS_SKEW", None)
        else:
            os.environ["SMVP_TJDS_SKEW"] = mode
        T = eng.TjdsMatrix.build_device(r, c, v, m, n, nnz)
        nbytes = T.bytes_per_mult
        T.set_x_device(x)
        for name, variant in (("atomic", eng.TJDS_ATOMIC), ("deterministic", eng.TJDS_DETERMINISTIC),
                              ("det. fast", eng.TJDS_DETERMINISTIC_FAST)):
            y.fill_(float("nan"))
            ms = timeit(lambda: T.mult_device(y, variant), args.steps)
            err = float(torch.linalg.norm(y - y_csr) / torch.linalg.norm(y_csr))
            tag = "rel_l2 vs CSR %.2e" % err
            if variant != eng.TJDS_ATOMIC:
                y2 = torch.empty_like(y)
                T.mult_device(y2, variant)
                tag += ", run-to-run " + ("bit-identical" if torch.equal(y, y2) else "DIFFERS")
                if variant not in det_keep:
                    det_keep[variant] = y.clone()
                else:
                    tag += ", vs first walk " + ("bit-identical" if torch.equal(y, det_keep[variant]) else "DIFFERS")
            print("skew=%-4s plan=%s ndiag=%d  %-13s: %8.3f ms  %8.1f GB/s  %s" %
                  (mode, T.plan(), T.ndiag, name, ms, nbytes / ms / 1e6, tag), flush=True)
        T.free()


if __name__ == "__main__":
    main()
