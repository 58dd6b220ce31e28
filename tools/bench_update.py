#!/usr/bin/env python3
"""Cost of an in-place value update (smvp_*_update_values_device) against a rebuild, on the benchmark's matrices:
    python tools/bench_update.py [--grid 369] [--scale 26] [--edge-factor 16] [--rounds 3] [--workloads stencil,rmat]
Two costs, alternated round by round in one process:
    rebuild   build from the device COO + the first pass (every plan the pass needs decided), freed afterwards
    update    the same handle, kept across rounds, given new values on
                all       every entry, in build order
                shuffled  every entry, in a random order (a permutation drawn once, on the device)
                diagonal  the stored diagonal only (A - sigma I)
Workloads:
    stencil  27-point stencil grid^3, CSR with the row-pattern plan.  The values alternate between the stencil's {26, -1}
             (fp16 copy) and hashed values (fp64): every "all" / "shuffled" update changes the width (2 -> 8, 8 -> 2); the
             diagonal update sets 25.5 and back to 26 (the width stays 2, the copy is narrowed in place)
    rmat     R-MAT 2^scale x 2^scale with edge_factor * 2^scale generated edges: CSR (its AUTO plan relabels the columns),
             then TJDS -- the same updates before any deterministic pass (atomic: nothing value-dependent to decide) and
             after one (deterministic: the row bounds are decided again).  Values alternate between v and 1.5 v.
Milliseconds are host wall clock around the synchronous call (a device synchronise before it).  GB/s are over the update's
own bytes: 16 B read (row, col, value) and 8 B written per list entry; the pattern plan adds 8 nnz read and value_bytes nnz
written (a narrow copy only); the TJDS bound pass reads row_ind and val (12 nnz).  The binary searches' reads of the
structure are not counted.  After the timed rounds the script checks that each updated handle's y is bit-identical to a
fresh build's (TJDS atomic: within 1e-12).  The card's name and power limit are printed beside the numbers."""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import smvp_toolkit_b200 as eng  # noqa: E402

GPU = ""


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def t(a):
    return torch.as_tensor(a, device="cuda")


class Lists:
    """the update lists of one matrix: build order, one shuffled order, the stored diagonal; two value sets each"""

    def __init__(self, r, c, v0, v1):
        self.n = r.n
        self.r, self.c = t(r), t(c)
        self.v = [t(v0), v1]
        perm = torch.randperm(self.n, device="cuda")
        self.rs, self.cs = self.r[perm], self.c[perm]
        self.vs = [self.v[0][perm], self.v[1][perm]]
        del perm
        d = (self.r == self.c).nonzero().squeeze(1)
        self.rd, self.cd = self.r[d], self.c[d]
        self.vd = [self.v[0][d], self.v[0][d] - 0.5]
        torch.cuda.empty_cache()

    def apply(self, A, kind, k):
        if kind == "all":
            A.update_values_device(self.r, self.c, self.v[k], self.n)
        elif kind == "shuffled":
            A.update_values_device(self.rs, self.cs, self.vs[k], self.n)
        else:
            A.update_values_device(self.rd, self.cd, self.vd[k], len(self.rd))

    def count(self, kind):
        return len(self.rd) if kind == "diagonal" else self.n


def report(name, times, nbytes):
    for kind, ts in times.items():
        extra = "" if kind == "rebuild" else "   %7.1f GB/s at min" % (nbytes[kind] / min(ts) / 1e6)
        print("  %-34s %-20s " % (name, kind) + " ".join("%9.2f" % x for x in ts) + "   min %9.2f ms%s" % (min(ts), extra), flush=True)
    reb = min(times["rebuild"])
    for kind in times:
        if kind != "rebuild":
            print("  %-34s %-20s rebuild / update = %.1fx   [%s]" % (name, kind, reb / min(times[kind]), GPU), flush=True)


def same_bits(a, b):
    return torch.equal(a.view(torch.int64), b.view(torch.int64))


def stencil(args):
    nx = args.grid
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    r2, c2, vh = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH)
    r2.free()
    c2.free()
    L = Lists(r, c, v, t(vh).clone())
    vh.free()
    x = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, m, 7)
    y = torch.empty_like(x)

    def rebuild(vals):
        A = eng.CsrMatrix.build_device(r, c, vals, m, m, L.n)
        A.mult_device(x, y, eng.CSR_MERGE)
        return A

    H = rebuild(v)
    assert H.row_patterns == 27 and H.value_bytes == 2
    nnz = H.nnz
    labels = {("all", 1): "all fp16->fp64", ("all", 0): "all fp64->fp16", ("shuffled", 1): "shuffled fp16->fp64",
              ("shuffled", 0): "shuffled fp64->fp16", ("diagonal", 1): "diagonal 25.5", ("diagonal", 0): "diagonal 26"}
    times = {k: [] for k in ("rebuild",) + tuple(labels.values())}
    for rnd in range(args.rounds):
        F = [None]
        times["rebuild"].append(wall(lambda: F.__setitem__(0, rebuild(v))))
        F[0].free()
        torch.cuda.empty_cache()
        for kind in ("all", "shuffled", "diagonal"):
            for k in (1, 0):  # hashed values (fp64) then back to the stencil's (fp16); diagonal: 25.5 then 26
                times[labels[kind, k]].append(wall(lambda: L.apply(H, kind, k)))
                assert H.value_bytes == (8 if k == 1 and kind != "diagonal" else 2), (kind, k, H.value_bytes)
    # the pattern plan reads val once (8 nnz) and writes the narrow copy when the new width is 2 (2 nnz)
    nbytes = {lab: 24 * L.count(kind) + 8 * nnz + (2 * nnz if kind == "diagonal" or k == 0 else 0) for (kind, k), lab in labels.items()}
    report("stencil %d^3 CSR row-pattern" % nx, times, nbytes)
    # the updated handle against fresh builds, in both value states
    for vals, k, name in ((v, 0, "stencil values"), (L.v[1], 1, "hashed values")):
        L.apply(H, "shuffled", k)
        F = rebuild(vals)
        y0, y1 = torch.empty_like(y), torch.empty_like(y)
        H.mult_device(x, y0, eng.CSR_MERGE)
        F.mult_device(x, y1, eng.CSR_MERGE)
        torch.cuda.synchronize()
        assert same_bits(y0, y1) and H.value_bytes == F.value_bytes, name
        print("  check: updated handle == fresh build, y bit-identical (%s, value_bytes %d)" % (name, H.value_bytes), flush=True)
        F.free()
    H.free()
    for a in (r, c, v):
        a.free()
    del L
    torch.cuda.empty_cache()


def rmat(args):
    n = 1 << args.scale
    r, c, v = eng.synth_rmat(args.scale, args.edge_factor << args.scale, value_mode=eng.VAL_HASH, seed=42)
    L = Lists(r, c, v, t(v) * 1.5)
    x = torch.empty(n, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, n, 7)
    y = torch.empty_like(x)

    def csr(vals):
        A = eng.CsrMatrix.build_device(r, c, vals, n, n, L.n)
        A.set_x_device(x)
        A.mult_device(None, y, eng.CSR_AUTO)
        return A

    def tjds(vals, variant):
        A = eng.TjdsMatrix.build_device(r, c, vals, n, n, L.n)
        A.set_x_device(x)
        A.mult_device(y, variant)
        return A

    kinds = ("all", "shuffled", "diagonal")
    runs = [("R-MAT %d CSR" % args.scale, lambda vals: csr(vals), None),
            ("R-MAT %d TJDS atomic" % args.scale, lambda vals: tjds(vals, eng.TJDS_ATOMIC), eng.TJDS_ATOMIC),
            ("R-MAT %d TJDS deterministic" % args.scale, lambda vals: tjds(vals, eng.TJDS_DETERMINISTIC), eng.TJDS_DETERMINISTIC)]
    H = None
    for name, make, variant in runs:
        if H is None or variant is None:
            H = make(L.v[0])  # the TJDS handle is kept from the atomic run into the deterministic one
        elif variant == eng.TJDS_DETERMINISTIC:
            H.mult_device(y, variant)  # the deterministic state now exists: updates decide the row bounds again
        nnz = H.nnz
        if variant is None:
            print("  (CSR x_relabel %d, row_patterns %d)" % (H.x_relabel, H.row_patterns), flush=True)
        else:
            print("  (TJDS y_relabel %d, (skewed_walk, det_route) %s)" % (H.y_relabel, H.plan()), flush=True)
        times = {k: [] for k in ("rebuild",) + kinds}
        for rnd in range(args.rounds):
            F = [None]
            times["rebuild"].append(wall(lambda: F.__setitem__(0, make(L.v[0]))))
            F[0].free()
            torch.cuda.empty_cache()
            for kind in kinds:
                for k in (1, 0):
                    times[kind].append(wall(lambda: L.apply(H, kind, k)))
        extra = 12 * nnz if variant == eng.TJDS_DETERMINISTIC else 0
        report(name, times, {kind: 24 * L.count(kind) + extra for kind in kinds})
        # the updated handle (new values on every entry) against a fresh build
        L.apply(H, "shuffled", 1)
        F = make(L.v[1])
        y0, y1 = torch.empty_like(y), torch.empty_like(y)
        if variant is None:
            H.mult_device(x, y0, eng.CSR_AUTO)
            F.mult_device(x, y1, eng.CSR_AUTO)
        else:
            H.mult_device(y0, variant)
            F.mult_device(y1, variant)
        torch.cuda.synchronize()
        if variant == eng.TJDS_ATOMIC:
            err = float(torch.linalg.norm(y0 - y1) / torch.linalg.norm(y1))
            assert err <= 1e-12, err
            print("  check: updated handle == fresh build within %.1e (atomic)" % err, flush=True)
        else:
            assert same_bits(y0, y1), name
            print("  check: updated handle == fresh build, y bit-identical", flush=True)
        F.free()
        L.apply(H, "shuffled", 0)
        if variant is None or variant == eng.TJDS_DETERMINISTIC:
            H.free()
            H = None
        torch.cuda.empty_cache()
    for a in (r, c, v):
        a.free()


def main(argv=None):
    global GPU
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=369)
    ap.add_argument("--scale", type=int, default=26)
    ap.add_argument("--edge-factor", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--workloads", default="stencil,rmat")
    args = ap.parse_args(argv)
    work = args.workloads.split(",")
    if args.rounds < 1 or not work or any(w not in ("stencil", "rmat") for w in work):
        ap.error("--rounds must be at least 1, --workloads a list of stencil and rmat")
    if not torch.cuda.is_available():
        sys.exit("bench_update.py measures on the GPU: no CUDA device")
    GPU = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    print("gpu: %s" % GPU, flush=True)
    print("ms per call, rounds 1..%d (each update kind: two calls per round)" % args.rounds, flush=True)
    if "stencil" in work:
        stencil(args)
    if "rmat" in work:
        rmat(args)
    print("gpu at the end: %s" % subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                                 capture_output=True, text=True).stdout.strip(), flush=True)


if __name__ == "__main__":
    main()
