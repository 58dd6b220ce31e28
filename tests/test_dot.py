"""Fused inner product in the multiply (smvp_csr_mult_device_axpby_dot, smvp_tjds_mult_device_axpby_dot,
smvp_tjds_mult_transpose_device_axpby_dot).  The contract (include/smvp_cuda.h): y is bit for bit what the matching *_axpby
call stores; *d_dot is the sum of fl(w[r] * y_new[r]) in a fixed order -- one partial per work unit of the plan, then a
tree that depends on the number of partials only -- within gamma_k * sum |w_r y_r| of the exact sum, and bit-identical run
to run wherever y is.  The exact sum here is math.fsum over each product and its exact error (Dekker's two-product)."""
import ctypes
import math
import os
import re
import subprocess

import numpy as np
import pytest

import synth_ref
import util
from oracle import oracle

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(REPO, "smvp-toolkit_b200", "lib", "libsmvp_cuda.so")
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"
U = 2.0 ** -53

PAIRS = [(1.0, 0.0), (-1.0, 1.0), (2.5, -0.75)]
# unit depth d of each plan (smvp_cuda.h); every matrix here has fewer than 2^21 partials, so k = 1 + d + 48 + 1
DEPTH = {"pattern": 5, "merge": 20, "vector": 8, "tjds": 8}


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def same(got, want):
    nan = np.isnan(want)
    return np.array_equal(np.isnan(got), nan) and np.array_equal(bits(got[~nan]), bits(want[~nan]))


def _band(m, offsets, rng):
    r = np.arange(m)
    rows = np.concatenate([r[(r + d >= 0) & (r + d < m)] for d in offsets])
    cols = np.concatenate([r[(r + d >= 0) & (r + d < m)] + d for d in offsets])
    return oracle.make_coo(rows, cols, rng.uniform(-1, 1, len(rows)))


def _stencil(nx, rng):
    coo = synth_ref.stencil27(nx, nx, nx)
    coo["val"] = rng.uniform(-1, 1, len(coo))
    return coo


def _cases():
    """(name, m, n, coo): golden samples, rectangular and degenerate shapes, power-law, banded and stencil matrices."""
    for name in util.SAMPLES:
        m, n, coo = util.load_sample(name)
        yield name, m, n, coo
    rng = np.random.default_rng(21)
    yield "random 700x1900", 700, 1900, util.random_coo(rng, 700, 1900, 20000)
    yield "random 2500x300", 2500, 300, util.random_coo(rng, 2500, 300, 30000)
    coo = util.random_coo(rng, 400, 500, 3000)
    keep = (coo["row"] % 7 != 0) & (coo["col"] % 5 != 0)  # empty rows and empty columns
    yield "empty rows and columns", 400, 500, coo[keep]
    yield "1x1", 1, 1, oracle.make_coo(np.array([0]), np.array([0]), np.array([-2.5]))
    yield "nnz 0", 30, 40, oracle.make_coo(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0))
    yield "rmat 16", 1 << 16, 1 << 16, synth_ref.rmat(16, 16 << 16)
    yield "band 7", 3000, 3000, _band(3000, (-300, -2, -1, 0, 1, 2, 300), rng)
    yield "stencil 20^3", 20 ** 3, 20 ** 3, _stencil(20, rng)


CASES = list(_cases())
IDS = [c[0] for c in CASES]


@pytest.fixture(scope="module")
def eng():
    import smvp_toolkit_b200 as e

    if not os.path.exists(e.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return e


# ---------------------------------------------------------------------------- numpy restatements
def exact_dot(w, y):
    """Correctly rounded sum of w * y: each product split into fl(w y) and its exact error (Dekker, no FMA)."""
    w, y = np.asarray(w, np.float64), np.asarray(y, np.float64)
    p = w * y
    sp = 134217729.0  # 2^27 + 1

    def split(a):
        c = sp * a
        hi = c - (c - a)
        return hi, a - hi

    wh, wl = split(w)
    yh, yl = split(y)
    e = ((wh * yh - p) + wh * yl + wl * yh) + wl * yl
    return math.fsum(np.concatenate([p, e]).tolist())


def bound(w, y, d):
    k = 1 + d + 49
    return k * U / (1 - k * U) * float(np.sum(np.abs(w * y))) + abs(exact_dot(w, y)) * U


def tree(a):
    """Pairwise tree along the last axis (a power of two long): what the lane / thread butterflies compute."""
    while a.shape[-1] > 1:
        a = a[..., 0::2] + a[..., 1::2]
    return a[..., 0]


def unit_partials(terms, rows_per_unit):
    n = len(terms)
    units = -(-n // rows_per_unit)
    a = np.zeros(units * rows_per_unit)
    a[:n] = terms
    return tree(a.reshape(units, rows_per_unit))


def reduce_partials(part):
    """dot_reduce_kernel (dot.cu): CTAs of 8192 partials, thread t adds partials t, t + 256, ... from +0.0, pairwise tree
    over the 256 threads; then the CTA sums the same way in one CTA."""
    p = len(part)
    g = max(1, -(-p // 8192))
    a = np.zeros(g * 8192)
    a[:p] = part
    a = a.reshape(g, 32, 256)
    s = np.zeros((g, 256))
    for i in range(32):
        s = s + a[:, i, :]
    cta = tree(s)
    h = -(-g // 256)
    b = np.zeros(h * 256)
    b[:g] = cta
    b = b.reshape(h, 256)
    s2 = np.zeros(256)
    for i in range(h):
        s2 = s2 + b[i]
    return tree(s2)


# ---------------------------------------------------------------------------- CPU
def test_null_handle_and_null_dot_are_rejected(eng):
    L = eng.lib()
    y = np.zeros(4)
    p = eng.engine._ptr(y)
    assert L.smvp_csr_mult_device_axpby_dot(None, 1.0, p, 0.0, p, None, p, eng.CSR_AUTO, None) == eng.E_ARG
    assert L.smvp_tjds_mult_device_axpby_dot(None, 1.0, 0.0, p, None, p, eng.TJDS_ATOMIC, 0, None) == eng.E_ARG
    assert L.smvp_tjds_mult_transpose_device_axpby_dot(None, 1.0, p, 0.0, p, None, p, None) == eng.E_ARG


def test_dot_mode_kernels_are_in_the_library_spill_free():
    """Every Dot store-mode instantiation and the reduction exist with no stack frame, and each kernel family that stores
    y is instantiated with exactly its store modes: a dot pass always runs the epilogue, never the fan-out."""
    if not os.path.exists(LIB) or not os.path.exists(CUOBJDUMP):
        pytest.skip("library or cuobjdump not available")
    res = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = re.findall(r"Function (\S+):\s*\n\s*REG:\d+ STACK:(\d+)", res)
    D = util.ystore("Dot")
    wanted = {
        "pattern": (r"csr_pattern_kernelIdLi4ELi1ELi1ELi14ELi7E" + D, 1),
        "merge, stencil configuration": (r"csr_merge_warp_kernelILi4ELi14ELi8ELb[01]ELb1E" + D, 2),
        "merge, skewed configuration": (r"csr_merge_warp_kernelILi2ELi10ELi14ELb[01]ELb0E" + D, 2),
        "fix-up": (r"merge_fixup_kernelI" + D, 1),
        "vector": (r"csr_vector_kernelILi\d+E" + D, 5),
        "det-finalize": (r"tjds_det_finalize_kernelI" + D, 1),
        "unrank": (r"tjds_unrank_y_kernelI" + D, 1),
        "transpose": (r"tjds_transpose_kernelI" + D, 1),
        "combine": (r"tjds_transpose_combine_kernelI" + D, 1),
        "empty transpose": (r"tjds_axpby_empty_kernelI" + D, 1),
        "reduction": (r"dot_reduce_kernel", 1),
    }
    for what, (pat, count) in wanted.items():
        hits = [(name, stack) for name, stack in found if re.search(pat, name)]
        assert len(hits) == count, (what, hits)
        assert all(stack == "0" for _, stack in hits), (what, hits)
    csr, tjds = {"Plain", "Fanout", "Axpby", "Dot"}, {"Plain", "Axpby", "Dot"}
    assert util.store_modes(res) == {
        "csr_vector_kernel": csr, "csr_merge_warp_kernel": csr, "merge_fixup_kernel": csr, "csr_pattern_kernel": csr,
        "tjds_det_finalize_kernel": tjds, "tjds_unrank_y_kernel": tjds, "tjds_transpose_kernel": tjds,
        "tjds_transpose_combine_kernel": tjds, "tjds_axpby_empty_kernel": {"Axpby", "Dot"},
    }


# ---------------------------------------------------------------------------- GPU helpers
def _cuda(a):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a, np.float64), device="cuda")


def _dot_buf(nan=True):
    import torch

    return torch.full((1,), float("nan") if nan else 0.0, dtype=torch.float64, device="cuda")


def _y0(rng, n, beta):
    return np.full(n, np.nan) if beta == 0.0 else rng.uniform(-2, 2, n)


def _csr_plan(eng, A, variant):
    v = A.auto_variant if variant == eng.CSR_AUTO else variant
    if v == eng.CSR_VECTOR:
        return "vector"
    return "pattern" if A.row_patterns > 0 else "merge"


def _csr_run(A, alpha, dx, beta, y0, w, variant, stream=None):
    """(y after the dot call, dot)"""
    dy = _cuda(y0)
    dd = _dot_buf()
    A.mult_device_axpby_dot(alpha, dx, beta, dy, None if w is None else w, dd, variant, stream)
    return dy.cpu().numpy(), dd.cpu().numpy()[0]


def _ws(rng, x, m):
    """w = NULL, w = x (square matrices: CG's p^T A p), an unrelated w"""
    out = [("null", None)]
    if len(x) == m:
        out.append(("x", _cuda(x)))
    out.append(("other", _cuda(rng.uniform(-3, 3, m))))
    return out


def _check_dot(got, w_host, y, d, what):
    w = y if w_host is None else w_host
    fin = np.isfinite(w * y).all()
    if not fin:
        return
    ex = exact_dot(w, y)
    assert abs(got - ex) <= bound(w, y, d), (what, got, ex)


def _transpose_plan(J):
    """(d, units) of the transposed dot pass as smvp_cuda.h states them: d = 9 + ceil((cols - nslots) / (256 * gather
    CTAs)) (8 for a handle without entries), units = gather CTAs + combine CTAs.  The gather's CTAs are the handle's
    segment table (tjds_plan): ceil((L_g + extra) / 256) per segment of 32 diagonals, L_g the length of its first
    diagonal, extra = 31 on the skewed walk."""
    _, sp, _, _ = J.export()
    if J.ndiag == 0:
        return 8, -(-J.cols // 256)
    extra = 31 if J.plan()[0] == 1 else 0
    blocks = sum(-(-(int(sp[32 * g + 1] - sp[32 * g]) + extra) // 256) for g in range(-(-J.ndiag // 32)))
    nslots = int(sp[1] - sp[0])
    nlong = int(sp[33] - sp[32]) if J.ndiag > 32 else 0
    nwide = int(sp[1025] - sp[1024]) if J.ndiag > 1024 else 0
    combine = -(-(32 * nwide + nlong - nwide) // 256) if J.ndiag > 32 else 0
    return 9 + -(-(J.cols - nslots) // (256 * blocks)), blocks + combine


def _scratch_bytes(units):
    """device_bytes of the dot scratch sized for `units` work units: partials, reduction CTA sums, counter"""
    return 8 * (units + max(1, -(-units // 8192)) + 1)


# ---------------------------------------------------------------------------- GPU: every case, every variant
@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(CASES)), ids=IDS)
def test_y_is_the_axpby_result_and_the_dot_is_within_the_bound(eng, case):
    """For every CSR variant, every TJDS variant and the transposed call: y equals the *_axpby call bit for bit, the dot
    is within gamma_k of the exact sum for w = NULL, w = x and an unrelated w, and three runs give the same bits."""
    name, m, n, coo = CASES[case]
    rng = np.random.default_rng(500 + case)
    x = rng.uniform(-1, 1, n)
    dx = _cuda(x)
    A = eng.CsrMatrix.build(coo, m, n)
    for variant in (eng.CSR_AUTO, eng.CSR_VECTOR, eng.CSR_MERGE):
        for alpha, beta in PAIRS:
            y0 = _y0(rng, m, beta)
            ref = _cuda(y0)
            A.mult_device_axpby(alpha, dx, beta, ref, variant)
            ref = ref.cpu().numpy()
            d = DEPTH[_csr_plan(eng, A, variant)]
            for wname, w in _ws(rng, x, m):
                y, dot = _csr_run(A, alpha, dx, beta, y0, w, variant)
                assert same(y, ref), (name, variant, alpha, beta, wname)
                _check_dot(dot, None if w is None else w.cpu().numpy(), y, d, (name, variant, alpha, beta, wname))
                if (alpha, beta) == (-1.0, 1.0):
                    for _ in range(2):
                        assert bits(np.array([_csr_run(A, alpha, dx, beta, y0, w, variant)[1]]))[0] == bits(np.array([dot]))[0]
    A.free()

    J = eng.TjdsMatrix.build(coo, m, n)
    J.set_x_device(dx)
    for variant in (eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST, eng.TJDS_ATOMIC):
        for alpha, beta in PAIRS:
            y0 = _y0(rng, m, beta)
            for wname, w in _ws(rng, x, m):
                ref = _cuda(y0)
                J.mult_device_axpby(alpha, beta, ref, variant)
                dy, dd = _cuda(y0), _dot_buf()
                J.mult_device_axpby_dot(alpha, beta, dy, w, dd, variant)
                y, dot = dy.cpu().numpy(), dd.cpu().numpy()[0]
                if variant != eng.TJDS_ATOMIC:
                    assert same(y, ref.cpu().numpy()), (name, variant, alpha, beta, wname)
                    dy2, dd2 = _cuda(y0), _dot_buf()
                    J.mult_device_axpby_dot(alpha, beta, dy2, w, dd2, variant)
                    assert bits(dd2.cpu().numpy())[0] == bits(np.array([dot]))[0]
                _check_dot(dot, None if w is None else w.cpu().numpy(), y, DEPTH["tjds"], (name, variant, alpha, beta, wname))

    # transposed: x has m entries, y n
    xt = rng.uniform(-1, 1, m)
    dxt = _cuda(xt)
    for alpha, beta in PAIRS:
        y0 = _y0(rng, n, beta)
        ref = _cuda(y0)
        J.mult_transpose_device_axpby(alpha, dxt, beta, ref)
        ref = ref.cpu().numpy()
        d_tr = _transpose_plan(J)[0]
        wlist = [("null", None), ("other", _cuda(rng.uniform(-3, 3, n)))] + ([("x", dxt)] if m == n else [])
        for wname, w in wlist:
            dy, dd = _cuda(y0), _dot_buf()
            J.mult_transpose_device_axpby_dot(alpha, dxt, beta, dy, w, dd)
            y, dot = dy.cpu().numpy(), dd.cpu().numpy()[0]
            assert same(y, ref), (name, "transpose", alpha, beta, wname)
            _check_dot(dot, None if w is None else w.cpu().numpy(), y, d_tr, (name, "transpose", alpha, beta, wname))
            dy2, dd2 = _cuda(y0), _dot_buf()
            J.mult_transpose_device_axpby_dot(alpha, dxt, beta, dy2, w, dd2)
            assert bits(dd2.cpu().numpy())[0] == bits(np.array([dot]))[0]
    J.free()


# ---------------------------------------------------------------------------- GPU: the documented order, restated
@pytest.mark.gpu
def test_row_pattern_and_tjds_deterministic_order_restated_bit_for_bit(eng):
    """Where the work units are fixed row blocks the dot equals the numpy restatement of the documented order: tiles of
    32 rows (CSR row-pattern plan) and blocks of 256 rows (TJDS deterministic finalize), then dot_reduce's tree."""
    rng = np.random.default_rng(11)
    nx = 22
    m = nx ** 3
    coo = _stencil(nx, rng)
    x = rng.uniform(-1, 1, m)
    dx = _cuda(x)
    w = rng.uniform(-1, 1, m)
    A = eng.CsrMatrix.build(coo, m, m)
    J = eng.TjdsMatrix.build(coo, m, m)
    J.set_x_device(dx)
    for alpha, beta in PAIRS:
        y0 = _y0(rng, m, beta)
        for wv in (None, w):
            y, dot = _csr_run(A, alpha, dx, beta, y0, None if wv is None else _cuda(wv), eng.CSR_MERGE)
            assert A.row_patterns > 0
            terms = (y if wv is None else wv) * y
            want = reduce_partials(unit_partials(terms, 32))
            assert bits(np.array([dot]))[0] == bits(np.array([want]))[0], (alpha, beta, wv is None)
            for variant in (eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST):
                dy, dd = _cuda(y0), _dot_buf()
                J.mult_device_axpby_dot(alpha, beta, dy, None if wv is None else _cuda(wv), dd, variant)
                y = dy.cpu().numpy()
                terms = (y if wv is None else wv) * y
                want = reduce_partials(unit_partials(terms, 256))
                assert bits(dd.cpu().numpy())[0] == bits(np.array([want]))[0], (variant, alpha, beta, wv is None)
    A.free()
    J.free()


def test_reduction_restatement_is_a_tree_over_all_partials():
    """The numpy restatement itself: with exactly representable partials it returns their exact sum, for counts on both
    sides of one reduction CTA (8192) and of one second-level round (256 CTAs)."""
    rng = np.random.default_rng(0)
    for p in (0, 1, 31, 8192, 8193, 300000, 256 * 8192 + 5):
        part = rng.integers(-1000, 1000, p).astype(np.float64)
        assert reduce_partials(part) == float(np.sum(part)), p


# ---------------------------------------------------------------------------- GPU: determinism across grids and plans
def _dot_bits(A, alpha, dx, beta, y0, w, variant=0):
    return bits(np.array([_csr_run(A, alpha, dx, beta, y0, w, variant)[1]]))[0]


@pytest.mark.gpu
@pytest.mark.parametrize("plan", ["pattern", "merge", "relabel"])
def test_dot_does_not_depend_on_the_grid(eng, monkeypatch, plan):
    """The same handle at co-runner headroom 0 and 1 gives the same dot bits.  The matrices are large enough that the
    persistent grid is capped by residency, so the headroom changes the grid and which CTA walks which tile."""
    import torch

    rng = np.random.default_rng(12)
    if plan == "relabel":
        monkeypatch.setenv("SMVP_CSR_RELABEL", "1")
        n = 1 << 18
        r, c, v = eng.synth_rmat(18, 16 << 18, seed=42)
        A = eng.CsrMatrix.build_device(r, c, v, n, n, r.n)
        for a in (r, c, v):
            a.free()
    elif plan == "pattern":
        nx = 100
        n = nx ** 3
        r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_HASH, seed=3)
        A = eng.CsrMatrix.build_device(r, c, v, n, n, r.n)
        for a in (r, c, v):
            a.free()
    else:
        n = 200000
        A = eng.CsrMatrix.build(util.random_coo(rng, n, n, 5000000), n, n)
    dx = torch.empty(n, dtype=torch.float64, device="cuda")
    eng.synth_vector(dx, n, 31)
    y0 = rng.uniform(-1, 1, n)
    w = _cuda(rng.uniform(-1, 1, n))
    want = [_dot_bits(A, -1.0, dx, 1.0, y0, wv, eng.CSR_MERGE) for wv in (None, w, dx)]
    for _ in range(2):
        assert [_dot_bits(A, -1.0, dx, 1.0, y0, wv, eng.CSR_MERGE) for wv in (None, w, dx)] == want
    A.set_corunner_headroom(1)
    assert [_dot_bits(A, -1.0, dx, 1.0, y0, wv, eng.CSR_MERGE) for wv in (None, w, dx)] == want
    assert {"pattern": A.row_patterns > 0, "merge": A.row_patterns < 0, "relabel": A.x_relabel == 1}[plan]
    A.free()


# ---------------------------------------------------------------------------- GPU: edge cases
@pytest.mark.gpu
def test_edges_nan_prefill_empty_and_nonfinite(eng):
    import torch

    # rows = 0 and nnz = 0: +0.0, a NaN-prefilled d_dot is overwritten
    for m, n in ((0, 5), (30, 40)):
        coo = oracle.make_coo(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0))
        A = eng.CsrMatrix.build(coo, m, n)
        dy = torch.full((max(m, 1),), float("nan"), dtype=torch.float64, device="cuda")
        dd = _dot_buf()
        A.mult_device_axpby_dot(-1.0, _cuda(np.ones(n)), 0.0, dy if m else None, None, dd)
        assert bits(dd.cpu().numpy())[0] == 0, (m, n)  # +0.0 (and not NaN)
        A.free()
        J = eng.TjdsMatrix.build(coo, m, n)
        J.set_x_device(_cuda(np.ones(n)))
        for variant in (eng.TJDS_ATOMIC, eng.TJDS_DETERMINISTIC):
            dd = _dot_buf()
            J.mult_device_axpby_dot(-1.0, 0.0, dy if m else None, None, dd, variant)
            assert bits(dd.cpu().numpy())[0] == 0, (m, n, variant)
        dd = _dot_buf()
        J.mult_transpose_device_axpby_dot(-1.0, _cuda(np.ones(max(m, 1))) if m else None, 0.0,
                                          torch.full((n,), float("nan"), dtype=torch.float64, device="cuda"), None, dd)
        assert bits(dd.cpu().numpy())[0] == 0, (m, n, "transpose")
        J.free()
    # Inf / NaN in x: a non-finite dot of numpy's class
    m, n, coo = util.load_sample("memplus")
    rng = np.random.default_rng(13)
    for bad in (np.inf, np.nan):
        x = rng.uniform(-1, 1, n)
        x[rng.choice(n, size=3, replace=False)] = bad
        dx = _cuda(x)
        A = eng.CsrMatrix.build(coo, m, n)
        J = eng.TjdsMatrix.build(coo, m, n)
        J.set_x_device(dx)
        for variant in (eng.CSR_VECTOR, eng.CSR_MERGE):
            y, dot = _csr_run(A, 1.0, dx, 0.0, np.zeros(m), None, variant)
            with np.errstate(invalid="ignore", over="ignore"):
                want = float(np.dot(y, y))
            assert np.isnan(dot) == np.isnan(want) and np.isinf(dot) == np.isinf(want), (bad, variant, dot, want)
        for variant in (eng.TJDS_ATOMIC, eng.TJDS_DETERMINISTIC):
            dy, dd = _cuda(np.zeros(m)), _dot_buf(nan=False)
            J.mult_device_axpby_dot(1.0, 0.0, dy, dx if m == n else None, dd, variant)
            y = dy.cpu().numpy()
            with np.errstate(invalid="ignore", over="ignore"):
                want = float(np.dot(x if m == n else y, y))
            dot = dd.cpu().numpy()[0]
            assert np.isnan(dot) == np.isnan(want) and np.isinf(dot) == np.isinf(want), (bad, variant, dot, want)
        A.free()
        J.free()


@pytest.mark.gpu
def test_aliasing_is_refused(eng):
    import torch

    m, n, coo = util.load_sample("memplus")
    A = eng.CsrMatrix.build(coo, m, n)
    J = eng.TjdsMatrix.build(coo, m, n)
    x, y, w = (torch.ones(n, dtype=torch.float64, device="cuda") for _ in range(3))
    J.set_x_device(x)
    dd = _dot_buf()
    bad = [lambda: A.mult_device_axpby_dot(1.0, x, 1.0, y, None, None),  # d_dot NULL
           lambda: A.mult_device_axpby_dot(1.0, x, 1.0, y, y, dd),  # d_w == d_y
           lambda: A.mult_device_axpby_dot(1.0, x, 1.0, y, w, x),  # d_dot == d_x
           lambda: A.mult_device_axpby_dot(1.0, x, 1.0, y, w, y),  # d_dot == d_y
           lambda: A.mult_device_axpby_dot(1.0, x, 1.0, y, w, w),  # d_dot == d_w
           lambda: A.mult_device_axpby_dot(1.0, x, 1.0, x, None, dd),  # an *_axpby rule: y == x
           lambda: J.mult_device_axpby_dot(1.0, 1.0, y, None, None),
           lambda: J.mult_device_axpby_dot(1.0, 1.0, y, y, dd),
           lambda: J.mult_device_axpby_dot(1.0, 1.0, y, w, y),
           lambda: J.mult_device_axpby_dot(1.0, 1.0, y, w, w),
           lambda: J.mult_transpose_device_axpby_dot(1.0, x, 1.0, y, y, dd),
           lambda: J.mult_transpose_device_axpby_dot(1.0, x, 1.0, y, w, x),
           lambda: J.mult_transpose_device_axpby_dot(1.0, x, 1.0, x, None, dd)]
    for i, call in enumerate(bad):
        with pytest.raises(eng.SmvpError) as ei:
            call()
        assert ei.value.code == eng.E_ARG, i
    A.mult_device_axpby_dot(1.0, x, 1.0, y, x, dd)  # w may be the x the kernels read
    torch.cuda.synchronize()
    A.free()
    J.free()


# ---------------------------------------------------------------------------- GPU: launches and graphs
def _launches(eng, fn):
    import torch

    fn()
    torch.cuda.synchronize()
    before = eng.launch_count()
    fn()
    torch.cuda.synchronize()
    return eng.launch_count() - before


@pytest.mark.gpu
@pytest.mark.parametrize("plan", ["pattern", "merge", "vector", "relabel"])
def test_csr_launches(eng, monkeypatch, plan):
    """A CSR dot pass launches what the *_axpby call with (alpha, beta) != (1, 0) launches, plus the reduction."""
    import torch

    rng = np.random.default_rng(14)
    if plan == "relabel":
        monkeypatch.setenv("SMVP_CSR_RELABEL", "1")
        coo, n = synth_ref.rmat(14, 16 << 14), 1 << 14
    elif plan == "pattern":
        coo, n = _stencil(12, rng), 12 ** 3
    elif plan == "merge":
        coo, n = util.random_coo(rng, 3000, 3000, 60000), 3000
    else:
        coo, n = _band(3000, (-300, -2, -1, 0, 1, 2, 300), rng), 3000
    A = eng.CsrMatrix.build(coo, n, n)
    variant = eng.CSR_VECTOR if plan == "vector" else eng.CSR_MERGE
    x = _cuda(rng.uniform(-1, 1, n))
    y = torch.zeros(n, dtype=torch.float64, device="cuda")
    dd = _dot_buf()

    def device_bytes():
        info = eng.engine._CsrInfo()
        assert eng.lib().smvp_csr_info(A._h, ctypes.byref(info)) == 0
        return info.device_bytes

    epi = _launches(eng, lambda: A.mult_device_axpby(-1.0, x, 1.0, y, variant))
    before = device_bytes()
    for alpha, beta in ((1.0, 0.0), (-1.0, 1.0)):
        assert _launches(eng, lambda: A.mult_device_axpby_dot(alpha, x, beta, y, None, dd, variant)) == epi + 1, (plan, alpha)
    # the scratch is sized at the first dot call for the most units any variant or plan can use: the vector kernel's
    # CTAs, the 32-row pattern tiles, the merge-path tiles of at least 320 items -- and never grows afterwards
    mean = A.nnz / A.rows
    lpr = 2 if mean <= 8 else 4 if mean <= 16 else 8 if mean <= 32 else 16 if mean <= 64 else 32
    units = max(-(-A.rows * lpr // 256), -(-A.rows // 32), -(-(A.rows + A.nnz) // 320))
    assert device_bytes() - before == _scratch_bytes(units), plan
    for v in (eng.CSR_AUTO, eng.CSR_VECTOR, eng.CSR_MERGE):
        A.mult_device_axpby_dot(-1.0, x, 1.0, y, x, dd, v)
    torch.cuda.synchronize()
    assert device_bytes() - before == _scratch_bytes(units), plan
    A.free()


@pytest.mark.gpu
@pytest.mark.parametrize("relabel", ["0", "1"])
def test_tjds_launches_and_scratch(eng, monkeypatch, relabel):
    """TJDS: the *_axpby (-1, 1) launches plus the reduction, also for (1, 0) -- a natural-order atomic dot pass runs the
    scratch y and the per-row pass; the partials scratch is counted in device_bytes."""
    import torch

    monkeypatch.setenv("SMVP_TJDS_RELABEL", relabel)
    coo, n = synth_ref.rmat(16, 16 << 16), 1 << 16
    J = eng.TjdsMatrix.build(coo, n, n)
    J.set_x_device(_cuda(np.random.default_rng(15).uniform(-1, 1, n)))
    y = torch.zeros(n, dtype=torch.float64, device="cuda")

    def device_bytes():
        info = eng.engine._TjdsInfo()
        assert eng.lib().smvp_tjds_info(J._h, ctypes.byref(info)) == 0
        return info.device_bytes

    units = -(-n // 256)  # A x: 256-row blocks
    first = None
    for variant in (eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST, eng.TJDS_ATOMIC):
        epi = _launches(eng, lambda: J.mult_device_axpby(-1.0, 1.0, y, variant))  # (the atomic y_sum scratch comes here)
        before = device_bytes()
        first = before if first is None else first
        for alpha, beta in ((1.0, 0.0), (-1.0, 1.0)):
            dd = _dot_buf()
            assert _launches(eng, lambda: J.mult_device_axpby_dot(alpha, beta, y, None, dd, variant)) == epi + 1, (variant, alpha)
        # the first dot call adds exactly the partials scratch; later calls add nothing
        assert device_bytes() - before == (_scratch_bytes(units) if before == first else 0), variant
    # the transposed call: its first dot call, after A x ones, grows the scratch to the transposed units if they are more
    dx = _cuda(np.ones(n))
    epi = _launches(eng, lambda: J.mult_transpose_device_axpby(-1.0, dx, 1.0, y))
    before = device_bytes()
    dd = _dot_buf()
    assert _launches(eng, lambda: J.mult_transpose_device_axpby_dot(1.0, dx, 0.0, y, None, dd)) == epi + 1
    tr_units = _transpose_plan(J)[1]
    assert device_bytes() - before == (_scratch_bytes(tr_units) - _scratch_bytes(units) if tr_units > units else 0)
    J.free()


@pytest.mark.gpu
def test_graph_replay_equals_eager_passes(eng):
    """Three dot passes captured in a CUDA graph after a warm-up call, replayed, give the bits of three eager passes."""
    import torch

    rng = np.random.default_rng(16)
    nx = 16
    m = nx ** 3
    coo = _stencil(nx, rng)
    A = eng.CsrMatrix.build(coo, m, m)
    J = eng.TjdsMatrix.build(coo, m, m)
    x = _cuda(rng.uniform(-1, 1, m))
    J.set_x_device(x)
    y0 = _cuda(rng.uniform(-1, 1, m))
    calls = {"csr": lambda y, d, st: A.mult_device_axpby_dot(-0.5, x, 1.0, y, x, d, eng.CSR_AUTO, st),
             "tjds": lambda y, d, st: J.mult_device_axpby_dot(-0.5, 1.0, y, x, d, eng.TJDS_DETERMINISTIC, 0, st),
             "transpose": lambda y, d, st: J.mult_transpose_device_axpby_dot(-0.5, x, 1.0, y, None, d, st)}
    for name, call in calls.items():
        y = y0.clone()
        dots = torch.full((3,), float("nan"), dtype=torch.float64, device="cuda")
        for i in range(3):
            call(y, dots[i:], None)
        torch.cuda.synchronize()
        want_y, want_d = y.clone(), dots.clone()
        g = torch.cuda.CUDAGraph()
        y.copy_(y0)
        gd = torch.full((3,), float("nan"), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            cur = torch.cuda.current_stream()
            for i in range(3):
                call(y, gd[i:], cur)
        y.copy_(y0)
        gd.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(y.view(torch.int64), want_y.view(torch.int64)), name
        assert torch.equal(gd.view(torch.int64), want_d.view(torch.int64)), name
        del g
    A.free()
    J.free()


# ---------------------------------------------------------------------------- GPU: full size and a solver
@pytest.mark.gpu
def test_full_size_stencil_dot_against_torch(eng):
    """369^3 stencil, row-pattern plan, w = x: the fused dot is within gamma_k (k = 1 + 5 + 49) of torch.dot(x, y) plus
    torch's own error, and y equals the *_axpby result."""
    import torch

    nx = int(os.environ.get("SMVP_TEST_GRID", "369"))
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    x = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, m, 21)
    y0 = torch.empty_like(x)
    eng.synth_vector(y0, m, 22)
    ref = y0.clone()
    A.mult_device_axpby(-1.0, x, 1.0, ref)
    y = y0.clone()
    dd = _dot_buf()
    A.mult_device_axpby_dot(-1.0, x, 1.0, y, x, dd)
    torch.cuda.synchronize()
    assert A.row_patterns == 27
    assert torch.equal(y.view(torch.int64), ref.view(torch.int64))
    t = float(torch.dot(x, y))
    k = 1 + DEPTH["pattern"] + 49
    s_abs = float(torch.sum(torch.abs(x * y)))
    tol = 2 * k * U / (1 - k * U) * s_abs + 64 * math.log2(m) * U * s_abs  # ours + a generous bound for torch's order
    assert abs(float(dd[0]) - t) <= tol, (float(dd[0]), t)
    A.free()


def _cg_numpy(a, b, tol, maxit):
    x = np.zeros_like(b)
    r = b.copy()
    p = r.copy()
    rr = r @ r
    nb = math.sqrt(b @ b)
    for it in range(1, maxit + 1):
        ap = a @ p
        alpha = rr / (p @ ap)
        x += alpha * p
        r -= alpha * ap
        rr_new = r @ r
        if math.sqrt(rr_new) <= tol * nb:
            return x, it
        p = r + (rr_new / rr) * p
        rr = rr_new
    return x, maxit


@pytest.mark.gpu
def test_conjugate_gradient_with_the_fused_dot(eng):
    """CG on the SPD 27-point stencil (26 on the diagonal, -1 off it), 24^3, with q = A p and p^T q from one fused pass,
    reaches a 1e-10 relative residual within one iteration of numpy's CG on the same matrix."""
    import scipy.sparse as sp
    import torch

    nx = 24
    m = nx ** 3
    coo = synth_ref.stencil27(nx, nx, nx)
    a = sp.csr_matrix((coo["val"], (coo["row"], coo["col"])), shape=(m, m))
    b = np.random.default_rng(17).uniform(-1, 1, m)
    _, it_np = _cg_numpy(a, b, 1e-10, 500)

    A = eng.CsrMatrix.build(coo, m, m)
    x = torch.zeros(m, dtype=torch.float64, device="cuda")
    r = _cuda(b)
    p = r.clone()
    q = torch.empty_like(r)
    pq = _dot_buf()
    rr = float(torch.dot(r, r))
    nb = math.sqrt(rr)
    it = 0
    for it in range(1, 501):
        A.mult_device_axpby_dot(1.0, p, 0.0, q, p, pq)  # q = A p, pq = p^T q
        alpha = rr / float(pq[0])
        x.add_(p, alpha=alpha)
        r.add_(q, alpha=-alpha)
        rr_new = float(torch.dot(r, r))
        if math.sqrt(rr_new) <= 1e-10 * nb:
            break
        p.mul_(rr_new / rr).add_(r)
        rr = rr_new
    res = np.linalg.norm(b - a @ x.cpu().numpy()) / np.linalg.norm(b)
    assert res <= 2e-10, res
    assert it <= it_np + 1, (it, it_np)
    A.free()
