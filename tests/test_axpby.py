"""Scaled, accumulating multiply y = alpha * A x + beta * y (smvp_csr_mult_device_axpby, smvp_tjds_mult_device_axpby,
smvp_tjds_mult_transpose_device_axpby).  The contract (include/smvp_cuda.h): with s the plain pass's result for the same
handle, variant and x, the calls store fl(fl(alpha * s) + fl(beta * y)), or fl(alpha * s) without reading y when
beta == 0.  numpy restates that exactly as alpha * s + beta * y0 (no FMA), so every check here is bit for bit, except
where the plain pass itself is not reproducible (TJDS atomic)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import synth_ref
import util
from oracle import oracle

TOL = 1e-12
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(REPO, "smvp-toolkit_b200", "lib", "libsmvp_cuda.so")
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"

PAIRS = [(1.0, 0.0), (0.5, 0.0), (-1.0, 1.0), (1.0, 1.0), (2.5, -0.75), (0.0, 1.0), (-0.0, 1.0)]


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def same(got, want):
    """Bit for bit, except that any NaN matches any NaN (the device and numpy encode a fresh NaN differently)."""
    nan = np.isnan(want)
    return np.array_equal(np.isnan(got), nan) and np.array_equal(bits(got[~nan]), bits(want[~nan]))


def expected(alpha, s, beta, y0):
    with np.errstate(invalid="ignore", over="ignore"):
        return alpha * s if beta == 0.0 else alpha * s + beta * y0


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


# ---------------------------------------------------------------------------- CPU
def test_null_handle_and_bad_arguments_are_rejected(eng):
    L = eng.lib()
    y = np.zeros(4)
    p = eng.engine._ptr(y)
    assert L.smvp_csr_mult_device_axpby(None, 1.0, p, 0.0, p, eng.CSR_AUTO, None) == eng.E_ARG
    assert L.smvp_tjds_mult_device_axpby(None, 1.0, 0.0, p, eng.TJDS_ATOMIC, 0, None) == eng.E_ARG
    assert L.smvp_tjds_mult_transpose_device_axpby(None, 1.0, p, 0.0, p, None) == eng.E_ARG


def test_epilogue_kernels_are_in_the_library_spill_free():
    """Each epilogue instantiation exists, has no stack frame, and none is paired with the fan-out."""
    if not os.path.exists(LIB) or not os.path.exists(CUOBJDUMP):
        pytest.skip("library or cuobjdump not available")
    res = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = re.findall(r"Function (\S+):\s*\n\s*REG:\d+ STACK:(\d+)", res)
    wanted = {
        "pattern": r"csr_pattern_kernelILi4ELi1ELi1ELi14ELi7ELb0ELb1EE",
        "merge, stencil configuration": r"csr_merge_warp_kernelILi4ELi14ELi8ELb0ELb[01]ELb1ELb1EE",
        "merge, skewed configuration": r"csr_merge_warp_kernelILi2ELi10ELi14ELb0ELb[01]ELb0ELb1EE",
        "fix-up": r"merge_fixup_kernelILb0ELb1EE",
        "vector": r"csr_vector_kernelILi\d+ELb0ELb1EE",
        "det-finalize": r"tjds_det_finalize_kernelILb1EE",
        "unrank": r"tjds_unrank_y_kernelILb1EE",
        "transpose": r"tjds_transpose_kernelILb1EE",
        "combine": r"tjds_transpose_combine_kernelILb1EE",
        "empty transpose": r"tjds_axpby_empty_kernel",
    }
    counts = {"merge, stencil configuration": 2, "merge, skewed configuration": 2, "vector": 5}
    for what, pat in wanted.items():
        hits = [(name, stack) for name, stack in found if re.search(pat, name)]
        assert len(hits) == counts.get(what, 1), (what, hits)
        assert all(stack == "0" for _, stack in hits), (what, hits)
    fanout_epi = [name for name, _ in found
                  if re.search(r"csr_vector_kernelILi\d+ELb1ELb1EE|csr_pattern_kernel\w*ELb1ELb1EE|merge_fixup_kernelILb1ELb1EE|"
                               r"csr_merge_warp_kernelILi\d+ELi\d+ELi\d+ELb1ELb[01]ELb[01]ELb1EE", name)]
    assert not fanout_epi, fanout_epi


# ---------------------------------------------------------------------------- GPU helpers
def _cuda(a):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a, np.float64), device="cuda")


def _y0(rng, n, beta):
    """y before the call: NaN when beta == 0 (it must not be read), random otherwise."""
    return np.full(n, np.nan) if beta == 0.0 else rng.uniform(-2, 2, n)


def _csr_checks(A, x, rng, variant, pairs=PAIRS, ref=None):
    """A.mult_device_axpby against the plain pass of the same handle (and `ref`, the exact s, when given)."""
    import torch

    m = A.rows
    dx = _cuda(x)
    dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    A.mult_device(dx, dy, variant)
    s = dy.cpu().numpy()
    if ref is not None:
        assert np.array_equal(bits(s), bits(ref))
    for alpha, beta in pairs:
        y0 = _y0(rng, m, beta)
        dy = _cuda(y0)
        A.mult_device_axpby(alpha, dx, beta, dy, variant)
        got = dy.cpu().numpy()
        assert same(got, expected(alpha, s, beta, y0)), (variant, alpha, beta)
        if beta == 0.0 and np.isfinite(s).all():
            assert not np.isnan(got).any()


def _tjds_checks(J, x, rng, variant, pairs=PAIRS, diag_limit=0, tol=None):
    import torch

    m = J.rows
    J.set_x_device(_cuda(x))
    dy = torch.full((m,), float("nan"), dtype=torch.float64, device="cuda")
    J.mult_device(dy, variant, diag_limit)
    s = dy.cpu().numpy()
    for alpha, beta in pairs:
        y0 = _y0(rng, m, beta)
        dy = _cuda(y0)
        J.mult_device_axpby(alpha, beta, dy, variant, diag_limit)
        got = dy.cpu().numpy()
        want = expected(alpha, s, beta, y0)
        if tol is None:
            assert same(got, want), (variant, alpha, beta)
        else:
            fin = np.isfinite(want)
            assert same(got[~fin], want[~fin]), (variant, alpha, beta)  # Inf / NaN do not depend on the summation order
            assert util.rel_l2(got[fin], want[fin]) <= tol, (variant, alpha, beta)
        if beta == 0.0 and np.isfinite(s).all():
            assert not np.isnan(got).any()


# ---------------------------------------------------------------------------- GPU: composition
@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(CASES)), ids=IDS)
def test_composition_is_bit_exact(eng, case):
    """Every CSR variant and both deterministic TJDS variants: y equals alpha * s + beta * y0 bit for bit for every
    (alpha, beta) pair; with beta == 0 a NaN-filled y is never read.  On the stencil, where the row-pattern plan
    applies, s is the sequential loop itself."""
    name, m, n, coo = CASES[case]
    rng = np.random.default_rng(300 + case)
    x = rng.uniform(-1, 1, n)
    A = eng.CsrMatrix.build(coo, m, n)
    for variant in (eng.CSR_AUTO, eng.CSR_VECTOR, eng.CSR_MERGE):
        _csr_checks(A, x, rng, variant)
    if name.startswith("stencil"):
        rp, ci, va = oracle.csr_build(coo, m, n)
        _csr_checks(A, x, rng, eng.CSR_MERGE, ref=oracle.csr_mult(rp, ci, va, x))
        assert A.row_patterns > 0
    A.free()
    J = eng.TjdsMatrix.build(coo, m, n)
    for variant in (eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST):
        _tjds_checks(J, x, rng, variant)
    J.free()


# ---------------------------------------------------------------------------- GPU: plans
@pytest.mark.gpu
def test_csr_relabelled_columns_are_bit_exact(eng, monkeypatch):
    monkeypatch.setenv("SMVP_CSR_RELABEL", "1")
    coo = synth_ref.rmat(14, 16 << 14)
    n = 1 << 14
    A = eng.CsrMatrix.build(coo, n, n)
    rng = np.random.default_rng(1)
    x = rng.uniform(-1, 1, n)
    for variant in (eng.CSR_AUTO, eng.CSR_VECTOR, eng.CSR_MERGE):
        _csr_checks(A, x, rng, variant)
    assert A.x_relabel == 1
    A.free()


@pytest.mark.gpu
def test_csr_transpose_handle_against_the_transposed_loop(eng):
    """The handle smvp_csr_transpose builds is an ordinary handle: on a stencil with random values (not symmetric) its
    fused update is alpha * (sequential transposed loop) + beta * y0 bit for bit."""
    rng = np.random.default_rng(3)
    nx = 11
    m = nx ** 3
    coo = _stencil(nx, rng)
    sw = oracle.make_coo(coo["col"], coo["row"], coo["val"])
    trp, tci, tva = oracle.csr_build(sw, m, m)
    x = rng.uniform(-1, 1, m)
    A = eng.CsrMatrix.build(coo, m, m)
    T = A.transpose()
    _csr_checks(T, x, rng, eng.CSR_MERGE, ref=oracle.csr_mult(trp, tci, tva, x))
    assert T.row_patterns > 0
    T.free()
    A.free()


@pytest.mark.gpu
@pytest.mark.parametrize("skew", ["0", "1"])
@pytest.mark.parametrize("relabel", ["0", "1"])
def test_tjds_walks_and_relabelled_rows(eng, monkeypatch, skew, relabel):
    """Deterministic variants bitwise, atomic within 1e-12 (its s is not reproducible), on either walk and with or
    without relabelled rows."""
    monkeypatch.setenv("SMVP_TJDS_SKEW", skew)
    monkeypatch.setenv("SMVP_TJDS_RELABEL", relabel)
    coo = synth_ref.rmat(16, 16 << 16)
    n = 1 << 16
    rng = np.random.default_rng(4)
    x = rng.uniform(-1, 1, n)
    J = eng.TjdsMatrix.build(coo, n, n)
    for variant in (eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST):
        _tjds_checks(J, x, rng, variant)
    _tjds_checks(J, x, rng, eng.TJDS_ATOMIC, tol=TOL)
    assert J.plan()[0] == (1 if skew == "1" else -1)
    assert J.y_relabel == (1 if relabel == "1" else -1)
    J.free()


@pytest.mark.gpu
def test_tjds_reference_diag_limit(eng):
    rng = np.random.default_rng(5)
    for name in util.SAMPLES:
        m, n, coo = util.load_sample(name)
        J = eng.TjdsMatrix.build(coo, m, n)
        x = rng.uniform(-1, 1, n)
        for variant in (eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST):
            _tjds_checks(J, x, rng, variant, diag_limit=J.ref_diag_limit)
        J.free()


@pytest.mark.gpu
def test_inf_and_nan_follow_ieee(eng):
    """An x holding Inf / NaN routes the deterministic variants to the atomic kernel: the Inf / NaN pattern of the
    result is the formula's, the finite rows within 1e-12; alpha = 0 still propagates NaN from A x."""
    m, n, coo = util.load_sample("memplus")
    rng = np.random.default_rng(6)
    x = rng.uniform(-1, 1, n)
    x[rng.choice(n, size=4, replace=False)] = [np.inf, -np.inf, np.nan, np.inf]
    J = eng.TjdsMatrix.build(coo, m, n)
    for variant in (eng.TJDS_ATOMIC, eng.TJDS_DETERMINISTIC):
        _tjds_checks(J, x, rng, variant, tol=TOL)
    assert J.plan()[1] == -1
    J.free()
    A = eng.CsrMatrix.build(coo, m, n)
    for variant in (eng.CSR_VECTOR, eng.CSR_MERGE):
        _csr_checks(A, x, rng, variant)
    A.free()


# ---------------------------------------------------------------------------- GPU: transposed TJDS
@pytest.mark.gpu
def test_tjds_transpose_composition(eng):
    """alpha * (plain transposed pass) + beta * y0 bit for bit on a stencil (one launch), a matrix with a column of more
    than 32 entries (two launches), a matrix with empty columns, and a handle without entries, where beta == 0 stores
    the signed zero fl(alpha * 0) without reading y."""
    import torch

    rng = np.random.default_rng(7)
    coo = util.random_coo(rng, 400, 500, 3000)
    keep = coo["col"] % 5 != 0
    key = np.unique(np.concatenate([rng.choice(3000, size=100, replace=False) * 200 + 7, np.arange(3000) * 200 + np.arange(3000) % 200]))
    long_col = oracle.make_coo(key // 200, key % 200, rng.uniform(-1, 1, len(key)))  # column 7 holds ~115 entries
    cases = [("stencil 12^3", 12 ** 3, 12 ** 3, _stencil(12, rng), 1), ("long column", 3000, 200, long_col, 2),
             ("empty columns", 400, 500, coo[keep], 1),
             ("nnz 0", 30, 40, oracle.make_coo(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0)), 1)]
    for name, m, n, c, launches in cases:
        J = eng.TjdsMatrix.build(c, m, n)
        x = _cuda(rng.uniform(-1, 1, m))
        dy = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
        J.mult_transpose_device(x, dy)
        s = dy.cpu().numpy()
        for alpha, beta in PAIRS:
            y0 = _y0(rng, n, beta)
            dy = _cuda(y0)
            before = eng.launch_count()
            J.mult_transpose_device_axpby(alpha, x, beta, dy)
            assert eng.launch_count() - before == (0 if (alpha, beta) == (1.0, 0.0) and name == "nnz 0" else launches), name
            got = dy.cpu().numpy()
            assert same(got, expected(alpha, s, beta, y0)), (name, alpha, beta)
        if name == "nnz 0":
            dy = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
            J.mult_transpose_device_axpby(-1.0, x, 0.0, dy)
            assert np.array_equal(bits(dy.cpu().numpy()), bits(np.full(n, -0.0)))
        J.free()


# ---------------------------------------------------------------------------- GPU: launches
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
def test_csr_launches_match_the_plain_pass(eng, monkeypatch, plan):
    import torch

    rng = np.random.default_rng(8)
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
    plain = _launches(eng, lambda: A.mult_device(x, y, variant))
    assert _launches(eng, lambda: A.mult_device_axpby(-1.0, x, 1.0, y, variant)) == plain
    assert _launches(eng, lambda: A.mult_device_axpby(2.0, x, 0.0, y, variant)) == plain
    assert _launches(eng, lambda: A.mult_device_axpby(1.0, x, 0.0, y, variant)) == plain
    info = eng.engine._CsrInfo()
    assert eng.lib().smvp_csr_info(A._h, ctypes.byref(info)) == 0
    if A.x_relabel != 1:  # a relabelled pass with d_x also permutes x: one launch more than launches_per_mult counts
        assert plain == info.launches_per_mult[variant]
    assert {"pattern": A.row_patterns > 0, "merge": A.row_patterns < 0, "vector": True, "relabel": A.x_relabel == 1}[plan]
    A.free()


@pytest.mark.gpu
@pytest.mark.parametrize("relabel", ["0", "1"])
def test_tjds_launches(eng, monkeypatch, relabel):
    """Deterministic and relabelled atomic: the plain pass's launches; atomic in natural order one more, with a scratch
    of `rows` doubles counted in device_bytes; (1, 0) runs exactly the plain launches."""
    import torch

    monkeypatch.setenv("SMVP_TJDS_RELABEL", relabel)
    coo, n = synth_ref.rmat(16, 16 << 16), 1 << 16
    J = eng.TjdsMatrix.build(coo, n, n)
    J.set_x_device(_cuda(np.random.default_rng(9).uniform(-1, 1, n)))
    y = torch.zeros(n, dtype=torch.float64, device="cuda")

    def device_bytes():
        info = eng.engine._TjdsInfo()
        assert eng.lib().smvp_tjds_info(J._h, ctypes.byref(info)) == 0
        return info.device_bytes

    for variant in (eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST, eng.TJDS_ATOMIC):
        plain = _launches(eng, lambda: J.mult_device(y, variant))
        assert _launches(eng, lambda: J.mult_device_axpby(1.0, 0.0, y, variant)) == plain
        extra = 1 if variant == eng.TJDS_ATOMIC and relabel == "0" else 0
        assert _launches(eng, lambda: J.mult_device_axpby(-1.0, 1.0, y, variant)) == plain + extra
    assert J.y_relabel == (1 if relabel == "1" else -1)
    J.free()
    J = eng.TjdsMatrix.build(coo, n, n)
    J.set_x_device(_cuda(np.ones(n)))
    J.mult_device(y, eng.TJDS_ATOMIC)
    torch.cuda.synchronize()
    before = device_bytes()
    J.mult_device_axpby(-1.0, 1.0, y, eng.TJDS_ATOMIC)
    torch.cuda.synchronize()
    assert device_bytes() - before == (8 * n if relabel == "0" else 0)
    J.free()


# ---------------------------------------------------------------------------- GPU: repeated accumulation, graphs
@pytest.mark.gpu
def test_repeated_accumulation_on_a_stream_and_in_a_graph(eng):
    """Ten back-to-back beta = 1 calls on a non-default stream equal the numpy loop bit for bit; so do ten calls
    captured in a CUDA graph after one warm-up call, replayed: later calls only enqueue work."""
    import torch

    rng = np.random.default_rng(10)
    nx = 16
    m = nx ** 3
    coo = _stencil(nx, rng)
    x = rng.uniform(-1, 1, m)
    y0 = rng.uniform(-1, 1, m)
    alpha = -0.375
    A = eng.CsrMatrix.build(coo, m, m)
    J = eng.TjdsMatrix.build(coo, m, m)
    dx = _cuda(x)
    J.set_x_device(dx)
    s_csr, s_tjds = torch.empty_like(dx), torch.empty_like(dx)
    A.mult_device(dx, s_csr)
    J.mult_device(s_tjds, eng.TJDS_DETERMINISTIC)
    torch.cuda.synchronize()
    calls = {"csr": lambda y, st: A.mult_device_axpby(alpha, dx, 1.0, y, eng.CSR_AUTO, st),
             "tjds": lambda y, st: J.mult_device_axpby(alpha, 1.0, y, eng.TJDS_DETERMINISTIC, 0, st)}
    for name, s in (("csr", s_csr.cpu().numpy()), ("tjds", s_tjds.cpu().numpy())):
        want = y0.copy()
        for _ in range(10):
            want = alpha * s + 1.0 * want
        st = torch.cuda.Stream()
        y = _cuda(y0)
        torch.cuda.synchronize()
        with torch.cuda.stream(st):
            for _ in range(10):
                calls[name](y, st)
        st.synchronize()
        assert np.array_equal(bits(y.cpu().numpy()), bits(want)), name
        y = _cuda(y0)
        calls[name](y, None)  # warm-up: plans and scratch exist from here on
        torch.cuda.synchronize()
        y.copy_(_cuda(y0))
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            cur = torch.cuda.current_stream()
            for _ in range(10):
                calls[name](y, cur)
        y.copy_(_cuda(y0))
        g.replay()
        torch.cuda.synchronize()
        assert np.array_equal(bits(y.cpu().numpy()), bits(want)), name + " graph"
        del g
    A.free()
    J.free()


# ---------------------------------------------------------------------------- GPU: aliasing
@pytest.mark.gpu
def test_y_aliasing_x_is_refused(eng):
    import torch

    m, n, coo = util.load_sample("memplus")
    A = eng.CsrMatrix.build(coo, m, n)
    v = torch.ones(n, dtype=torch.float64, device="cuda")
    with pytest.raises(eng.SmvpError) as ei:
        A.mult_device_axpby(1.0, v, 1.0, v)
    assert ei.value.code == eng.E_ARG
    A.set_x_device(v)
    with pytest.raises(eng.SmvpError):
        A.mult_device_axpby(-1.0, None, 1.0, v)
    A.free()
    J = eng.TjdsMatrix.build(coo, m, n)
    with pytest.raises(eng.SmvpError) as ei:
        J.mult_transpose_device_axpby(1.0, v, 1.0, v)
    assert ei.value.code == eng.E_ARG
    J.set_x_device(v)  # A x reads the handle's permuted copy of x: y may be the caller's x
    J.mult_device_axpby(-1.0, 1.0, v, eng.TJDS_DETERMINISTIC)
    torch.cuda.synchronize()
    J.free()


# ---------------------------------------------------------------------------- GPU: full size
@pytest.mark.gpu
def test_full_size_stencil_residual(eng):
    """369^3 (stencil values: A ones = 27 - count): with y0 = b = 27 - count, x = ones, alpha = -1, beta = 1 the residual
    b - A x is exactly zero in every row, on the CSR row-pattern plan and on TJDS deterministic.  With a random x and y0
    the result equals -s + y0 computed elementwise from the plain pass, bit for bit."""
    import torch

    nx = int(os.environ.get("SMVP_TEST_GRID", "369"))
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    J = eng.TjdsMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    counts = torch.as_tensor(synth_ref.stencil27_row_counts(nx, nx, nx)).to("cuda").to(torch.float64)
    b = 27 - counts
    ones = torch.ones(m, dtype=torch.float64, device="cuda")
    y = b.clone()
    A.mult_device_axpby(-1.0, ones, 1.0, y, eng.CSR_MERGE)
    torch.cuda.synchronize()
    assert A.row_patterns == 27
    assert torch.equal(y, torch.zeros_like(y))
    J.set_x_device(ones)
    y = b.clone()
    J.mult_device_axpby(-1.0, 1.0, y, eng.TJDS_DETERMINISTIC)
    torch.cuda.synchronize()
    assert torch.equal(y, torch.zeros_like(y))
    x = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, m, 11)
    y0 = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(y0, m, 12)
    J.set_x_device(x)
    s = torch.empty_like(x)
    runs = ((lambda out: A.mult_device(x, out, eng.CSR_MERGE), lambda out: A.mult_device_axpby(-1.0, x, 1.0, out, eng.CSR_MERGE)),
            (lambda out: J.mult_device(out, eng.TJDS_DETERMINISTIC),
             lambda out: J.mult_device_axpby(-1.0, 1.0, out, eng.TJDS_DETERMINISTIC)))
    for plain, fused in runs:
        plain(s)
        want = torch.add(torch.mul(s, -1.0), torch.mul(y0, 1.0))  # two elementwise kernels: no FMA
        y = y0.clone()
        fused(y)
        torch.cuda.synchronize()
        assert torch.equal(y.view(torch.int64), want.view(torch.int64))
    A.free()
    J.free()
