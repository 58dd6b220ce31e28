"""Transposed product y = A^T x: the CSR transpose (smvp_csr_transpose, a second handle) and the TJDS gather along the
columns (smvp_tjds_mult_transpose*).  References: the sequential transposed loop (tests/transpose_loop.c), scipy, and a
numpy restatement of the order the TJDS kernels sum in (chunks of 32 entries per column)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import synth_ref
import util
from oracle import oracle

TOL = 1e-12
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(REPO, "smvp-toolkit_b200", "lib", "libsmvp_cuda.so")
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"
LOOP_SRC = os.path.join(REPO, "tests", "transpose_loop.c")


# ---------------------------------------------------------------------------- references
@pytest.fixture(scope="module")
def loop_lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("transpose_loop") / "libtransposeloop.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O3", "-ffp-contract=off", "-fPIC", "-shared", "-o", so, LOOP_SRC])
    L = ctypes.CDLL(so)
    L.oracle_csr_mult_transpose.argtypes = [ctypes.c_int32, ctypes.c_int32] + [ctypes.c_void_p] * 5
    L.oracle_csr_mult_transpose.restype = None
    return L


def loop_transpose(L, rp, ci, va, x, cols):
    """The sequential transposed loop: y[col_ind[j]] += val[j] * x[r] over the rows in order."""
    x = np.ascontiguousarray(x, np.float64)
    y = np.full(cols, np.nan)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    L.oracle_csr_mult_transpose(len(rp) - 1, cols, p(rp), p(ci), p(va), p(x), p(y))
    return y


def chunked_transpose(rp, ci, va, x, cols):
    """The order smvp_tjds_mult_transpose* sums in: column c's terms val * x[row] in ascending row order, cut into
    chunks of 32; each chunk summed left to right from +0.0, the chunk sums added left to right from +0.0.  Vectorised:
    position k within the chunk, then chunk g."""
    rows, nnz = len(rp) - 1, len(ci)
    row_of = np.repeat(np.arange(rows, dtype=np.int64), np.diff(rp))
    order = np.argsort(ci, kind="stable")  # CSR order is row-major: a stable sort by column keeps rows ascending
    c = ci[order].astype(np.int64)
    with np.errstate(invalid="ignore", over="ignore"):
        t = va[order] * x[row_of[order]]
    counts = np.bincount(ci, minlength=cols).astype(np.int64)
    start = np.cumsum(counts) - counts
    pos = np.arange(nnz, dtype=np.int64) - start[c]
    nch = (counts + 31) // 32
    base = np.cumsum(nch) - nch
    chunk = base[c] + pos // 32
    part = np.zeros(int(nch.sum()))
    with np.errstate(invalid="ignore", over="ignore"):
        for k in range(32):
            m = pos % 32 == k
            part[chunk[m]] += t[m]
        y = np.zeros(cols)
        chunk_col = np.repeat(np.arange(cols, dtype=np.int64), nch)
        chunk_g = np.arange(len(part), dtype=np.int64) - base[chunk_col]
        by_g = np.argsort(chunk_g, kind="stable")
        bounds = np.searchsorted(chunk_g[by_g], np.arange(int(nch.max(initial=0)) + 1))
        for g in range(len(bounds) - 1):
            sel = by_g[bounds[g]:bounds[g + 1]]
            y[chunk_col[sel]] += part[sel]
    return y


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def swapped(coo):
    return oracle.make_coo(coo["col"], coo["row"], coo["val"])


def scipy_csr(coo, m, n):
    return sp.csr_matrix((coo["val"], (coo["row"].astype(np.int64), coo["col"].astype(np.int64))), shape=(m, n))


# ---------------------------------------------------------------------------- matrices
def _band(m, offsets, rng):
    r = np.arange(m)
    rows = np.concatenate([r[(r + d >= 0) & (r + d < m)] for d in offsets])
    cols = np.concatenate([r[(r + d >= 0) & (r + d < m)] + d for d in offsets])
    return oracle.make_coo(rows, cols, rng.uniform(-1, 1, len(rows)))


def _one_long_column(m, n, length, rng):
    """Column 3 holds `length` entries, every other column a few."""
    rows = [rng.choice(m, size=length, replace=False)]
    cols = [np.full(length, 3)]
    r = rng.integers(0, m, size=4 * n)
    c = rng.integers(0, n, size=4 * n)
    rows.append(r[c != 3])
    cols.append(c[c != 3])
    key = np.unique(np.concatenate(rows).astype(np.int64) * n + np.concatenate(cols))
    return oracle.make_coo(key // n, key % n, rng.uniform(-1, 1, len(key)))


def _cases():
    """(name, m, n, coo): golden samples, rectangular and degenerate shapes, power-law and banded matrices."""
    for name in util.SAMPLES:
        m, n, coo = util.load_sample(name)
        yield name, m, n, coo
    rng = np.random.default_rng(11)
    yield "random 700x1900", 700, 1900, util.random_coo(rng, 700, 1900, 20000)
    yield "random 2500x300", 2500, 300, util.random_coo(rng, 2500, 300, 30000)
    coo = util.random_coo(rng, 400, 500, 3000)
    keep = (coo["row"] % 7 != 0) & (coo["col"] % 5 != 0)  # empty rows and empty columns
    yield "empty rows and columns", 400, 500, coo[keep]
    yield "1x1", 1, 1, oracle.make_coo(np.array([0]), np.array([0]), np.array([-2.5]))
    yield "nnz 0", 30, 40, oracle.make_coo(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0))
    yield "rmat 16", 1 << 16, 1 << 16, synth_ref.rmat(16, 16 << 16)
    yield "band 7", 3000, 3000, _band(3000, (-300, -2, -1, 0, 1, 2, 300), rng)


CASES = list(_cases())
IDS = [c[0] for c in CASES]


# ---------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("case", range(len(CASES)), ids=IDS)
def test_transposed_loop_is_the_forward_loop_of_the_swapped_matrix(loop_lib, case):
    """The reference loop over A's rows, scattering into y, equals the oracle's forward loop on the CSR of the swapped
    COO bit for bit (both add each column's terms in ascending row order), and scipy's A.T @ x within 1e-12."""
    _, m, n, coo = CASES[case]
    x = np.random.default_rng(case).uniform(-1, 1, m)
    rp, ci, va = oracle.csr_build(coo, m, n)
    y = loop_transpose(loop_lib, rp, ci, va, x, n)
    trp, tci, tva = oracle.csr_build(swapped(coo), n, m)
    assert np.array_equal(bits(y), bits(oracle.csr_mult(trp, tci, tva, x)))
    assert util.rel_l2(y, scipy_csr(coo, m, n).T @ x) <= TOL
    # the chunked order is the loop's order wherever no column holds more than 32 entries
    if len(coo) == 0 or np.bincount(coo["col"], minlength=n).max() <= 32:
        assert np.array_equal(bits(chunked_transpose(rp, ci, va, x, n)), bits(y))


def test_transposed_loop_on_random_rectangular_shapes(loop_lib):
    rng = np.random.default_rng(42)
    for _ in range(6):
        m, n = (int(v) for v in rng.integers(1, 300, size=2))
        coo = util.random_coo(rng, m, n, int(rng.integers(0, m * n // 3 + 1)))
        x = rng.uniform(-1, 1, m)
        rp, ci, va = oracle.csr_build(coo, m, n)
        y = loop_transpose(loop_lib, rp, ci, va, x, n)
        trp, tci, tva = oracle.csr_build(swapped(coo), n, m)
        assert np.array_equal(bits(y), bits(oracle.csr_mult(trp, tci, tva, x))), (m, n)
        assert util.rel_l2(y, scipy_csr(coo, m, n).T @ x) <= TOL


def test_transpose_kernels_are_in_the_library_spill_free():
    if not os.path.exists(LIB) or not os.path.exists(CUOBJDUMP):
        pytest.skip("library or cuobjdump not available")
    res = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = dict((name, stack) for name, stack in re.findall(r"Function (\S*tjds_transpose\w*kernel\S*):\s*\n\s*REG:\d+ STACK:(\d+)", res))
    for kernel in ("tjds_transpose_kernel", "tjds_transpose_combine_kernel"):
        hits = [s for name, s in found.items() if kernel in name]
        assert hits and all(s == "0" for s in hits), (kernel, found)
    assert "sm_100a" in subprocess.run([CUOBJDUMP, "-lelf", LIB], capture_output=True, text=True).stdout


def test_null_arguments_are_rejected():
    import smvp_toolkit_b200 as eng

    if not os.path.exists(eng.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    L = eng.lib()
    h = ctypes.c_void_p(0)
    assert L.smvp_csr_transpose(None, ctypes.byref(h)) == eng.E_ARG and not h.value
    assert L.smvp_csr_transpose(None, None) == eng.E_ARG
    assert L.smvp_tjds_mult_transpose_device(None, None, None, None) == eng.E_ARG
    y = np.zeros(4)
    assert L.smvp_tjds_mult_transpose(None, eng.engine._ptr(y), eng.engine._ptr(y), 1, None) == eng.E_ARG


# ---------------------------------------------------------------------------- GPU: CSR transpose
def _export_equals_scipy(T, coo, m, n):
    ref = scipy_csr(coo, m, n).T.tocsr()
    ref.sort_indices()
    rp, ci, va = T.export()
    assert (T.rows, T.cols, T.nnz) == (n, m, len(coo))
    assert np.array_equal(rp, ref.indptr) and np.array_equal(ci, ref.indices) and np.array_equal(bits(va), bits(ref.data))


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(CASES)), ids=IDS)
def test_csr_transpose_arrays_and_product(loop_lib, case):
    """For each arrival order of A's COO: export(A^T) == scipy's A.T.tocsr() bit for bit; A's export, info and A x are
    unchanged by the transpose; T x is within 1e-12 of the transposed loop; the handles free in either order."""
    import smvp_toolkit_b200 as eng

    _, m, n, coo = CASES[case]
    rng = np.random.default_rng(100 + case)
    x = rng.uniform(-1, 1, m)
    xa = rng.uniform(-1, 1, n)
    rp, ci, va = oracle.csr_build(coo, m, n)
    y_loop = loop_transpose(loop_lib, rp, ci, va, x, n)
    by_row = coo[np.lexsort((coo["col"], coo["row"]))]
    by_col = coo[np.lexsort((coo["row"], coo["col"]))]
    shuffled = coo.copy()
    rng.shuffle(shuffled)
    for k, arrival in enumerate((by_row, by_col, shuffled)):
        A = eng.CsrMatrix.build(arrival, m, n)
        before = A.export()
        ya, _ = A.mult(xa)
        info = eng.engine._CsrInfo()
        assert eng.lib().smvp_csr_info(A._h, ctypes.byref(info)) == 0
        info_before = bytes(info)
        T = A.transpose()
        _export_equals_scipy(T, coo, m, n)
        after = A.export()
        assert all(np.array_equal(bits(a) if a.dtype == np.float64 else a, bits(b) if b.dtype == np.float64 else b)
                   for a, b in zip(before, after))
        assert eng.lib().smvp_csr_info(A._h, ctypes.byref(info)) == 0
        assert bytes(info) == info_before
        ya2, _ = A.mult(xa)
        assert np.array_equal(bits(ya), bits(ya2))
        yt, _ = T.mult(x)
        assert util.rel_l2(yt, y_loop) <= TOL
        (A if k % 2 == 0 else T).free()
        (T if k % 2 == 0 else A).free()


@pytest.mark.gpu
def test_csr_transpose_of_a_relabelled_handle(monkeypatch):
    """A handle whose multiply reads relabelled columns still transposes from its natural col_ind."""
    import smvp_toolkit_b200 as eng

    monkeypatch.setenv("SMVP_CSR_RELABEL", "1")
    coo = synth_ref.rmat(14, 16 << 14)
    m = n = 1 << 14
    A = eng.CsrMatrix.build(coo, m, n)
    A.mult(np.ones(n))
    assert A.x_relabel == 1
    T = A.transpose()
    _export_equals_scipy(T, coo, m, n)
    T.free()
    A.free()


@pytest.mark.gpu
def test_csr_transpose_takes_the_row_pattern_plan(loop_lib):
    """A stencil (pattern transposed = pattern mirrored) and a non-symmetric band: A^T has row patterns, and its merge
    pass is bit-identical to the sequential transposed loop."""
    import smvp_toolkit_b200 as eng

    rng = np.random.default_rng(7)
    stencil = synth_ref.stencil27(11, 9, 7)
    stencil["val"] = rng.uniform(-1, 1, len(stencil))
    for m, coo in ((11 * 9 * 7, stencil), (3000, _band(3000, (-300, -2, -1, 0, 1, 2, 5, 300), rng))):
        x = rng.uniform(-1, 1, m)
        rp, ci, va = oracle.csr_build(coo, m, m)
        A = eng.CsrMatrix.build(coo, m, m)
        T = A.transpose()
        assert T.row_patterns == 0  # every plan starts undecided
        y, _ = T.mult(x, variant=eng.CSR_MERGE)
        assert T.row_patterns > 0
        assert np.array_equal(bits(y), bits(loop_transpose(loop_lib, rp, ci, va, x, m)))
        A.free()
        T.free()


# ---------------------------------------------------------------------------- GPU: TJDS transposed product
TJDS_CASES = CASES + [
    ("rmat 17", 1 << 17, 1 << 17, synth_ref.rmat(17, 16 << 17)),
    ("rmat 18", 1 << 18, 1 << 18, synth_ref.rmat(18, 16 << 18)),
    ("one column of 100000", 150000, 2000, _one_long_column(150000, 2000, 100000, np.random.default_rng(5))),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(TJDS_CASES)), ids=[c[0] for c in TJDS_CASES])
def test_tjds_transpose_follows_the_chunked_order(loop_lib, case):
    """Bit-identical to the numpy restatement of the chunked order (and so to the sequential loop where no column
    holds more than 32 entries); y pre-filled with NaN is overwritten everywhere; run to run identical; the host call
    equals the device call."""
    import torch

    import smvp_toolkit_b200 as eng

    _, m, n, coo = TJDS_CASES[case]
    x = np.random.default_rng(200 + case).uniform(-1, 1, m)
    rp, ci, va = oracle.csr_build(coo, m, n)
    y_ref = chunked_transpose(rp, ci, va, x, n)
    if len(coo) == 0 or np.bincount(coo["col"], minlength=n).max() <= 32:
        assert np.array_equal(bits(y_ref), bits(loop_transpose(loop_lib, rp, ci, va, x, n)))
    assert util.rel_l2(y_ref, scipy_csr(coo, m, n).T @ x) <= TOL
    A = eng.TjdsMatrix.build(coo, m, n)
    dx = torch.as_tensor(x, device="cuda")
    dy = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
    A.mult_transpose_device(dx, dy)
    y_dev = dy.cpu().numpy()
    assert np.array_equal(bits(y_dev), bits(y_ref))
    dy.fill_(float("nan"))
    A.mult_transpose_device(dx, dy)
    assert np.array_equal(bits(dy.cpu().numpy()), bits(y_dev))
    y_host, td = A.mult_transpose(x)
    assert np.array_equal(bits(y_host), bits(y_dev)) and len(td.time_each) == 1
    with pytest.raises(ValueError):
        A.mult_transpose(np.ones(m + 1))
    A.free()


@pytest.mark.gpu
@pytest.mark.parametrize("skew", ["0", "1"])
def test_tjds_transpose_with_either_walk_and_relabelled_rows(monkeypatch, skew):
    """The transposed pass walks the segment table straight whichever walk A x took, and reads row_ind whether or not
    A x scatters through relabelled rows: all handles give the same bits, before and after an A x pass."""
    import smvp_toolkit_b200 as eng

    coo = synth_ref.rmat(16, 16 << 16)
    m = n = 1 << 16
    x = np.random.default_rng(1).uniform(-1, 1, m)
    rp, ci, va = oracle.csr_build(coo, m, n)
    y_ref = chunked_transpose(rp, ci, va, x, n)
    monkeypatch.setenv("SMVP_TJDS_SKEW", skew)
    A = eng.TjdsMatrix.build(coo, m, n)
    y0, _ = A.mult_transpose(x)
    assert A.plan()[0] == (1 if skew == "1" else -1)
    assert np.array_equal(bits(y0), bits(y_ref))
    monkeypatch.setenv("SMVP_TJDS_RELABEL", "1")
    B = eng.TjdsMatrix.build(coo, m, n)
    B.mult(np.ones(n))  # A x decides the row relabelling
    assert B.y_relabel == 1
    y1, _ = B.mult_transpose(x)
    assert np.array_equal(bits(y1), bits(y_ref))
    A.free()
    B.free()


@pytest.mark.gpu
def test_tjds_transpose_inf_and_nan_follow_the_order():
    import smvp_toolkit_b200 as eng

    rng = np.random.default_rng(9)
    for name, m, n, coo in (TJDS_CASES[-1], CASES[util.SAMPLES.index("memplus")]):
        coo = coo.copy()
        x = rng.uniform(-1, 1, m)
        x[rng.choice(m, size=5, replace=False)] = [np.inf, -np.inf, np.nan, np.inf, 0.0]
        coo["val"][rng.choice(len(coo), size=3, replace=False)] = [np.nan, np.inf, 0.0]
        rp, ci, va = oracle.csr_build(coo, m, n)
        A = eng.TjdsMatrix.build(coo, m, n)
        y, _ = A.mult_transpose(x)
        assert np.array_equal(y, chunked_transpose(rp, ci, va, x, n), equal_nan=True), name
        A.free()


@pytest.mark.gpu
def test_tjds_transpose_batched_loop_and_launches():
    """The batched `-n` loop (small matrix, 100 passes) gives the single pass's y and 100 times; a pass on a stencil is
    one launch, on a matrix with columns longer than 32 two."""
    import torch

    import smvp_toolkit_b200 as eng

    m, n, coo = util.load_sample("memplus")
    x = np.random.default_rng(3).uniform(-1, 1, m)
    A = eng.TjdsMatrix.build(coo, m, n)
    y1, _ = A.mult_transpose(x, iters=1)
    y100, td = A.mult_transpose(x, iters=100)
    assert np.array_equal(bits(y100), bits(y1))
    assert len(td.time_each) == 100 and np.all(td.time_each > 0)
    A.free()
    for (nx, expect) in ((20, 1),):
        coo = synth_ref.stencil27(nx, nx, nx)
        m = nx ** 3
        S = eng.TjdsMatrix.build(coo, m, m)
        dx = torch.ones(m, dtype=torch.float64, device="cuda")
        dy = torch.empty(m, dtype=torch.float64, device="cuda")
        S.mult_transpose_device(dx, dy)  # plan
        before = eng.launch_count()
        for _ in range(3):
            S.mult_transpose_device(dx, dy)
        assert eng.launch_count() - before == 3 * expect
        counts = torch.as_tensor(synth_ref.stencil27_row_counts(nx, nx, nx)).to("cuda")
        assert torch.equal(dy, (27 - counts).to(torch.float64))
        S.free()
    R = eng.TjdsMatrix.build(synth_ref.rmat(14, 16 << 14), 1 << 14, 1 << 14)
    assert R.ndiag > 32
    dx = torch.ones(1 << 14, dtype=torch.float64, device="cuda")
    dy = torch.empty_like(dx)
    R.mult_transpose_device(dx, dy)
    before = eng.launch_count()
    R.mult_transpose_device(dx, dy)
    assert eng.launch_count() - before == 2
    R.free()


@pytest.mark.gpu
def test_full_size_stencil_transposes_to_itself():
    """369^3 with stencil values (26 on the diagonal, -1 elsewhere: A is symmetric): export(A^T) == export(A), A^T takes
    the 27-pattern plan, and A^T x (CSR) and A^T x (TJDS) are bit-identical to A x for a random x; x = ones gives the
    closed form 27 - count."""
    import torch

    import smvp_toolkit_b200 as eng

    nx = int(os.environ.get("SMVP_TEST_GRID", "369"))
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    J = eng.TjdsMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    T = A.transpose()
    for a, b in zip(A.export(), T.export()):
        assert np.array_equal(a, b)
    x = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(x, m, 5)
    y = torch.empty(m, dtype=torch.float64, device="cuda")
    yt = torch.full_like(y, float("nan"))
    yj = torch.full_like(y, float("nan"))
    A.mult_device(x, y)
    T.mult_device(x, yt)
    J.mult_transpose_device(x, yj)
    torch.cuda.synchronize()
    assert T.row_patterns == 27
    assert torch.equal(yt.view(torch.int64), y.view(torch.int64))
    assert torch.equal(yj.view(torch.int64), y.view(torch.int64))
    counts = torch.as_tensor(synth_ref.stencil27_row_counts(nx, nx, nx)).to("cuda").to(torch.float64)
    x.fill_(1.0)
    T.mult_device(x, yt)
    J.mult_transpose_device(x, yj)
    torch.cuda.synchronize()
    assert torch.equal(yt, 27 - counts) and torch.equal(yj, 27 - counts)
    A.free()
    T.free()
    J.free()
